// Body of the K1 kernels materialise_kernel and materialise_target_kernel (evaluate.cuh), included inside each: the
// including kernel defines RIG, OWN_IS_VIEW and L as template parameters and Poses, its ChunkPoses with the corner
// source (chunk.cuh: TARGET).  Textual inclusion, not a force-inlined function: a body function is optimised before it
// is inlined and then compiles materialise_kernel to different SASS (so does a local constexpr TARGET here).
  using ER = EvalRec<RIG>;
  using MS = MatSmem<RIG>;
  constexpr int BPW = PassGeom<RIG>::BPW;
  extern __shared__ __align__(128) double smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int chunk_id = blockIdx.x * MAT_WARPS + warp;
  if (chunk_id >= a.n_chunks) return;
  double* wsm = smem + (size_t)warp * MS::TOTAL;
  double* wrec = wsm;                 // Ceres-layout rows of the current group of 8 blocks
  const Chunk ch = a.chunks[chunk_id];
  const int b = lane >> 2, t = lane & 3;
  Poses poses(a, ch, wsm + ER::SIZE, lane);
  poses.start();
  auto load_pos = [&](int it) -> int {   // caller position of the lane's block
    return (it + b < ch.count) ? (a.orig ? a.orig[(int64_t)ch.start + it + b] : ch.start + it + b) : 0;
  };
  int pos_nxt = load_pos(0);
  double cost = 0.0;
  int buf = 0;
  for (int it = 0; it < ch.count; it += BPW, buf ^= 1) {
    double2 px;
    BlockGeom<RIG> geo;
    double ox, oy;
    const int pos = pos_nxt;
    if (it + BPW < ch.count) pos_nxt = load_pos(it + BPW);
    const bool valid = poses.group(it, buf, px, geo, ox, oy);
    // the previous group's bulk copies must have read the staging rows before they are rewritten
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    __syncwarp();
    double r2 = 0.0;
    if (valid) {
      CeresSink<RIG, OWN_IS_VIEW> sink{wrec, b, t, {0, 0, 0, 0, 0}};
      double r0, r1;
      const double depth = eval_corner<RIG, true, L>(geo, poses.sh, ox, oy, px.x, px.y, sink, r0, r1);
      if (!(depth > 0.0) || !isfinite(r0) || !isfinite(r1)) *a.fail_flag = 1;
      r2 = r0 * r0 + r1 * r1;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // staged rows -> visible to the async proxy
    __syncwarp();
    // copy-out by the TMA engine: one bulk copy per output array when the group's blocks are
    // consecutive in caller order, one per (block, array) otherwise
    const int nblk = min(BPW, ch.count - it);
    const int p0 = __shfl_sync(0xffffffffu, pos, 0);
    const bool run = __all_sync(0xffffffffu, !valid || pos == p0 + b);
    constexpr int NARR = RIG ? 6 : 5;
    const int n_copies = run ? NARR : nblk * NARR;
    for (int idx = lane; idx < ((n_copies + 31) & ~31); idx += 32) {   // uniform trip count: shuffle inside
      const int qq = run ? 0 : idx / NARR, arr = run ? idx : idx - qq * NARR;
      const int64_t o = __shfl_sync(0xffffffffu, pos, (qq & 7) * 4);
      double* dst = nullptr;
      int off = 0, k = 0;
      switch (arr) {
        case 0: dst = a.residuals; off = ER::RES; k = 8; break;
        case 1: dst = a.jac_intr; off = ER::JI; k = 32; break;
        case 2: dst = a.jac_dist; off = ER::JD; k = 40; break;
        case 3: dst = a.jac_view; off = ER::JV; k = 48; break;
        case 4: dst = a.jac_marker; off = ER::JM; k = 48; break;
        default: dst = a.jac_ext; off = ER::JX; k = 48; break;
      }
      if (idx < n_copies && dst)
        bulk_store(dst + o * k, wrec + off + qq * k, (run ? nblk : 1) * k * (int)sizeof(double));
    }
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    if (a.loss != 0) {
      double sb = r2 + __shfl_xor_sync(0xffffffffu, r2, 1);
      sb += __shfl_xor_sync(0xffffffffu, sb, 2);
      double rho1;
      r2 = valid ? 0.25 * robust_rho(a.loss, a.loss_a2, sb, rho1) : 0.0;
    }
    cost += r2;
  }
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // smem must outlive the reads
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cost += __shfl_xor_sync(0xffffffffu, cost, o);
  if (lane == 0 && a.cost2_partials) a.cost2_partials[chunk_id] = cost;
