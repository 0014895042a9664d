// The chunk pose pipeline of K1 (materialise_kernel, evaluate.cu) and K2 (assemble_kernel, assemble.cu).
//
// One warp walks one chunk: `count` sorted observation blocks that share the own 6-dof block and the camera, in
// groups of BPW = 8 blocks, and lane 4b + t evaluates corner t of block b of the group.  The own pose, the camera's
// body_T_cam (rig) and its shared parameters stay in the warp's shared memory for the whole chunk.  The other-block
// indices are fetched two groups ahead (lane q holds block q of the group), the other-pose records are staged one
// group ahead by cp.async into a double buffer, and every lane's pixel pair is loaded one group ahead.
//
// TARGET selects where a lane's tag corner comes from (its corner source): false, the square (-+s/2, -+s/2) of the
// marker's size; true, the corner layout of rcc_ba_set_corner_layout, whose slot of each block is fetched with the
// other-block index (Args::slot, in the pass's sorted order) and whose 64-byte slot record is read through the
// read-only path.  Slot -1 keeps the square.
#pragma once

#include "kernels.h"
#include "model.cuh"

namespace rcc {

// corner t of layout slot `slot`: the slot record is the 4 corners (x, y), 64 bytes, read through the read-only path
__device__ __forceinline__ void layout_corner(const double* corners, int slot, int t, double& ox, double& oy) {
  const double2 c = __ldg(reinterpret_cast<const double2*>(corners) + 4 * slot + t);
  ox = c.x;
  oy = c.y;
}

// 16-byte asynchronous copy global -> shared, cached in L1
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(d), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// doubles of a warp's pose region of shared memory:
// [2][BPW][POSEX] staged other-pose records | own pose | body_T_cam | shared parameters
template <bool RIG>
constexpr int CHUNK_POSE_SMEM = (2 * PassGeom<RIG>::BPW + 2) * POSEX + 16;

template <bool RIG, bool OWN_IS_VIEW, class Args, bool TARGET = false>
struct ChunkPoses {
  static constexpr int BPW = PassGeom<RIG>::BPW, SP = PassGeom<RIG>::SP;
  const Args& a;             // AssembleArgs or EvalArgs: oth, pix, view_x, marker_x, ext_x, shared
  const Chunk ch;
  const double* oth_table;   // expanded poses of the other blocks
  double* stage;             // [2][BPW][POSEX] other-pose records, double buffered
  double* own_x;             // [POSEX] own pose
  double* ext_x;             // [POSEX] body_T_cam (rig)
  double* sh;                // [SP] shared parameters of the chunk's camera
  const int lane, b, t;
  int oth_nxt;               // other blocks of the next group
  int slot_cur, slot_nxt;    // TARGET: layout slots of this group's and the next group's blocks (lane q: block q)
  double2 px_nxt;            // this lane's pixel pair of the next group

  // chunk constants -> the pose region `smem` (CHUNK_POSE_SMEM doubles of the warp's shared memory)
  __device__ __forceinline__ ChunkPoses(const Args& args, const Chunk& chunk, double* smem, int lane_)
      : a(args), ch(chunk), oth_table(OWN_IS_VIEW ? a.marker_x : a.view_x), stage(smem),
        own_x(smem + 2 * BPW * POSEX), ext_x(own_x + POSEX), sh(ext_x + POSEX), lane(lane_), b(lane_ >> 2),
        t(lane_ & 3) {
    const double* src = (OWN_IS_VIEW ? a.view_x : a.marker_x) + (size_t)ch.own * POSEX;
    if (lane < POSEX) own_x[lane] = src[lane];
    if (RIG && lane < POSEX) ext_x[lane] = a.ext_x[(size_t)ch.cam * POSEX + lane];
    if (lane < SP) sh[lane] = a.shared[ch.cam * SP + lane];
  }
  // the first group's other-pose records and pixels in flight
  __device__ __forceinline__ void start() {
    const int oth_cur = load_oth(0);
    oth_nxt = load_oth(BPW);
    if constexpr (TARGET) {
      slot_cur = load_slot(0);
      slot_nxt = load_slot(BPW);
    }
    issue_stage(0, 0, oth_cur);
    px_nxt = make_double2(0.0, 0.0);
    if (b < ch.count) px_nxt = *reinterpret_cast<const double2*>(a.pix + ((int64_t)ch.start + b) * 8 + 2 * t);
  }

  __device__ __forceinline__ int load_oth(int it) const {
    return (lane < BPW && it + lane < ch.count) ? a.oth[(int64_t)ch.start + it + lane] : 0;
  }
  __device__ __forceinline__ int load_slot(int it) const {
    return (lane < BPW && it + lane < ch.count) ? a.slot[(int64_t)ch.start + it + lane] : -1;
  }
  __device__ __forceinline__ void issue_stage(int it, int to, int oth_reg) {
    constexpr int PIECES = BPW * (POSEX / 2);   // 8 records x 12 16-byte pieces = 3 per lane
#pragma unroll
    for (int r = 0; r < PIECES / 32; ++r) {
      const int idx = lane + 32 * r;
      const int q = idx / (POSEX / 2), c = idx - q * (POSEX / 2);
      const int o = __shfl_sync(0xffffffffu, oth_reg, q);
      if (it + q < ch.count) cp_async16(stage + (to * BPW + q) * POSEX + 2 * c, oth_table + (size_t)o * POSEX + 2 * c);
    }
    cp_async_commit();
  }

  // Group `it` of the chunk (it = 0, BPW, 2 BPW, ... in turn; buf = 0, 1, 0, ... its staging buffer): waits for its
  // pose records and sets the next group in flight, then gives this lane's pixel pair and, if the lane's block
  // exists (the return value), its block geometry and tag corner.
  __device__ __forceinline__ bool group(int it, int buf, double2& px, BlockGeom<RIG>& geo, double& ox, double& oy) {
    const bool valid = (it + b) < ch.count;
    const int64_t g = (int64_t)ch.start + it + b;
    cp_async_wait_all();
    __syncwarp();
    px = px_nxt;
    int slot = -1;
    if constexpr (TARGET) {
      slot = __shfl_sync(0xffffffffu, slot_cur, b);
      slot_cur = slot_nxt;
    }
    if (it + BPW < ch.count) {
      issue_stage(it + BPW, buf ^ 1, oth_nxt);
      oth_nxt = load_oth(it + 2 * BPW);
      if constexpr (TARGET) slot_nxt = load_slot(it + 2 * BPW);
      if (it + BPW + b < ch.count)
        px_nxt = *reinterpret_cast<const double2*>(a.pix + (g + BPW) * 8 + 2 * t);
    }
    const double* ox_rec = stage + (buf * BPW + b) * POSEX;
    const double* vx = OWN_IS_VIEW ? own_x : ox_rec;
    const double* mx = OWN_IS_VIEW ? ox_rec : own_x;
    ox = 0.0, oy = 0.0;
    if (valid) {
      block_geometry<RIG>(vx, mx, RIG ? ext_x : nullptr, geo);
      if constexpr (TARGET) {
        if (slot >= 0) layout_corner(a.corners, slot, t, ox, oy);   // the only branch on the corner source
        else corner_xy(t, mx[PX_HS], ox, oy);
      } else {
        corner_xy(t, mx[PX_HS], ox, oy);
      }
    }
    return valid;
  }
};

}  // namespace rcc
