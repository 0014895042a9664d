"""Command line of the optimisation stage the reference pipeline is built around and does not ship ("Milestone 3",
real_preprocessing/README.md): read the `detections/` directory camera_pose_node leaves behind (targets.yaml +
detections_N.yaml with initial world_T_camera / world_T_target guesses, camera_pose.cpp:83-129, plus camera.yaml),
run the GPU bundle adjustment, and write the refined poses back in the same formats, where opt_vis_node
(opt_visualization.cpp:162-220) picks them up.

    python -m robot_camera_calibration_b200 <detections directory> [--fix-intrinsics | --intrinsics-sigma F C D] ...

With --initialise the directory needs only the detections and camera.yaml: the initial poses come from a batched
GPU PnP per tag, or per (frame, board) with --target, chained the way camera_pose_node chains tags.  Adding
--image-size W H calibrates a camera without camera.yaml: its intrinsics start from the board detections.
"""
from __future__ import annotations

import argparse
import json
import sys

# rcc_lm_summary.termination (include/rcc_ba.h)
TERMINATION = {0: "no_convergence (iteration limit)", 1: "convergence (function tolerance)",
               2: "convergence (gradient tolerance)", 3: "convergence (parameter tolerance)", 4: "failure"}


def parser():
    ap = argparse.ArgumentParser(prog="python -m robot_camera_calibration_b200", description=__doc__.split("\n\n")[0])
    ap.add_argument("directory", help="the detections directory (camera_pose.cpp:41-51: <package>/detections)")
    ap.add_argument("--device", type=int, default=0, help="CUDA device")
    intr = ap.add_mutually_exclusive_group()
    intr.add_argument("--fix-intrinsics", action="store_true",
                      help="keep camera.yaml's intrinsics and distortion constant (default: refined, written to "
                           "camera_refined.yaml)")
    intr.add_argument("--intrinsics-sigma", type=float, nargs=3, metavar=("FOCAL_PX", "PRINCIPAL_PX", "DIST"),
                      default=None,
                      help="refine the intrinsics under a Gaussian prior centred on camera.yaml: standard deviations "
                           "of fx fy, of cx cy (pixels) and of every distortion coefficient")
    ap.add_argument("--target", action="append", default=None, metavar="FILE",
                    help="a rigid tag board in Kalibr's AprilGrid format (target_type: aprilgrid, tagRows, tagCols, "
                         "tagSize, tagSpacing, optional firstTagId); repeatable.  Its detected tags are solved with "
                         "one pose per board; a tag id on two targets is an error")
    ap.add_argument("--initialise", action="store_true",
                    help="start from detections_N.yaml and camera.yaml alone: targets.yaml and any world_T_camera "
                         "stanzas are ignored, the initial poses come from PnP on the GPU (one per (frame, board) "
                         "with --target), and every frame that could not be chained loses its stanza")
    ap.add_argument("--image-size", type=int, nargs=2, metavar=("W", "H"), default=None,
                    help="with --initialise and --target: calibrate the camera from the board detections alone.  The "
                         "start comes from one homography per (frame, board) and OpenCV's closed form with the "
                         "principal point at the image centre, with zero distortion; camera.yaml is neither read nor "
                         "written, and camera_refined.yaml gets this size")
    ap.add_argument("--lens", choices=("radtan", "equidistant"), default=None,
                    help="with --image-size: the lens model to calibrate (default radtan)")
    ap.add_argument("--max-iterations", type=int, default=50)
    ap.add_argument("--function-tolerance", type=float, default=None)
    ap.add_argument("--gradient-tolerance", type=float, default=None)
    ap.add_argument("--parameter-tolerance", type=float, default=None)
    ap.add_argument("--precision", default=None,
                    help="'repr' writes poses with full round-trip precision instead of the reference's stream format")
    ap.add_argument("--verbose", action="store_true", help="one line per LM iteration on stderr")
    return ap


def main(argv=None):
    ap = parser()
    args = ap.parse_args(argv)
    if args.intrinsics_sigma is not None and not all(0 < s < float("inf") for s in args.intrinsics_sigma):
        ap.error("--intrinsics-sigma: every sigma must be positive and finite")
    if args.lens is not None and args.image_size is None:
        ap.error("--lens names the model to calibrate: it needs --image-size")
    if args.image_size is not None:
        if not args.initialise or not args.target:
            ap.error("--image-size estimates the intrinsics from board detections: it needs --initialise and --target")
        if args.fix_intrinsics or args.intrinsics_sigma is not None:
            ap.error("--image-size calibrates the intrinsics: it excludes --fix-intrinsics and --intrinsics-sigma")
        if not all(0 < v for v in args.image_size):
            ap.error("--image-size: width and height must be positive")
    from . import io_yaml
    opts = {"max_iterations": args.max_iterations, "verbose": int(args.verbose)}
    for k in ("function_tolerance", "gradient_tolerance", "parameter_tolerance"):
        if getattr(args, k) is not None:
            opts[k] = getattr(args, k)
    try:
        summary = io_yaml.optimise_directory(args.directory, device=args.device,
                                             refine_intrinsics=not args.fix_intrinsics, precision=args.precision,
                                             intrinsics_sigma=args.intrinsics_sigma, targets=args.target,
                                             initialise=args.initialise, image_size=args.image_size, lens=args.lens,
                                             **opts)
    except (FileNotFoundError, ValueError) as e:          # missing camera.yaml / targets.yaml, empty dataset, bad target
        print(f"error: {e}", file=sys.stderr)
        return 2
    summary["termination_name"] = TERMINATION.get(summary["termination"], "?")
    print(json.dumps(summary))
    return 0 if summary["termination"] != 4 else 1


if __name__ == "__main__":
    sys.exit(main())
