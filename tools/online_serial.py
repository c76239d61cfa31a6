"""Where a batch of the online k-means kernel (k_online, gsc_online.cuh) spends its cycles.

Builds the GSC_ONLINE_TIMING variant of the library (or takes one given with --so), loads it through GSC_CUDA_SO,
encodes bench-shape frames (bench.make_frames: 4 s stereo, ChunkCount = 4096, 12-bit) on one stream and prints, per
batch of 32 points, the cycles of each section warp 0 times (see GSC_ONLINE_TIMING in gsc_online.cuh), the share of
the batch in which warp 0 alone issues, (a+b+c+d)/f, and the kernel's path counters.

  python tools/online_serial.py [--frames 148] [--so LIB] [--json OUT]
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SECTIONS = ["(a) batch open + first proposals", "(b) R3 commit", "(c) R3 take-over / re-scans",
            "(d) R3' + R1, later rounds", "(e) R2 + bar 2 / bar 3", "(f) whole batch"]
COUNTERS = ["batches", "points", "exhaustive", "rounds", "full lists", "candidates", "moved again"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=148)
    ap.add_argument("--so", help="a library built with GSC_ONLINE_TIMING (default: build one under tools/_variants)")
    ap.add_argument("--json", help="write the per-frame counters and cycles here")
    args = ap.parse_args()
    so = args.so
    if not so:
        from soundchunks_b200 import build as b
        so = os.path.join(ROOT, "tools", "_variants", "libgsc_cuda_timing.so")
        os.makedirs(os.path.dirname(so), exist_ok=True)
        b.build_variant(so, 0, timing=True)
    os.environ["GSC_CUDA_SO"] = os.path.abspath(so)   # read when the package is imported
    os.environ["GSC_STREAMS"] = "1"                    # one lane: the counters of every frame stay in one context
    import bench
    import soundchunks_b200 as sc

    frames = bench.make_frames(args.frames, bench.FRAME_SECONDS, seed=1234)
    with sc.Context(0) as ctx:
        ctx.encode_frames(frames, chunk_bit_depth=12, chunks_per_frame=4096)
        cn = ctx.online_counters(args.frames)
    if not cn[:, 10:16].any():
        raise SystemExit(f"{so} records no cycles: it was not built with GSC_ONLINE_TIMING")
    tot = cn.sum(axis=0).astype(np.float64)
    nb = tot[0]
    print(f"{args.frames} frames, {int(nb)} batches, {int(tot[1])} points, {tot[3] / nb:.3f} rounds per batch")
    for i, name in enumerate(SECTIONS):
        print(f"  {name:34s} {tot[10 + i] / nb:9.1f} cycles/batch  {100 * tot[10 + i] / tot[15]:5.1f} %")
    serial = tot[10:14].sum()
    print(f"  warp 0 alone (a+b+c+d)             {serial / nb:9.1f} cycles/batch  {100 * serial / tot[15]:5.1f} %")
    print("  counters: " + ", ".join(f"{n} {int(tot[i])}" for i, n in enumerate(COUNTERS)))
    bad = cn[:, 8] > 0
    if bad.any():   # a build with GSC_ONLINE_CHECKS as well
        print(f"  CHECKS FAILED: {int(cn[:, 8].sum())} in {int(bad.sum())} frames (first at gsc_online.cuh:{int(cn[bad][0, 9])})")
    if args.json:
        with open(args.json, "w") as fh:
            json.dump({"so": os.path.basename(so), "counters": COUNTERS, "sections": SECTIONS,
                       "per_frame": cn[:, :16].astype(np.int64).tolist()}, fh)


if __name__ == "__main__":
    main()
