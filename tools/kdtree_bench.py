"""kmeans_mode 3 (the reference's kd-tree searches) against mode 0 (exact search) on bench-shape frames, in one run.

  python tools/kdtree_bench.py --out profiles/kdtree_bench.json

Legs (device-resident PCM, gsc_encode_frames_dev, host clock around the call and a stream synchronise):
  * 4 s stereo 44.1 kHz frames, K = 4096, 12-bit (bench.py's shape) at 148 / 592 / 1184 frames, mode 3 and mode 0
    alternating, `--reps` timed runs each after a two-frame warm-up;
  * the speculative k-means kernel against GSC_DBG_KDTREE_SERIAL (one point per round) on the smallest batch;
  * K = 256, 8-bit at the middle batch size;
  * speculation counters of every mode-3 run: points committed per round;
  * 2 frames checked against oracle.encode_frame(kmeans_mode=3);
  * the oracle's mode 3 on one frame per host core (bench.py's CPU arm), for the ratio;
  * the card's name and power limit (nvidia-smi), read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="148,592,1184")
    ap.add_argument("--reps", type=int, default=1)
    ap.add_argument("--seconds", type=float, default=4.0)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "kdtree_bench.json"))
    args = ap.parse_args()

    import torch
    import soundchunks_b200 as sc
    from bench import make_frames, cpu_encode_sample, SAMPLE_RATE
    from oracle import gsc_oracle as O

    if not torch.cuda.is_available():
        raise SystemExit("kdtree_bench.py needs a CUDA device")
    sizes = [int(s) for s in args.sizes.split(",")]
    ctx = sc.Context(0)
    result = {"card": card(), "frame_seconds": args.seconds, "sample_rate": SAMPLE_RATE, "channels": 2, "legs": []}

    def run(frames, dev, layout, params, serial=False):
        ctx.set_debug(sc.Context.DBG_KDTREE_SERIAL if serial else 0)
        ctx.synchronize()
        t0 = time.perf_counter()
        ctx.encode_frames_dev(dev.data_ptr(), layout, params)
        ctx.synchronize()
        dt = time.perf_counter() - t0
        ctx.set_debug(0)
        return dt

    def counters(n, params):
        if params.kmeans_mode != 3:
            return None
        # both internal lanes write their own counter buffer; the main context's lane holds the even frames
        c = ctx.online_counters(n if n < 16 else (n + 1) // 2).astype(np.float64)
        return {"rounds": float(c[:, 0].sum()), "points": float(c[:, 1].sum()), "lane_searches": float(c[:, 2].sum()),
                "overflowed_lists": float(c[:, 3].sum()), "points_per_round": float(c[:, 1].sum() / max(c[:, 0].sum(), 1))}

    def leg(n, K, bits, modes, serial_too=False):
        frames = make_frames(n, args.seconds, seed=1234)
        S = frames[0].shape[1]
        dev = torch.from_numpy(np.stack(frames)).to("cuda")
        layout = [(i * 2 * S, S, 2, S) for i in range(n)]
        audio = n * S / SAMPLE_RATE
        out = {"frames": n, "K": K, "bits": bits, "audio_seconds": audio}
        variants = [(m, False) for m in modes] + ([(3, True)] if serial_too else [])
        for m, ser in variants:                                  # warm-up: module load, kernel attributes
            p = sc.default_params(chunk_bit_depth=bits, chunks_per_frame=K, kmeans_mode=m)
            run(frames[:2], dev, layout[:2], p, ser)
        times = {v: [] for v in variants}
        stats = {}
        for _ in range(args.reps):                               # alternating
            for m, ser in variants:
                p = sc.default_params(chunk_bit_depth=bits, chunks_per_frame=K, kmeans_mode=m)
                times[(m, ser)].append(run(frames, dev, layout, p, ser))
                if m == 3:
                    stats[(m, ser)] = counters(n, p)
        for (m, ser), ts in times.items():
            name = f"mode{m}" + ("_serial" if ser else "")
            out[name] = {"seconds": ts, "audio_s_per_s": audio / min(ts), "counters": stats.get((m, ser))}
        return out, frames

    first = None
    for n in sizes:
        o, frames = leg(n, 4096, 12, (3, 0), serial_too=(n == sizes[0]))
        result["legs"].append(o)
        print(json.dumps(o), flush=True)
        if first is None:
            first = frames
    o, _ = leg(sizes[len(sizes) // 2], 256, 8, (3, 0))
    result["legs"].append(o)
    print(json.dumps(o), flush=True)

    # 2 frames of the first leg against the oracle
    res = ctx.encode_frames(first[:2], chunk_bit_depth=12, chunks_per_frame=4096, kmeans_mode=3)
    ok = []
    for f, r in zip(first[:2], res):
        ref = O.encode_frame(f, chunk_bit_depth=12, chunks_per_frame=4096, kmeans_mode=3)
        ok.append(bool((r.N, r.R, r.divider, r.passes, r.err) == (ref.N, ref.R, ref.divider, ref.passes, ref.err)
                       and np.array_equal(r.dict, ref.dict) and np.array_equal(r.index, ref.index)
                       and np.array_equal(r.attr, ref.attr)))
    result["oracle_check_2_frames"] = ok

    # the oracle's mode 3 on one frame per host core (all cores), as bench.py's CPU arm runs it
    cores = os.cpu_count() or 1
    dt, cres = cpu_encode_sample(first[:cores] if len(first) >= cores else make_frames(cores, args.seconds, seed=1234),
                                 4096, 12, cores, "kdtree")
    cpu = cores * args.seconds / dt
    result["cpu_oracle_mode3"] = {"cores": cores, "frames": cores, "seconds": dt, "audio_s_per_s": cpu}
    for o in result["legs"]:
        if o["K"] == 4096:
            o["mode3_vs_cpu_oracle"] = o["mode3"]["audio_s_per_s"] / cpu
    result["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as fh:
        json.dump(result, fh, indent=1)
    print(json.dumps({k: v for k, v in result.items() if k != "legs"}), flush=True)


if __name__ == "__main__":
    main()
