#!/usr/bin/env python
"""bench.py -- throughput of the SoundChunks encoder hot path (DoFrame, enc:1433-1447) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one pass of the whole per-frame hot path (attenuation divider, chunk features, yakmo
seeding, online k-means, dictionary, KNNFit, finalize) over one batch of synthetic frames of the
shape BASELINE.json names: 44.1 kHz stereo, 4 s frames, ChunkCount = 4096, 12-bit chunks.  Frames
are independent, so every rank (one per GPU) encodes its own batch: weak scaling, no collective on
the data path; torch.distributed is only the barrier and the max-over-ranks of the times.

Prints ONE JSON line (rank 0).  `value` = audio-seconds per second with the PCM already resident
in HBM (gsc_encode_frames_dev, CUDA events on the library's stream); `e2e` = the same metric
through the public host-buffer call gsc_encode_frames + gsc_fetch_stream (pinned staging + H2D + all
kernels + the device-side packer + ONE D2H of the .gsc stream's bytes inside the timed region).
Further keys: roofline (k_online, FP32), cpu_baseline, parity_check, lloyd_mode, and the
BASELINE.json configs[2..4] legs k256, strong_1h, split_frame (--no-extras skips them).

--impl reference times the CPU restatement of the reference (oracle/, all host threads) on a
bounded sample of the SAME workload: one 4 s frame of the same generator per host core and step,
searched the way the binary searches (ANN-1.1.2-style kd-tree rebuilt every pass); the FreePascal
encoder itself cannot be built here (DESIGN.md).  That, the cpu_baseline leg and the parity
probe (two of the step's frames against oracle.encode_frame, outside the timed region) are the
only places this file touches oracle/.

--dump-outputs DIR (e.g. bench_outputs, which git ignores) writes what the timed path computed in
its last step to DIR/*.npy; the inputs are seeded, so two builds run with the same arguments can
be compared file for file (dump_outputs lists the files).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SAMPLE_RATE = 44100
CHANNELS = 2
FRAME_SECONDS = 4.0
CHUNK_SIZE = 4
METRIC = "encoded audio-seconds per second (ChunkCount=4096, 12-bit chunks)"
UNIT = "audio-s/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="gsc_cuda", choices=["gsc_cuda", "reference"])
    ap.add_argument("--frames", type=int, default=1184,
                    help="frames per GPU per step (8 waves of 148 one-CTA-per-SM frames: 79 min of audio; the k-means tail of a\n"
                         "step, where the last 100-pass frames run alone, is amortised over more frames)")
    ap.add_argument("--chunks-per-frame", type=int, default=4096)
    ap.add_argument("--bits", type=int, default=12)
    ap.add_argument("--mode", default="online", choices=["online", "lloyd"],
                    help="online = the reference's rule (bit-exact vs the oracle); lloyd = batch Lloyd substitution")
    ap.add_argument("--lloyd-iters", type=int, default=30)
    ap.add_argument("--cpu-sample-seconds", type=float, default=FRAME_SECONDS,
                    help="length of each frame of the CPU sample (default: the workload's own 4 s frames)")
    ap.add_argument("--cpu-search", default="kdtree", choices=["kdtree", "exact"],
                    help="CPU arm: ANN-style kd-tree rebuilt per pass (what the binary does) or exhaustive exact search")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-lloyd", action="store_true", help="skip the secondary Lloyd-mode leg")
    ap.add_argument("--no-extras", action="store_true", help="skip the k256 / strong_1h / split_frame legs")
    ap.add_argument("--no-parity", action="store_true", help="skip the parity probe against the oracle")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step computed to DIR/*.npy (rank 0; see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ---------------------------------------------------------------------------------------------
# outputs of the timed path, for comparing two builds run with the same arguments
# ---------------------------------------------------------------------------------------------
DUMP_SAMPLE_FRAMES = 16
DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, res, gsc=None, gsc_sizes=None):
    """Write the per-frame results of the last timed step as float32 / float64 .npy files:

      frame_scalars  float64 [F][6]            N, R, divider, passes, err, overfull of every frame
      sample_frames  float64 [n]               a fixed, seeded sample of min(F, 16) frame numbers, ascending
      index, attr    float32 [sum N]           the sampled frames' arrays, concatenated in that order
      dict           float32 [sum R][chunk_size], datten float32 [sum R]   (split all four with N and R)
      gsc_sizes      float64 [F]               .gsc size of every frame      } only when the path packs the
      gsc_bytes      float32 [...]             the sampled frames' .gsc bytes } stream (not --impl reference)

    Every frame's arrays together would exceed 64 MB at the bench shape (1,184 frames of 88,200 indexes each), so
    they come from a sample; the scalars (the Double error sum among them) cover every frame."""
    F = len(res)
    pick = np.sort(np.random.default_rng(0).choice(F, min(F, DUMP_SAMPLE_FRAMES), replace=False))
    out = {
        "frame_scalars": np.array([[r.N, r.R, r.divider, r.passes, r.err, r.overfull] for r in res], np.float64),
        "sample_frames": pick.astype(np.float64),
        "index": np.concatenate([res[i].index for i in pick]).astype(np.float32),
        "attr": np.concatenate([res[i].attr for i in pick]).astype(np.float32),
        "dict": np.concatenate([res[i].dict for i in pick]).astype(np.float32),
        "datten": np.concatenate([res[i].datten for i in pick]).astype(np.float32),
    }
    if gsc is not None:
        offs = np.concatenate([[0], np.cumsum(gsc_sizes)])
        b = np.frombuffer(gsc, np.uint8)
        out["gsc_sizes"] = np.asarray(gsc_sizes, np.float64)
        out["gsc_bytes"] = np.concatenate([b[offs[i]:offs[i + 1]] for i in pick]).astype(np.float32)
    total = sum(a.nbytes for a in out.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of outputs, more than {DUMP_LIMIT_BYTES}")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------
# synthetic workload
# ---------------------------------------------------------------------------------------------
def make_frames(n, seconds, seed, sample_rate=SAMPLE_RATE):
    """n distinct synthetic frames, planar int16 [C][S]; 16 distinct signals are generated and
    re-mixed (channel swap / time reversal / polarity) so that the generation stays short."""
    from soundchunks_b200.synth import synth_frames
    base = synth_frames(min(n, 16), seconds, sample_rate, CHANNELS, seed=seed, chunk_size=CHUNK_SIZE)
    out = []
    for i in range(n):
        f = base[i % len(base)]
        v = (i // len(base)) % 8
        if v & 1:
            f = f[::-1]
        if v & 2:
            f = f[:, ::-1]
        if v & 4:
            f = -np.maximum(f, -32767)
        if i // len(base) >= 8:
            f = np.roll(f, 997 * (i // len(base)), axis=1)
        out.append(np.ascontiguousarray(f, dtype=np.int16))
    return out


# ---------------------------------------------------------------------------------------------
# clocks (B200_PROFILING.md: sample nvidia-smi DURING the timed region)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index):
        self.index, self.rows, self.proc, self.th = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.th = threading.Thread(target=self._read, daemon=True)
        self.th.start()

    def _read(self):
        for line in self.proc.stdout:
            p = [x.strip() for x in line.split(",")]
            if len(p) >= 7:
                self.rows.append(p)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for p in self.rows:
            try:
                sm.append(float(p[0])); mx.append(float(p[1])); pw.append(float(p[2]))
            except ValueError:
                continue
            for name, v in zip(self.NAMES, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle (C restatement of the reference path), frame-parallel over host threads
# like ProcThreadPool (mtprocs.pas:598-602, enc:1449)
# ---------------------------------------------------------------------------------------------
def cpu_encode_sample(frames, K, bits, threads, search="kdtree"):
    from concurrent.futures import ThreadPoolExecutor
    from oracle import gsc_oracle as O
    O.build()
    # kmeans_mode 3: enc:699-765 / 915-965 through an ANN-1.1.2-style kd-tree rebuilt every pass, as the binary does
    # (leaf distances on the live rows, planes from the pass start); 0: exhaustive exact search (the GPU's contract)
    p = O.default_params(chunk_bit_depth=bits, chunks_per_frame=K, kmeans_mode=3 if search == "kdtree" else 0)
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        res = list(ex.map(lambda f: O.encode_frame(f, p), frames))
    return time.perf_counter() - t0, res


def cpu_sample_text(cores, seconds, res, K, search, extra=""):
    how = ("nearest centroid / 64 nearest variants through an ANN-1.1.2-style kd-tree rebuilt every pass (enc:729, 945), "
           "as the binary searches" if search == "kdtree" else "exhaustive exact search (vectorised)")
    return (f"{cores} frames x {seconds:g} s of the same synthetic {SAMPLE_RATE} Hz stereo generator per step "
            f"(N={res[0].N} chunks/frame, K={K}), one frame per host thread{extra}; online passes "
            f"{[r.passes for r in res]}; C restatement of encoder.lpr's DoFrame (the FreePascal binary cannot be built "
            f"here); {how}")


def run_reference(args, rank):
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    frames = make_frames(cores, args.cpu_sample_seconds, seed=4321)
    audio_s = sum(f.shape[1] for f in frames) / SAMPLE_RATE
    for _ in range(min(args.warmup, 1)):        # one warm-up pass is enough for a CPU loop
        cpu_encode_sample(frames, args.chunks_per_frame, args.bits, cores, args.cpu_search)
    t = 0.0
    for _ in range(args.steps):
        dt, res = cpu_encode_sample(frames, args.chunks_per_frame, args.bits, cores, args.cpu_search)
        t += dt
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, res)
    value = audio_s * args.steps / t
    sample = cpu_sample_text(cores, args.cpu_sample_seconds, res, args.chunks_per_frame, args.cpu_search)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": 1e3 * t / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, args.frames, FRAME_SECONDS),
        # what one step of THIS arm really ran (a bounded sample of the workload `config` names)
        "sample": {"frames_per_step": cores, "frame_seconds": args.cpu_sample_seconds, "chunks_per_frame_N": res[0].N,
                   "search": args.cpu_search, "same_frame_shape_as_config": args.cpu_sample_seconds == FRAME_SECONDS},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, frames_per_gpu, seconds):
    return {
        "workload": "lame_test-shaped full-bitrate encode (BASELINE.json configs[1]): synthetic 44.1 kHz stereo, "
                    f"{seconds:g} s frames, ChunkSize=4, ChunkCount={args.chunks_per_frame}, {args.bits}-bit chunks",
        "frames_per_gpu_per_step": frames_per_gpu, "frame_seconds": seconds, "sample_rate": SAMPLE_RATE,
        "channels": CHANNELS, "chunks_per_frame": args.chunks_per_frame, "chunk_bit_depth": args.bits,
        "kmeans": args.mode, "parallelism": f"frame-sharded x{args.gpus}, no collective",
        "l2": "L2 flushed (256 MiB write) between steps; per-step working set (features) > 126 MB L2",
    }


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import soundchunks_b200 as sc

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (libgsc_cuda has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier(device_ids=[local_rank])
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    F = args.frames
    frames = make_frames(F, FRAME_SECONDS, seed=1234 + 100003 * rank)
    audio_s_rank = sum(f.shape[1] for f in frames) / SAMPLE_RATE
    params = sc.default_params(chunk_bit_depth=args.bits, chunks_per_frame=args.chunks_per_frame,
                               kmeans_mode=1 if args.mode == "lloyd" else 0, lloyd_iters=args.lloyd_iters)
    ctx = sc.Context(local_rank)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))

    # device-resident PCM for the `value` leg
    S = frames[0].shape[1]
    host = torch.from_numpy(np.stack(frames)).pin_memory()          # [F][C][S]
    dev = host.to("cuda", non_blocking=True)
    torch.cuda.synchronize()
    layout = [(i * CHANNELS * S, S, CHANNELS, S) for i in range(F)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def step_dev():
        with torch.cuda.stream(stream):
            flush.zero_()
        ctx.encode_frames_dev(dev.data_ptr(), layout, params)

    for _ in range(args.warmup):
        step_dev()
    ctx.synchronize()
    fp32_peak = ctx.fp32_peak_tflops()

    clocks = ClockSampler(local_rank)
    barrier()
    clocks.start()
    ctx.reset_stats()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    stage_acc = {}
    for _ in range(args.steps):
        step_dev()
    ev1.record(stream)
    ctx.synchronize()
    barrier()
    clk = clocks.stop()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    launches = ctx.stats()["kernel_launches"] + args.steps  # + the L2 flush fill kernel of each step
    res = ctx.fetch_results(layout, params)                 # also collects the stage events of the last step
    dev_stream, dev_sizes = ctx.fetch_stream(F, SAMPLE_RATE)   # .gsc bytes of the device-resident leg's last step
    stage_acc = ctx.stats()["stage_ms"]                     # last step's stage times (CUDA events, ctx stream)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, dev_stream, dev_sizes)
    passes = [r.passes for r in res]
    Ns = [r.N for r in res]
    total_audio = sum_over_ranks(audio_s_rank)
    value = total_audio * args.steps / (ms_total * 1e-3)

    # roofline of the dominant kernel (k-means stage = one launch of k_online, or the Lloyd launches)
    D = 2 * CHUNK_SIZE
    K = args.chunks_per_frame
    if args.mode == "online":
        flops = sum(2.0 * n * K * D * p for n, p in zip(Ns, passes))
        kname = "k_online"
    else:
        flops = sum(2.0 * n * K * D * (args.lloyd_iters + 1) for n in Ns)
        kname = "k_assign"
    # the library runs a batch on two streams (even / odd frames); stage_ms are the CUDA-event stage times of both
    # lanes ADDED UP; the roofline divides by the UNION of the two lanes' k-means intervals (wall time with a
    # k-means kernel running on either stream)
    km_ms = ctx.stage_busy_ms("kmeans")     # wall time with a k-means kernel running on either stream (union)
    achieved = flops / (km_ms * 1e-3) / 1e12 if km_ms > 0 else 0.0
    traffic, traffic_src = None, None
    try:    # dram bytes per launch of the dominant kernel, from the committed `ncu --set full` capture at the bench shape
        with open(os.path.join(ROOT, "profiles", "r2_traffic.json")) as fh:
            tj = json.load(fh)
        traffic, traffic_src = tj.get(kname, {}).get("dram_bytes_per_launch"), tj.get(kname, {}).get("source")
    except (OSError, ValueError):
        pass
    roofline = {
        "bound": "fp32", "kernel": kname, "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
        "frac": achieved / fp32_peak if fp32_peak else None, "traffic": traffic, "traffic_source": traffic_src,
        "note": "algorithmic flops = 2*N*K*D per pass (dense count, SURVEY.md 8d), D=8; duration = CUDA events "
                "around the k-means stage of the last timed step; peak = FFMA probe measured in this run "
                "(MEASURED_PEAKS.json has no FP32 figure); share of step = %.3f" % (km_ms / max(stage_acc["total"], 1e-9)),
    }

    # e2e leg: public host-buffer call
    e2e = None
    if not args.no_e2e:
        # host PCM in -> .gsc bytes out: gsc_encode_frames (pinned staging, H2D, all kernels, the device-side
        # .gsc packer) + gsc_fetch_stream (D2H of the stream) -- what an encoder front-end calls per batch
        import hashlib
        ref_stream = dev_stream
        ctx.encode_to_stream(frames, SAMPLE_RATE, params)       # warm-up (allocates the pinned staging)
        barrier()
        ctx.reset_stats()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            blob, sizes = ctx.encode_to_stream(frames, SAMPLE_RATE, params)
        ctx.synchronize()
        dt = time.perf_counter() - t0
        barrier()
        dt = max_over_ranks(dt)
        s2 = ctx.stats()
        e2e = {"value": total_audio * args.steps / dt, "unit": UNIT,
               "h2d_bytes_per_step": sum_over_ranks(s2["h2d_bytes"]) / args.steps,
               "d2h_bytes_per_step": sum_over_ranks(s2["d2h_bytes"]) / args.steps,
               "ms_per_step": 1e3 * dt / args.steps, "gsc_bytes_per_step_this_rank": len(blob),
               "api": "gsc_encode_frames(host PCM, results=NULL) + gsc_fetch_stream -> .gsc bytes in host memory"}
        assert hashlib.sha256(blob).digest() == hashlib.sha256(ref_stream).digest(), "host-buffer and device-resident legs disagree"

    # secondary leg: the batch-Lloyd substitution (kmeans_mode = 1, BASELINE.json's register-tiled distance+argmin
    # kernel) on the same frames, one step, to report the roofline of k_assign next to the default mode
    lloyd = None
    if args.mode == "online" and not args.no_lloyd:
        lp = sc.default_params(chunk_bit_depth=args.bits, chunks_per_frame=args.chunks_per_frame, kmeans_mode=1,
                               lloyd_iters=args.lloyd_iters)
        ctx.encode_frames_dev(dev.data_ptr(), layout, lp)       # warm-up
        ctx.synchronize()
        l0, l1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0.record(stream)
        ctx.encode_frames_dev(dev.data_ptr(), layout, lp)
        l1.record(stream)
        ctx.synchronize()
        lres = ctx.fetch_results(layout, lp)
        lst = ctx.stats()["stage_ms"]
        lflops = sum(2.0 * r.N * K * D * (args.lloyd_iters + 1) for r in lres)
        lms = l0.elapsed_time(l1)
        lkm = ctx.stage_busy_ms("kmeans")
        lloyd = {"value": audio_s_rank / (lms * 1e-3), "unit": UNIT + " (this rank)", "lloyd_iters": args.lloyd_iters,
                 "ms_per_step": lms, "kmeans_stage_ms_sum_of_streams": lst["kmeans"], "kmeans_stage_busy_ms": lkm,
                 "roofline": {"bound": "fp32", "kernel": "k_assign + k_scatter_sums_d", "unit": "TFLOP/s",
                              "achieved": lflops / (lkm * 1e-3) / 1e12, "peak": fp32_peak,
                              "frac": lflops / (lkm * 1e-3) / 1e12 / fp32_peak if fp32_peak else None,
                              "note": "dense count 2*N*K*D*(iters+1) / wall time with the stage running on either stream; "
                                      "other stages of the other stream share the GPU during that time"}}

    # parity probe, OUTSIDE every timed region: two frames of the step's batch (one per internal lane) re-encoded by the
    # CPU oracle (exhaustive exact search: the library's contract) and compared bit for bit, fields and .gsc bytes
    parity = None
    if rank == 0 and not args.no_parity and args.mode == "online":
        from concurrent.futures import ThreadPoolExecutor
        from oracle import gsc_oracle as O
        probe = [0, 1] if F > 1 else [0]
        op = O.default_params(chunk_bit_depth=args.bits, chunks_per_frame=K, band_all=1)
        t0 = time.perf_counter()
        with ThreadPoolExecutor(len(probe)) as ex:
            refs = list(ex.map(lambda i: O.encode_frame(frames[i], op), probe))
        gblob, gsz = dev_stream, dev_sizes
        goff = np.concatenate([[0], np.cumsum(gsz)])
        same = []
        for i, ref in zip(probe, refs):
            r = res[i]
            ok = ((r.N, r.R, r.divider, r.passes, r.err, r.overfull) == (ref.N, ref.R, ref.divider, ref.passes, ref.err, ref.overfull)
                  and np.array_equal(r.dict, ref.dict) and np.array_equal(r.datten, ref.datten)
                  and np.array_equal(r.index, ref.index) and np.array_equal(r.attr, ref.attr)
                  and gblob[goff[i]:goff[i + 1]] == O.write_frame(ref, CHANNELS, CHUNK_SIZE, args.bits, SAMPLE_RATE))
            same.append(bool(ok))
        parity = {"frames": probe, "identical": all(same), "per_frame": same, "passes": [r.passes for r in refs],
                  "oracle_s": round(time.perf_counter() - t0, 1),
                  "what": "frames of the timed batch vs oracle.encode_frame (N=%d, K=%d, <=100 passes): divider, passes, Double "
                          "error sum, dictionary, attenuations, indexes, attributes and .gsc bytes" % (refs[0].N, K)}
        assert parity["identical"], "GPU result differs from the oracle: %r" % (parity,)

    # extra legs (driver-visible): BASELINE.json configs[2] (K=256 / 8-bit) and configs[4] (1 h of 48 kHz stereo = 900 frames,
    # STRONG scaling: the one stream's frames are split over the ranks)
    extras = {}
    if not args.no_extras and args.mode == "online":
        def timed_dev(devbuf, lay, prm, nsteps=1):
            ctx.encode_frames_dev(devbuf.data_ptr(), lay, prm)     # warm-up (buffers of this shape)
            ctx.synchronize()
            barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(stream)
            for _ in range(nsteps):
                with torch.cuda.stream(stream):
                    flush.zero_()
                ctx.encode_frames_dev(devbuf.data_ptr(), lay, prm)
            a1.record(stream)
            ctx.synchronize()
            barrier()
            return max_over_ranks(a0.elapsed_time(a1)) / nsteps
        # -- k256
        p256 = sc.default_params(chunk_bit_depth=8, chunks_per_frame=256)
        ms = timed_dev(dev, layout, p256)
        r256 = ctx.fetch_results(layout, p256)
        km = ctx.stage_busy_ms("kmeans")
        fl = sum(2.0 * r.N * 256 * D * r.passes for r in r256)
        extras["k256"] = {"config": "BASELINE.json configs[2] shape: ChunkCount=256, 8-bit chunks, same %d frames per GPU" % F,
                          "value": total_audio / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms,
                          "online_passes_median": statistics.median([r.passes for r in r256]),
                          "k_online_dense_tflops": fl / (km * 1e-3) / 1e12 if km > 0 else None,
                          "k_online_frac_of_fp32_peak": fl / (km * 1e-3) / 1e12 / fp32_peak if km > 0 and fp32_peak else None,
                          "stages_ms": {k: round(v, 3) for k, v in ctx.stats()["stage_ms"].items()}}
        # -- strong_1h
        n1h = 900
        mine = list(range(rank, n1h, world))
        base48 = make_frames(min(len(mine), 64), FRAME_SECONDS, seed=777 + rank, sample_rate=48000)
        f48 = [base48[i % len(base48)] for i in range(len(mine))]
        S48 = f48[0].shape[1]
        h48 = torch.from_numpy(np.stack(f48)).pin_memory()
        d48 = h48.to("cuda", non_blocking=True)
        torch.cuda.synchronize()
        lay48 = [(i * CHANNELS * S48, S48, CHANNELS, S48) for i in range(len(mine))]
        ms = timed_dev(d48, lay48, params)
        extras["strong_1h"] = {"config": "BASELINE.json configs[4]: one synthetic 1-hour 48 kHz stereo stream = 900 frames of 4 s "
                                         "(N=96,000 chunks, K=%d, %d-bit), frames split over %d rank(s)" % (K, args.bits, world),
                               "scaling": "strong", "frames_per_rank": len(mine), "value": 3600.0 / (ms * 1e-3), "unit": UNIT,
                               "ms_per_step": ms}
        del d48, h48
        # -- split_frame: BASELINE.json configs[3], the only collective of the encoder (inside the library, NCCL)
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        from split_frame import run_split

        def bcast(b):
            obj = [b]
            dist.broadcast_object_list(obj, src=0)
            return obj[0]
        extras["split_frame"] = run_split(ctx, rank, world, 1 << 20, 4096, 10, bcast, max_over_ranks)

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        cf = make_frames(cores, args.cpu_sample_seconds, seed=4321)
        dt, cres = cpu_encode_sample(cf, K, args.bits, cores, args.cpu_search)
        cpu = {"value": sum(f.shape[1] for f in cf) / SAMPLE_RATE / dt, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": cpu_sample_text(cores, args.cpu_sample_seconds, cres, K, args.cpu_search, f", {dt:.1f} s wall")}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, F, FRAME_SECONDS),
            "e2e": e2e, "gpu_launches": int(launches), "clocks": clk, "roofline": roofline, "cpu_baseline": cpu,
            "parity_check": parity, "lloyd_mode": lloyd, **extras,
            "stages_ms": {k: round(v, 3) for k, v in stage_acc.items()},
            "online_passes": {"min": min(passes), "median": statistics.median(passes), "max": max(passes)},
            "chunks_per_frame_N": Ns[0],
            "nn_queries_per_s": sum_over_ranks(float(sum(Ns))) / (stage_acc["knnfit"] * 1e-3) if stage_acc["knnfit"] > 0 else None,
        }
        print(json.dumps(line), flush=True)
    else:
        # keep collective call counts aligned with rank 0
        sum_over_ranks(float(sum(Ns)))
    ctx.close()
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
