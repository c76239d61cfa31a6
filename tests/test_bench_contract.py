"""bench.py's JSON line and its --dump-outputs files: the reference arm on the CPU, the GPU arm on a B200."""
import json
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_contract():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--cpu-sample-seconds", "0.15", "--chunks-per-frame", "256"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "audio-s/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "workload" in d["config"]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"], capture_output=True,
                       text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def _bench(args, out_dir, timeout):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=timeout)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    out = {p[:-4]: np.load(os.path.join(out_dir, p)) for p in sorted(os.listdir(out_dir))}
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    return d, out


def _split(out, key, col):
    """the sampled frames' rows of a concatenated array (col 0 of frame_scalars = N, col 1 = R)"""
    n = out["frame_scalars"][out["sample_frames"].astype(int), col].astype(int)
    return np.split(out[key], np.cumsum(n)[:-1])


def test_reference_arm_dump_outputs_repeat(tmp_path):
    """--dump-outputs writes the last timed step's frame results; the same arguments give the same files."""
    args = ["--impl", "reference", "--steps", "2", "--warmup", "0", "--cpu-sample-seconds", "0.15", "--chunks-per-frame", "256"]
    d, a = _bench(args, tmp_path / "a", 600)
    _, b = _bench(args, tmp_path / "b", 600)
    assert d["steps"] == 2 and sorted(a) == sorted(b) == ["attr", "datten", "dict", "frame_scalars", "index", "sample_frames"]
    assert all(np.array_equal(a[k], b[k]) for k in a)
    sc = a["frame_scalars"]
    assert sc.shape == (d["cpu_baseline"]["cores"], 6) and np.all(sc[:, 0] == d["sample"]["chunks_per_frame_N"])
    assert len(a["index"]) == sc[a["sample_frames"].astype(int), 0].sum() and a["dict"].shape[1] == 4
    assert all(len(x) and x.max() < r for x, r in zip(_split(a, "index", 0), sc[a["sample_frames"].astype(int), 1]))


@pytest.mark.gpu
def test_gpu_arm_dump_outputs_are_the_oracles(tmp_path):
    """The GPU arm's dump holds what the device-resident path computed for the bench's own frames: the oracle's
    results and .gsc bytes, frame for frame."""
    from oracle import gsc_oracle as O
    import bench
    K, bits, F = 256, 8, 3
    d, out = _bench(["--frames", str(F), "--steps", "2", "--warmup", "1", "--chunks-per-frame", str(K), "--bits", str(bits),
                     "--no-cpu-baseline", "--no-e2e", "--no-lloyd", "--no-extras", "--no-parity"], tmp_path, 900)
    assert d["steps"] == 2 and out["sample_frames"].tolist() == list(range(F))
    frames = bench.make_frames(F, bench.FRAME_SECONDS, seed=1234)
    op = O.default_params(chunk_bit_depth=bits, chunks_per_frame=K, band_all=1)
    with ThreadPoolExecutor(F) as ex:
        refs = list(ex.map(lambda f: O.encode_frame(f, op), frames))
    want = [O.write_frame(r, bench.CHANNELS, bench.CHUNK_SIZE, bits, bench.SAMPLE_RATE) for r in refs]
    assert np.array_equal(out["frame_scalars"], [[r.N, r.R, r.divider, r.passes, r.err, r.overfull] for r in refs])
    for k, col in (("index", 0), ("attr", 0), ("dict", 1), ("datten", 1)):
        assert all(np.array_equal(g, getattr(r, k)) for g, r in zip(_split(out, k, col), refs)), k
    assert out["gsc_sizes"].tolist() == [len(w) for w in want]
    assert out["gsc_bytes"].astype(np.uint8).tobytes() == b"".join(want)
