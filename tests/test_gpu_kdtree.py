"""kmeans_mode 3: KNNScanReduce and KNNFit through the reference's ANN kd-tree (csrc/gsc_kdtree.cuh) against the
oracle's restatement (gsc_ref_knn_scan_reduce_kdtree, gsc_ref_knnfit_kdtree, encode_frame(kmeans_mode=3)).
Every comparison is bit-exact; float arrays by bit pattern, NaN-aware where centroids can be NaN."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from tests.golden_util import EXCERPTS as GOLD, FULL, ids, load_full

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THREADS = max(1, min(32, os.cpu_count() or 1))


def _same_f32(a, b):
    a = np.asarray(a, np.float32)
    b = np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb])


def _audio(seconds, sr=44100, ch=1, seed=7, cs=4):
    from soundchunks_b200.synth import synth_audio
    a = synth_audio(seconds, sr, ch, seed)
    return np.ascontiguousarray(a[:, : a.shape[1] // cs * cs])


def _quiet(a):
    """digital silence and very quiet stretches spliced in: many duplicate points"""
    a = a.copy()
    n = a.shape[1]
    a[:, n // 5: n // 5 + n // 10] = 0
    a[:, n // 2: n // 2 + n // 8] //= 512
    return a


# ---- CPU ---------------------------------------------------------------------------------------------------------
def test_kdtree_host_option():
    from soundchunks_b200 import host
    host.load_host_library()
    assert host.default_options("-kdtree").kmeans_mode == 3
    assert host.default_options().kmeans_mode == 0


def test_kdtree_kernels_compile_without_spills(tmp_path):
    """The kd-tree kernels build for sm_100a with no register spills (their stacks and k-lists are local arrays)."""
    import subprocess
    from soundchunks_b200 import build
    src = os.path.join(build.CSRC, "gsc_api.cu")
    cmd = [build.nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false",
           "-Xptxas", "-v", "-cubin", "-o", str(tmp_path / "gsc_api.cubin"), src]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    cur, seen = None, set()
    for line in (r.stdout + r.stderr).splitlines():
        if "Compiling entry function" in line:
            cur = line.split("'")[1]
        elif cur and "k_kdt" in cur and "spill stores" in line:
            seen.add(cur)
            assert " 0 bytes spill stores" in line, (cur, line)
    assert len(seen) == 2 + 3 + 3          # k_kdt_scan<4, 8>, k_kdt_fit_build / k_kdt_fit <2, 4, 8>


# ---- GPU: k-means stage ------------------------------------------------------------------------------------------
def _features(oracle, seconds, ch, seed, cs, bits=12, quiet=True):
    pcm = _audio(seconds, 44100, ch, seed, cs)
    if quiet:
        pcm = _quiet(pcm)
    div = oracle.find_attenuation_divider(pcm, cs, bits)
    return oracle.make_chunks(pcm, cs, bits, div)[3]


SCAN_CASES = [(1, 8, 5, 0.1), (33, 8, 100, 0.3), (256, 8, 100, 0.5), (256, 4, 40, 0.5), (700, 4, 12, 0.6),
              (700, 8, 1, 0.6), (4096, 8, 3, 1.0), (4096, 4, 2, 1.0)]


@pytest.mark.gpu
@pytest.mark.parametrize("serial", [0, 1], ids=["speculative", "serial"])
@pytest.mark.parametrize("K,D,passes,seconds", SCAN_CASES)
def test_kdtree_scan_reduce_matches_oracle(ctx, oracle, K, D, passes, seconds, serial):
    X = _features(oracle, seconds, 2, 40 + K, D // 2)
    cen0, _, _ = oracle.yakmo(X, K)
    ref = oracle.knn_scan_reduce_kdtree(X, cen0, 3, passes)
    ctx.set_debug(ctx.DBG_KDTREE_SERIAL if serial else 0)
    try:
        got = ctx.knn_scan_reduce_kdtree(X, cen0, 3, passes)
    finally:
        ctx.set_debug(0)
    assert (got[2], got[3]) == (ref[2], ref[3])
    assert np.array_equal(got[1], ref[1]) and _same_f32(got[0], ref[0])


@pytest.mark.gpu
@pytest.mark.parametrize("serial", [0, 1], ids=["speculative", "serial"])
def test_kdtree_scan_reduce_nan_start(ctx, oracle, serial):
    """An empty seed cell gives NaN centroids (full_60_f0_k4096_12): the tree is built and searched with NaN rows."""
    pcm, sr, bits, K, scal, hs, hist = load_full(os.path.join(ROOT, "tests", "golden", "full_60_f0_k4096_12.npz"))
    div = oracle.find_attenuation_divider(pcm, 4, bits)
    X = oracle.make_chunks(pcm, 4, bits, div)[3]
    cen0, _, _ = oracle.yakmo(X, K)
    assert np.isnan(cen0).any()
    ref = oracle.knn_scan_reduce_kdtree(X, cen0, 3, 2)
    ctx.set_debug(ctx.DBG_KDTREE_SERIAL if serial else 0)
    try:
        got = ctx.knn_scan_reduce_kdtree(X, cen0, 3, 2)
    finally:
        ctx.set_debug(0)
    assert got[2] == ref[2] and (got[3] == ref[3] or (np.isnan(got[3]) and np.isnan(ref[3])))
    assert np.array_equal(got[1], ref[1]) and _same_f32(got[0], ref[0])


# ---- GPU: KNNFit stage -------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("path", GOLD, ids=ids(GOLD))
def test_kdtree_knnfit_on_excerpts(ctx, oracle, path):
    g = np.load(path)
    pcm, bits, div = g["pcm"], int(g["bits"]), int(g["divider"])
    raw = oracle.make_chunks(pcm, 4, bits, div)[0]
    ref = oracle.knnfit_kdtree(g["dict_q"], g["dict_atten"], raw, bits, div)
    got = ctx.knnfit_kdtree(g["dict_q"], g["dict_atten"], pcm, 4, bits, div)
    assert np.array_equal(got["best"], ref["best"]) and np.array_equal(got["use"], ref["use"])


@pytest.mark.gpu
@pytest.mark.parametrize("cs", [2, 4])
def test_kdtree_knnfit_large_dictionary(ctx, oracle, cs):
    """R = 4096: 16,384 variant rows in the tree."""
    pcm = _quiet(_audio(1.2, 44100, 2, 61, cs))
    raw, attr, atten, feat, dst = oracle.make_chunks(pcm, cs, 12, 7)
    labels = np.random.default_rng(9).integers(0, 4096, len(feat)).astype(np.int32)
    d = oracle.build_dictionary(labels, raw, attr, 4096, 12, 7)
    ref = oracle.knnfit_kdtree(d["dict"], d["datten"], raw, 12, 7)
    got = ctx.knnfit_kdtree(d["dict"], d["datten"], pcm, cs, 12, 7)
    assert np.array_equal(got["best"], ref["best"]) and np.array_equal(got["use"], ref["use"])


# ---- GPU: whole frames -------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def full_refs(oracle):
    """oracle.encode_frame(kmeans_mode=3) of every full-frame fixture, computed in parallel (seconds per frame)."""
    def one(path):
        pcm, sr, bits, K, *_ = load_full(path)
        return oracle.encode_frame(pcm, chunk_bit_depth=bits, chunks_per_frame=K, kmeans_mode=3)
    with ThreadPoolExecutor(THREADS) as ex:
        return dict(zip(FULL, ex.map(one, FULL)))


def _same_frame(r, ref):
    assert (r.N, r.R, r.divider, r.passes, r.overfull) == (ref.N, ref.R, ref.divider, ref.passes, 0)
    assert r.err == ref.err or (np.isnan(r.err) and np.isnan(ref.err))
    assert np.array_equal(r.dict, ref.dict) and np.array_equal(r.datten, ref.datten)
    assert np.array_equal(r.index, ref.index) and np.array_equal(r.attr, ref.attr)


@pytest.mark.gpu
@pytest.mark.parametrize("path", FULL, ids=ids(FULL))
def test_kdtree_full_frames(ctx, oracle, full_refs, path):
    pcm, sr, bits, K, *_ = load_full(path)
    ref = full_refs[path]
    r = ctx.encode_frames([pcm], chunk_bit_depth=bits, chunks_per_frame=K, kmeans_mode=3)[0]
    _same_frame(r, ref)
    blob, sizes = ctx.fetch_stream(1, sr)
    assert bytes(blob) == oracle.write_frame(ref, pcm.shape[0], 4, bits, sr)


@pytest.mark.gpu
def test_kdtree_batches_both_lanes_and_device_path(ctx, oracle):
    """A batch of >= 16 frames (two internal streams) with mixed lengths and a passthrough frame: every frame equals
    its single-frame encode; the device-resident path gives the same bytes as the host-buffer path."""
    import soundchunks_b200 as sc
    import torch
    frames = [_quiet(_audio(0.08 + 0.01 * (i % 5), 48000, 1 + (i % 2), 700 + i)) for i in range(18)]
    frames[5] = _audio(0.004, 48000, 2, 5)                       # passthrough frame (N <= K) in the odd lane
    kw = dict(chunk_bit_depth=12, chunks_per_frame=256, kmeans_mode=3)
    batch = ctx.encode_frames(frames, **kw)
    blob_host, sizes_host = ctx.fetch_stream(len(frames), 48000)
    for i, f in enumerate(frames):
        one = ctx.encode_frames([f], **kw)[0]
        b = batch[i]
        assert (b.N, b.R, b.divider, b.passes, b.err, b.overfull) == (one.N, one.R, one.divider, one.passes, one.err, one.overfull)
        assert np.array_equal(b.dict, one.dict) and np.array_equal(b.datten, one.datten)
        assert np.array_equal(b.index, one.index) and np.array_equal(b.attr, one.attr)
    for i in (0, 5):
        _same_frame(batch[i], oracle.encode_frame(frames[i], **kw))
    flat = np.concatenate([f.ravel() for f in frames])
    dev = torch.from_numpy(flat).to("cuda")
    layout, off = [], 0
    for f in frames:
        layout.append((off, f.shape[1], f.shape[0], f.shape[1]))
        off += f.size
    p = sc.default_params(**kw)
    ctx.encode_frames_dev(dev.data_ptr(), layout, p)
    res = ctx.fetch_results(layout, p)
    blob_dev, sizes_dev = ctx.fetch_stream(len(frames), 48000)
    assert bytes(blob_dev) == bytes(blob_host) and np.array_equal(sizes_dev, sizes_host)
    for a, b in zip(res, batch):
        assert np.array_equal(a.index, b.index) and (a.passes, a.err) == (b.passes, b.err)


@pytest.mark.gpu
def test_kdtree_speculation_counters(ctx, oracle):
    """The speculative kernel commits several points per round; the serial one exactly one."""
    pcm = _audio(1.0, 44100, 2, 12)
    kw = dict(chunk_bit_depth=12, chunks_per_frame=1024, kmeans_mode=3)
    r = ctx.encode_frames([pcm], **kw)[0]
    c = ctx.online_counters(1)[0]
    assert c[1] == r.N * r.passes and c[2] >= c[1] and c[1] > 2 * c[0]
    ctx.set_debug(ctx.DBG_KDTREE_SERIAL)
    try:
        s = ctx.encode_frames([pcm], **kw)[0]
        cs = ctx.online_counters(1)[0]
    finally:
        ctx.set_debug(0)
    assert cs[0] == cs[1] == cs[2] == s.N * s.passes
    _same_frame(s, r)


@pytest.mark.gpu
def test_kdtree_refuses_chunk_size_8(ctx):
    import soundchunks_b200 as sc
    with pytest.raises(sc.GscError):
        ctx.encode_frames([_audio(0.2, 44100, 1, 3, 8)], chunk_size=8, chunk_bit_depth=12, chunks_per_frame=256, kmeans_mode=3)


@pytest.mark.gpu
def test_kdtree_host_encode_pcm(oracle):
    """libgsc_host.so with -kdtree == the oracle's mode-3 frames over the planner's frame starts."""
    from soundchunks_b200 import host
    sr = 44100
    pcm = _audio(2.2, sr, 2, 29)[:, : int(2.2 * sr) - 2]
    o = host.default_options("-cbd12", "-kdtree", "-cpf256", "-fl700")
    blob, rep = host.encode_pcm(pcm, sr, o)
    ref_blob, ref_frames, starts, padded = oracle.encode_pcm(pcm, sr, chunk_bit_depth=12, chunks_per_frame=256,
                                                            frame_length_ms=700.0, kmeans_mode=3, threads=THREADS)
    assert rep["frames"] == len(ref_frames) >= 3
    assert blob == ref_blob
