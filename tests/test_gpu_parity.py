"""GPU parity: every stage of libgsc_cuda.so against the CPU oracle on the same seeded inputs.

Bit-exact for integer/byte/index work and for every float path whose operation
order the reference fixes (distances, online updates, means); 1e-4 relative for
the Lloyd substitution (BASELINE.json).  All calls go through the C ABI.
"""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from soundchunks_b200.synth import synth_audio  # noqa: E402


def _same_f32(a, b):
    """bit-identical floats; NaNs compare equal whatever their payload (x86 0/0 and CUDA 0/0 differ in it)"""
    a = np.asarray(a, np.float32)
    b = np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb])


def _audio(seconds, sr=44100, ch=1, seed=7, cs=4):
    a = synth_audio(seconds, sr, ch, seed)
    S = a.shape[1] // cs * cs
    return np.ascontiguousarray(a[:, :S])


def _quiet(a, seed=3):
    """Splice digital silence and very quiet stretches in (the hihat.wav-like case)."""
    a = a.copy()
    n = a.shape[1]
    a[:, n // 5: n // 5 + n // 10] = 0
    a[:, n // 2: n // 2 + n // 8] //= 512
    return a


def test_find_attenuation_divider(ctx, oracle):
    for ch, bits, seed in [(1, 12, 1), (2, 8, 2), (2, 12, 3)]:
        pcm = _quiet(_audio(0.25, 48000, ch, seed))
        d_ref, v_ref = oracle.find_attenuation_divider(pcm, 4, bits, return_v=True)
        d_gpu, v_gpu = ctx.find_attenuation_divider(pcm, 4, bits, return_v=True)
        assert d_gpu == d_ref
        assert np.array_equal(v_gpu, v_ref), "Double sums must match bit for bit"
    z = np.zeros((1, 4096), np.int16)     # digital silence: all v = 0 -> first divider wins
    assert ctx.find_attenuation_divider(z, 4, 12) == oracle.find_attenuation_divider(z, 4, 12) == 1


def test_make_chunks(ctx, oracle):
    for ch, bits, div, seed in [(1, 12, 6, 1), (2, 8, 3, 2), (2, 12, 64, 5)]:
        pcm = _quiet(_audio(0.5, 48000, ch, seed))
        raw, attr, atten, feat, dst = oracle.make_chunks(pcm, 4, bits, div)
        g_attr, g_atten, g_feat, g_dst = ctx.make_chunks(pcm, 4, bits, div)
        assert np.array_equal(g_attr, attr)
        assert np.array_equal(g_atten, atten)
        assert np.array_equal(g_dst, dst)
        # DCT half: pure +,* on host-computed tables; cepstral half: the shared correctly-rounded logarithm
        # (csrc/gsc_log.h, the same IEEE operations on both sides) -> all eight features bit exact
        assert np.array_equal(g_feat.view(np.uint32), feat.view(np.uint32))


def _features(oracle, seconds=0.5, ch=1, seed=11, sr=44100, cs=4):
    pcm = _quiet(_audio(seconds, sr, ch, seed))
    raw, attr, atten, feat, dst = oracle.make_chunks(pcm, cs, 12, 6)
    return pcm, raw, attr, feat


@pytest.mark.parametrize("K,seconds", [(64, 0.1), (256, 0.25), (1024, 0.5)])
def test_yakmo_seeding(ctx, oracle, K, seconds):
    pcm, raw, attr, feat = _features(oracle, seconds)
    c_ref, l_ref, s_ref = oracle.yakmo(feat, K)
    c_gpu, l_gpu, s_gpu = ctx.yakmo(feat, K)
    assert np.array_equal(s_gpu, s_ref), "seed sequence"
    assert _same_f32(c_gpu, c_ref), "means over the seed cells (NaN for empty cells included)"
    assert np.array_equal(l_gpu, l_ref), "reassignment labels"


def test_yakmo_seeding_full_size_and_scan_modes(ctx, oracle):
    """Full-size frame (N ~ 96k, K = 4096): the incremental seeding kernel (window summaries + exact chain,
    gsc_seed.cuh) must give the oracle's seed sequence, and so must the two cross-check evaluations (every step a
    block-wide exact scan of all points; a one-warp serial chain)."""
    pcm = _quiet(_audio(4.0, 48000, 2, 77))
    raw, attr, atten, feat, dst = oracle.make_chunks(pcm, 4, 12, 6)
    c_ref, l_ref, s_ref = oracle.yakmo(feat, 4096)
    c_gpu, l_gpu, s_gpu = ctx.yakmo(feat, 4096)
    assert np.array_equal(s_gpu, s_ref), f"first divergence at seed {int(np.argmax(s_gpu != s_ref))}"
    assert _same_f32(c_gpu, c_ref) and np.array_equal(l_gpu, l_ref)
    c3, l3, s3 = ctx.yakmo(feat[:20000], 300)
    for flag in (ctx.DBG_SEED_FULLSCAN, ctx.DBG_SEED_SERIAL):
        ctx.set_debug(flag)
        try:
            c2, l2, s2 = ctx.yakmo(feat[:20000], 300)
        finally:
            ctx.set_debug(0)
        assert np.array_equal(s2, s3) and _same_f32(c2, c3) and np.array_equal(l2, l3)
    ctx.set_debug(ctx.DBG_SEED_FULLSCAN)
    try:
        c4, l4, s4 = ctx.yakmo(feat, 4096)
    finally:
        ctx.set_debug(0)
    assert np.array_equal(s4, s_ref) and _same_f32(c4, c_ref)


@pytest.mark.parametrize("kind", ["ragged", "silence_runs", "duplicates", "tiny"])
def test_yakmo_seeding_edge_cases(ctx, oracle, kind):
    """Inputs that stress the prefix-sum machinery: window-ragged N, long runs of zero distances (digital silence:
    duplicate points), massively duplicated chunks, and N barely above K."""
    rng = np.random.default_rng(17)
    pcm = _quiet(_audio(0.45, 44100, 1, 31))
    if kind == "silence_runs":
        pcm = pcm.copy(); pcm[:, 3000:9000] = 0; pcm[:, 12000:12800] = 0
    if kind == "duplicates":
        pcm = np.ascontiguousarray(np.tile(pcm[:, :2000], (1, 9)))
    raw, attr, atten, feat, dst = oracle.make_chunks(pcm, 4, 12, 6)
    if kind == "ragged":
        feat = np.ascontiguousarray(feat[:4099])
    K = {"ragged": 300, "silence_runs": 256, "duplicates": 200, "tiny": 64}[kind]
    if kind == "tiny":
        feat = np.ascontiguousarray(feat[:65])
    c_ref, l_ref, s_ref = oracle.yakmo(feat, K)
    c_gpu, l_gpu, s_gpu = ctx.yakmo(feat, K)
    assert np.array_equal(s_gpu, s_ref), f"{kind}: first divergence at seed {int(np.argmax(s_gpu != s_ref))}"
    assert _same_f32(c_gpu, c_ref) and np.array_equal(l_gpu, l_ref)


@pytest.mark.parametrize("shape", ["256x2", "256x3", "128x4", "128x6"])
def test_yakmo_seeding_cta_shapes(ctx, oracle, shape, monkeypatch):
    """k_seed2 is instantiated for four CTA shapes (threads x resident CTAs per SM; the library picks by batch size,
    GSC_SEED_SHAPE overrides): each must give the oracle's seed sequence."""
    pcm, raw, attr, feat = _features(oracle, 0.6)
    c_ref, l_ref, s_ref = oracle.yakmo(feat, 700)
    monkeypatch.setenv("GSC_SEED_SHAPE", shape)
    c_gpu, l_gpu, s_gpu = ctx.yakmo(feat, 700)
    assert np.array_equal(s_gpu, s_ref), f"{shape}: first divergence at seed {int(np.argmax(s_gpu != s_ref))}"
    assert _same_f32(c_gpu, c_ref) and np.array_equal(l_gpu, l_ref)


def test_yakmo_random_init_and_iters(ctx, oracle):
    pcm, raw, attr, feat = _features(oracle, 0.1)
    c_ref, l_ref, s_ref = oracle.yakmo(feat, 32, init_type=0, max_iter=0)
    c_gpu, l_gpu, s_gpu = ctx.yakmo(feat, 32, init_type=0, max_iter=0)
    assert np.array_equal(s_gpu, s_ref)
    assert _same_f32(c_gpu, c_ref)
    assert np.array_equal(l_gpu, l_ref)


# D = 8 (-cs 4) and D = 4 (-cs 2, its own features): both sides of every CTA-shape bucket of k_online (gsc_api.cu
# stage_online: K <= 256 / 512 / 1024 / 2048 / 4096)
ONLINE_CASES = [(256, 0.25, 100, 8), (100, 0.1, 7, 8), (4096, 0.6, 4, 8), (700, 0.3, 20, 8), (1500, 0.4, 8, 8), (400, 0.2, 12, 8)]
ONLINE_CASES += [(K, 0.3, 6, D) for D in (4, 8) for K in (257, 512, 513, 1024, 1025, 2048, 2049, 4096)]


@pytest.mark.parametrize("K,seconds,passes,D", ONLINE_CASES)
def test_online_kmeans_bit_exact(ctx, oracle, K, seconds, passes, D):
    """k_online (and k_online_warp for K <= 256) with its filter and scoring every centroid exactly
    (GSC_DBG_ONLINE_EXACT): the oracle bit for bit."""
    pcm, raw, attr, feat = _features(oracle, seconds, ch=2 if K >= 2048 else 1, cs=D // 2)
    assert len(feat) > K
    c0, _, _ = oracle.yakmo(feat, K)
    c_ref, l_ref, it_ref, err_ref = oracle.knn_scan_reduce(feat, c0, 3, passes)
    for flag in (0, ctx.DBG_ONLINE_EXACT):
        ctx.set_debug(flag)
        try:
            c_gpu, l_gpu, it_gpu, err_gpu = ctx.knn_scan_reduce(feat, c0, 3, passes)
        finally:
            ctx.set_debug(0)
        assert it_gpu == it_ref, flag
        assert np.array_equal(l_gpu, l_ref), flag
        assert np.array_equal(c_gpu.view(np.uint32), c_ref.view(np.uint32)), flag
        assert err_gpu == err_ref, flag


@pytest.mark.parametrize("K,seconds,passes,D", [(256, 0.25, 100, 8), (100, 0.1, 9, 8), (33, 0.1, 30, 8), (200, 0.15, 12, 4)])
def test_online_small_dictionary_both_kernels(ctx, oracle, K, seconds, passes, D, monkeypatch):
    """K <= 256 runs one warp per frame with the codebook in registers (k_online_warp; GSC_OW_WARPS=2 splits the
    codebook over two warps); the batched CTA-per-frame kernel stays available (GSC_DBG_ONLINE_BATCHED): all three
    must be the oracle bit for bit."""
    pcm, raw, attr, feat = _features(oracle, seconds)
    feat = np.ascontiguousarray(feat[:, :D])
    c0, _, _ = oracle.yakmo(feat, K)
    ref = oracle.knn_scan_reduce(feat, c0, 3, passes)
    for flag, warps in ((0, "1"), (0, "2"), (ctx.DBG_ONLINE_BATCHED, "1")):
        monkeypatch.setenv("GSC_OW_WARPS", warps)
        ctx.set_debug(flag)
        try:
            got = ctx.knn_scan_reduce(feat, c0, 3, passes)
        finally:
            ctx.set_debug(0)
        assert got[2] == ref[2] and got[3] == ref[3], (flag, warps)
        assert np.array_equal(got[1], ref[1]) and np.array_equal(got[0].view(np.uint32), ref[0].view(np.uint32)), (flag, warps)


def test_online_kmeans_filter_equals_exhaustive(ctx, oracle):
    """The lower-bound filter must give exactly what scoring every centroid exactly gives."""
    pcm, raw, attr, feat = _features(oracle, 0.3)
    c0, _, _ = oracle.yakmo(feat, 512)
    fast = ctx.knn_scan_reduce(feat, c0, 3, 10)
    ctx.set_debug(ctx.DBG_ONLINE_EXACT)
    try:
        slow = ctx.knn_scan_reduce(feat, c0, 3, 10)
    finally:
        ctx.set_debug(0)
    assert fast[2] == slow[2] and fast[3] == slow[3]
    assert np.array_equal(fast[1], slow[1])
    assert np.array_equal(fast[0].view(np.uint32), slow[0].view(np.uint32))


@pytest.mark.parametrize("K,iters", [(256, 5), (1024, 3)])
def test_lloyd(ctx, oracle, K, iters):
    pcm, raw, attr, feat = _features(oracle, 0.5)
    c0, _, _ = oracle.yakmo(feat, K)
    c0 = np.nan_to_num(c0, nan=0.0)
    c_ref, l_ref = oracle.lloyd(feat, c0, iters)
    c_gpu, l_gpu = ctx.lloyd(feat, c0, iters)
    # 1e-4 relative (BASELINE.json); the GPU sums in the same order so it is normally exact
    scale = np.maximum(np.abs(c_ref), 1e-6)
    assert np.max(np.abs(c_gpu - c_ref) / scale) <= 1e-4
    assert np.mean(l_gpu != l_ref) < 1e-3


@pytest.mark.parametrize("pts", [2, 4, 8])
def test_assign_points_per_thread_variants(ctx, oracle, pts, monkeypatch):
    """k_assign<D, P>: the three points-per-thread instantiations (chosen by launch size) give the oracle's labels and
    distances bit for bit."""
    pcm, raw, attr, feat = _features(oracle, 0.3)
    c0, _, _ = oracle.yakmo(feat, 1000)
    l_ref, d_ref = oracle.assign(feat, c0)
    monkeypatch.setenv("GSC_ASSIGN_PTS", str(pts))
    l_gpu, d_gpu = ctx.assign(feat, c0)
    assert np.array_equal(l_gpu, l_ref)
    assert np.array_equal(d_gpu.view(np.uint32), d_ref.view(np.uint32))


def test_assign_exact(ctx, oracle):
    pcm, raw, attr, feat = _features(oracle, 0.4)
    c0, _, _ = oracle.yakmo(feat, 777)
    l_ref, d_ref = oracle.assign(feat, c0)
    l_gpu, d_gpu = ctx.assign(feat, c0)
    assert np.array_equal(l_gpu, l_ref)
    assert np.array_equal(d_gpu.view(np.uint32), d_ref.view(np.uint32))


@pytest.mark.parametrize("bits,div,K", [(12, 6, 256), (8, 3, 512)])
def test_build_dictionary(ctx, oracle, bits, div, K):
    pcm = _quiet(_audio(0.4, 48000, 2, 21))
    raw, attr, atten, feat, dst = oracle.make_chunks(pcm, 4, bits, div)
    c0, _, _ = oracle.yakmo(feat, K)
    _, labels, _, _ = oracle.knn_scan_reduce(feat, c0, 3, 3)
    ref = oracle.build_dictionary(labels, raw, attr, K, bits, div)
    gpu = ctx.build_dictionary(labels, pcm, attr, K, 4, bits, div)
    for k in ("counts", "order", "entry", "dict", "datten", "dattr"):
        assert np.array_equal(gpu[k], ref[k]), k
    assert np.array_equal(gpu["means"].view(np.uint32), ref["means"].view(np.uint32))


@pytest.mark.parametrize("bits,div,K", [(12, 6, 256), (8, 3, 512), (12, 1, 64)])
def test_knnfit(ctx, oracle, bits, div, K):
    pcm = _quiet(_audio(0.4, 44100, 1, 31))
    raw, attr, atten, feat, dst = oracle.make_chunks(pcm, 4, bits, div)
    c0, _, _ = oracle.yakmo(feat, K)
    _, labels, _, _ = oracle.knn_scan_reduce(feat, c0, 3, 3)
    d = oracle.build_dictionary(labels, raw, attr, K, bits, div)
    ref = oracle.knnfit(d["dict"], d["datten"], raw, bits, div)
    gpu = ctx.knnfit(d["dict"], d["datten"], pcm, 4, bits, div)
    assert np.array_equal(gpu["band"], ref["band"]), "epsilon-band population"
    ok = ref["band"] <= 64          # where ANN's 64-candidate truncation cannot bite
    assert np.array_equal(gpu["best"][ok], ref["best"][ok])
    # the untruncated rule is what the kernel implements everywhere
    assert np.array_equal(gpu["best"], ref["best_all"])
    if ok.all():
        assert np.array_equal(gpu["use"], ref["use"])


def test_finalize_dictionary(ctx, oracle):
    rng = np.random.default_rng(5)
    for R in (1, 2, 63, 256, 4096):
        use = rng.integers(0, 6, R).astype(np.int32)
        use[rng.integers(0, R, max(1, R // 7))] = 0
        n_ref, remap_ref, order_ref = oracle.finalize_dictionary(use)
        n_gpu, remap_gpu, order_gpu = ctx.finalize_dictionary(use)
        assert n_gpu == n_ref
        assert np.array_equal(remap_gpu, remap_ref)
        assert np.array_equal(order_gpu, order_ref)


@pytest.mark.parametrize("ch,bits,K,seconds", [(1, 12, 256, 0.3), (2, 8, 256, 0.25), (2, 12, 1024, 0.4)])
def test_encode_frames_end_to_end(ctx, oracle, ch, bits, K, seconds):
    frames = [_quiet(_audio(seconds, 48000, ch, 100 + i)) for i in range(3)]
    frames.append(_audio(0.01, 48000, ch, 9))            # N <= K: passthrough frame (enc:891-912)
    res = ctx.encode_frames(frames, chunk_bit_depth=bits, chunks_per_frame=K)
    for f, r in zip(frames, res):
        # band_all: the epsilon-band rule over all rows, the library's contract (== the 64-row rule when overfull == 0)
        ref = oracle.encode_frame(f, chunk_bit_depth=bits, chunks_per_frame=K, band_all=1)
        assert r.divider == ref.divider and r.N == ref.N
        assert r.passes == ref.passes and r.err == ref.err
        assert r.R == ref.R and r.overfull == ref.overfull
        assert np.array_equal(r.dict, ref.dict)
        assert np.array_equal(r.datten, ref.datten)
        assert np.array_equal(r.index, ref.index)
        assert np.array_equal(r.attr, ref.attr)
        # decode round trip through the oracle's writer + reference decoder restatement
        blob = oracle.write_frame(oracle.FrameResult(r.N, r.R, r.divider, r.passes, r.err, r.dict, r.datten,
                                                     r.index, r.attr, r.overfull), ch, 4, bits, 48000)
        dec, sr = oracle.decode(blob)
        assert dec.shape == f.shape and sr == 48000
        assert oracle.snr_db(f, dec) > 10.0


def test_legacy_abi(ctx, oracle):
    import soundchunks_b200 as sc
    pcm, raw, attr, feat = _features(oracle, 0.1)
    c_ref, l_ref, _ = oracle.yakmo(feat, 48)
    c_gpu, l_gpu = sc.legacy_yakmo(feat, 48)
    assert np.array_equal(c_gpu.view(np.uint32), c_ref.view(np.uint32))
    assert np.array_equal(l_gpu, l_ref)
    pts = np.nan_to_num(c_ref, nan=0.0)
    ann = sc.LegacyAnn(pts)
    for i in (0, 17, 300):
        idx, err = ann.search(feat[i])
        l, d = oracle.assign(feat[i:i + 1], pts)
        assert idx == l[0] and np.float32(err) == d[0]
    idxs, errs = ann.pri_search_multi(feat[5], 16)
    dd = ((feat[5][None, :] - pts) ** 2)
    # exact float order: recompute with the oracle distance for each returned index
    assert len(set(idxs.tolist())) == 16 and np.all(np.diff(errs) >= 0)
    l, d = oracle.assign(feat[5:6], pts)
    assert idxs[0] == l[0] and errs[0] == d[0]
    ann.close()
    assert dd.shape[0] == pts.shape[0]


def test_two_stream_batches_match_single_frames(ctx):
    """Batches of >= 16 frames run on two internal streams (even / odd frames): results must be the frames'
    own results, in the caller's order; the stage busy time is the union of the two lanes' intervals."""
    frames = [_quiet(_audio(0.08 + 0.01 * (i % 5), 48000, 1 + (i % 2), 300 + i)) for i in range(21)]
    frames[7] = _audio(0.004, 48000, 2, 5)                       # passthrough frame in the odd lane
    batch = ctx.encode_frames(frames, chunk_bit_depth=12, chunks_per_frame=256)
    st = ctx.stats()["stage_ms"]
    busy = ctx.stage_busy_ms("kmeans")
    assert 0.0 < busy <= st["kmeans"] + 1e-6                     # union <= sum of the lanes
    for i in (0, 1, 7, 8, 19, 20):
        one = ctx.encode_frames([frames[i]], chunk_bit_depth=12, chunks_per_frame=256)[0]
        b = batch[i]
        assert (b.N, b.R, b.divider, b.passes, b.err, b.overfull) == (one.N, one.R, one.divider, one.passes, one.err, one.overfull)
        assert np.array_equal(b.dict, one.dict) and np.array_equal(b.datten, one.datten)
        assert np.array_equal(b.index, one.index) and np.array_equal(b.attr, one.attr)


def test_knnfit_windowed_equals_dense_on_large_dictionary(ctx, oracle):
    """The norm-window search must return what the oracle's scan over all 4R rows returns, also for R = 4096."""
    pcm = _quiet(_audio(1.2, 44100, 2, 61))
    raw, attr, atten, feat, dst = oracle.make_chunks(pcm, 4, 12, 7)
    rng = np.random.default_rng(9)
    labels = rng.integers(0, 4096, len(feat)).astype(np.int32)   # any labelling gives a valid dictionary
    d = oracle.build_dictionary(labels, raw, attr, 4096, 12, 7)
    ref = oracle.knnfit(d["dict"], d["datten"], raw, 12, 7)
    gpu = ctx.knnfit(d["dict"], d["datten"], pcm, 4, 12, 7)
    assert np.array_equal(gpu["band"], ref["band"]) and np.array_equal(gpu["best"], ref["best_all"])


@pytest.mark.parametrize("nframes,ch,bits", [(3, 1, 12), (18, 2, 8), (17, 2, 12)])
def test_device_stream_packer_and_quality(ctx, oracle, nframes, ch, bits):
    """SURVEY.md 8(f2)/(f3): .gsc bytes packed on the device == the host writer's (enc:980-1107), and the
    reconstruction error behind PsyADelta == the oracle's (enc:1862-1880); one-stream and two-stream batches."""
    from soundchunks_b200 import host
    frames = [_quiet(_audio(0.06 + 0.013 * (i % 4), 44100, ch, 500 + i)) for i in range(nframes)]
    frames[1] = _audio(0.003, 44100, ch, 77)                      # passthrough frame, tiny dictionary
    res = ctx.encode_frames(frames, chunk_bit_depth=bits, chunks_per_frame=256)
    blob, sizes = ctx.fetch_stream(nframes, 44100)
    want = [host.write_frame(r, ch, 4, bits, 44100) for r in res]
    assert sizes.tolist() == [len(w) for w in want]
    assert blob == b"".join(want)
    dec, sr = oracle.decode(blob)                                 # and the reference decoder restatement reads it
    assert sr == 44100 and dec.shape[1] == sum(f.shape[1] for f in frames)
    e2, ns = ctx.fetch_quality(nframes)
    tot = 0
    for f, r, e, n in zip(frames, res, e2, ns):
        rec = oracle.reconstruct_frame(oracle.FrameResult(r.N, r.R, r.divider, r.passes, r.err, r.dict, r.datten, r.index,
                                                          r.attr, r.overfull), ch, f.shape[1], 4, bits)
        d = f.astype(np.int64) - rec.astype(np.int64)
        assert int(e) == int((d * d).sum()) and int(n) == f.size
        tot += int(e)
    allsrc = np.concatenate([f.ravel() for f in frames])
    allrec = np.concatenate([oracle.reconstruct_frame(oracle.FrameResult(r.N, r.R, r.divider, r.passes, r.err, r.dict, r.datten,
                                                                         r.index, r.attr, r.overfull), ch, f.shape[1], 4, bits).ravel()
                             for f, r in zip(frames, res)])
    assert np.sqrt(tot / float(ns.sum())) == oracle.psy_a_delta(allsrc, allrec)


def test_split_lloyd_in_library_matches_oracle(ctx, oracle):
    """gsc_split_seed + gsc_split_lloyd (the oversized-frame entry points, NCCL communicator of one rank): the start
    is yakmo's seed sequence on the shard, the result is oracle.lloyd's within BASELINE.json's 1e-4 relative (and
    bit-identical to gsc_lloyd: Double accumulation, one rounding)."""
    import soundchunks_b200 as sc
    pcm, raw, attr, feat = _features(oracle, 1.5, ch=2, seed=5, sr=48000)
    K, iters = 512, 4
    uid = sc.Context.split_unique_id()
    ctx.split_comm_init(1, 0, uid)
    try:
        c0 = ctx.split_seed(feat, K)
        _, _, seeds = oracle.yakmo(feat, K)
        assert np.array_equal(c0.view(np.uint32), feat[seeds].view(np.uint32))
        cen, labels, ms = ctx.split_lloyd(feat, c0, iters)
    finally:
        ctx.split_comm_destroy()
    ref_cen, ref_lab = oracle.lloyd(feat, c0, iters)
    rel = np.max(np.abs(cen - ref_cen), axis=1) / np.maximum(np.max(np.abs(ref_cen), axis=1), 1e-12)
    assert rel.max() <= 1e-4 and np.mean(labels != ref_lab) < 1e-4
    g_cen, g_lab = ctx.lloyd(feat, c0, iters)
    assert np.array_equal(cen.view(np.uint32), g_cen.view(np.uint32)) and np.array_equal(labels, g_lab)
    assert ms["ms_loop"] > 0


def test_legacy_ann_sees_the_callers_live_rows(ctx, oracle):
    """ANN keeps the caller's row pointers (SURVEY.md 3.2): enc:725-746 moves Centroids[bestIdx] between queries on one
    tree and later queries must see the moved row.  Driving that loop through the legacy ABI must give what
    gsc_knn_scan_reduce gives."""
    import soundchunks_b200 as sc
    pcm, raw, attr, feat = _features(oracle, 0.06)
    feat = np.ascontiguousarray(feat[:600])
    K, D = 48, feat.shape[1]
    c0, _, _ = oracle.yakmo(feat, K)
    want = ctx.knn_scan_reduce(feat, c0, 3, 2)
    cen = np.array(c0, np.float32, copy=True)
    cnts = [np.ones(K, np.int32), np.ones(K, np.int32)]
    labels = np.zeros(len(feat), np.int32)
    for it in range(2):                                   # enc:725-761
        kdt = sc.LegacyAnn(cen, copy=False)               # rows of `cen` itself, mutated below
        err = 0.0
        for i in range(len(feat)):
            b, d2 = kdt.search(feat[i])
            rate = np.float32(1.0 / np.sqrt(float(cnts[1 - (it & 1)][b])))
            cen[b] = cen[b] + (feat[i] - cen[b]) * rate   # float32, operation by operation as enc:736-740
            labels[i] = b
            err += float(np.sqrt(np.float32(d2) / np.float32(D)))
            cnts[it & 1][b] += 1
        cnts[1 - (it & 1)][:] = 1
        kdt.close()
    assert np.array_equal(labels, want[1]) and np.array_equal(cen.view(np.uint32), want[0].view(np.uint32))
    assert err == want[3]


def test_member_lists_equal_label_scans(ctx, oracle):
    """Per-cluster sums over the stable member lists (k_group_labels, O(N)) == the per-cluster scans of all labels
    (O(K*N), GSC_DBG_LABEL_SCAN), on a frame with heavily skewed clusters (long silent stretch)."""
    pcm = _quiet(_audio(0.6, 44100, 2, 21)).copy()
    pcm[:, 5000:14000] = 0
    a = ctx.encode_frames([pcm], chunk_bit_depth=12, chunks_per_frame=1024)[0]
    sa, _ = ctx.fetch_stream(1, 44100)
    ctx.set_debug(ctx.DBG_LABEL_SCAN)
    try:
        b = ctx.encode_frames([pcm], chunk_bit_depth=12, chunks_per_frame=1024)[0]
        sb, _ = ctx.fetch_stream(1, 44100)
    finally:
        ctx.set_debug(0)
    assert (a.R, a.passes, a.err) == (b.R, b.passes, b.err) and sa == sb
    ref = oracle.encode_frame(pcm, chunk_bit_depth=12, chunks_per_frame=1024, band_all=1)
    assert sa == oracle.write_frame(ref, 2, 4, 12, 44100)


def test_divider_kernel_forms_agree(ctx, oracle):
    """k_find_divider2 (tabulated reciprocals, integer attenuation thresholds) == the straightforward kernel == the
    oracle, all 64 Double sums bit for bit; the reciprocal division is checked exhaustively."""
    assert ctx.selftest_divider_division(8) == 0 and ctx.selftest_divider_division(12) == 0
    for ch, bits, seed in [(1, 12, 1), (2, 8, 2), (2, 12, 3)]:
        pcm = _audio(0.4, 44100, ch, seed)          # full-scale: exercises the low attenuations and the clamps
        d_ref, v_ref = oracle.find_attenuation_divider(pcm, 4, bits, return_v=True)
        d2, v2 = ctx.find_attenuation_divider(pcm, 4, bits, return_v=True)
        ctx.set_debug(ctx.DBG_DIVIDER_V1)
        try:
            d1, v1 = ctx.find_attenuation_divider(pcm, 4, bits, return_v=True)
        finally:
            ctx.set_debug(0)
        assert d1 == d2 == d_ref and np.array_equal(v1, v_ref) and np.array_equal(v2, v_ref)
    v10 = ctx.find_attenuation_divider(_quiet(_audio(0.2, 44100, 1, 4)), 4, 10, return_v=True)   # other depth: plain division
    assert v10[0] == oracle.find_attenuation_divider(_quiet(_audio(0.2, 44100, 1, 4)), 4, 10)


@pytest.mark.parametrize("channels,sr,seconds,fl,vfr,kind", [(1, 44100, 21.3, 4000.0, 1.0, "music"), (2, 48000, 12.0, 700.0, 1.0, "music"),
                                                          (2, 44100, 9.0, 500.0, 0.5, "silence_lead"), (1, 32000, 6.5, 250.0, 1.0, "bursts"),
                                                          (2, 44100, 3.1, 4000.0, 1.0, "short")])
def test_frame_planner_on_device(ctx, oracle, channels, sr, seconds, fl, vfr, kind):
    """SURVEY.md 8(f1): gsc_plan_frames (power scan + boundary selection on the device, sequential Double sums
    evaluated exactly in parallel) == oracle.plan_frames (enc:1374-1425), frame start by frame start."""
    pcm = _audio(seconds, sr, channels, 41)
    S = pcm.shape[1] // 4 * 4
    pcm = np.ascontiguousarray(pcm[:, :S]).copy()
    if kind == "silence_lead":
        pcm[:, : int(2.2 * sr)] = 0                      # digital silence: the sums stay at +0 for 2.2 s
    if kind == "bursts":
        pcm[:, ::3] = (pcm[:, ::3].astype(np.int32) // 64).astype(np.int16)
        pcm[:, int(1.0 * sr):int(1.5 * sr)] = 32767      # full-scale stretch: smp > avg, terms near (and just below) zero
        pcm[:, int(3.0 * sr):int(3.2 * sr)] = -32768     # |x| > 1: slightly NEGATIVE terms
    want = oracle.plan_frames(pcm, sr, frame_length_ms=fl, vfr=vfr)
    got, st = ctx.plan_frames(pcm, sr, frame_length_ms=fl, vfr=vfr, return_stats=True)
    assert np.array_equal(got, want), (got[:8], want[:8], st)
    assert st["boundary_iterations"] <= 3 and st["exact_windows_pass1"] < st["windows_pass1"] // 4 + 64


def test_other_chunk_sizes(ctx, oracle):
    """-cs 2 (features of dimension 4) runs the same path bit for bit; -cs 8 (dimension 16) is refused loudly by the
    online k-means (its register tile is built for D <= 8) but runs in Lloyd mode."""
    import soundchunks_b200 as sc
    pcm = _quiet(_audio(0.25, 44100, 2, 61))
    r = ctx.encode_frames([pcm], chunk_size=2, chunk_bit_depth=12, chunks_per_frame=512)[0]
    blob, _ = ctx.fetch_stream(1, 44100)
    ref = oracle.encode_frame(pcm, chunk_size=2, chunk_bit_depth=12, chunks_per_frame=512, band_all=1)
    assert (r.N, r.R, r.divider, r.passes, r.err) == (ref.N, ref.R, ref.divider, ref.passes, ref.err)
    assert blob == oracle.write_frame(ref, 2, 2, 12, 44100)
    with pytest.raises(sc.GscError):
        ctx.encode_frames([pcm], chunk_size=8, chunk_bit_depth=12, chunks_per_frame=256)
    r8 = ctx.encode_frames([pcm], chunk_size=8, chunk_bit_depth=12, chunks_per_frame=256, kmeans_mode=1, lloyd_iters=3)[0]
    ref8 = oracle.encode_frame(pcm, chunk_size=8, chunk_bit_depth=12, chunks_per_frame=256, kmeans_mode=1, lloyd_iters=3, band_all=1)
    assert (r8.N, r8.divider) == (ref8.N, ref8.divider)
    dec_g, _ = oracle.decode(oracle.write_frame(oracle.FrameResult(r8.N, r8.R, r8.divider, 0, 0.0, r8.dict, r8.datten, r8.index, r8.attr, r8.overfull), 2, 8, 12, 44100))
    dec_r, _ = oracle.decode(oracle.write_frame(ref8, 2, 8, 12, 44100))
    assert abs(oracle.snr_db(pcm, dec_g) - oracle.snr_db(pcm, dec_r)) < 0.05
