"""Edges of the pruned searches and of the shapes the library dispatches, against the CPU oracle and against a plain
numpy restatement of the two rules everything rests on (nearest centroid in ANN order; the online update of
enc:699-765).

The search kernels prune with hand-tuned bounds and break ties by original index; audio rarely lands on the cases
those arguments depend on.  The generators below do: exact ties everywhere (small-integer lattices), duplicated
codebook rows, large common offsets, clusters of very different scales, long runs of identical points with K close
to N, NaN start rows.  Every float comparison is bit for bit (NaN-aware: x86 and CUDA NaN payloads differ)."""
import math
import os
import shutil
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
THREADS = max(1, min(32, os.cpu_count() or 1))


def _same_f32(a, b):
    a = np.asarray(a, np.float32)
    b = np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb])


def _same_err(a, b):
    return a == b or (np.isnan(a) and np.isnan(b))


def _audio(seconds, sr=44100, ch=1, seed=7, cs=4):
    from soundchunks_b200.synth import synth_audio
    a = synth_audio(seconds, sr, ch, seed)
    return np.ascontiguousarray(a[:, : a.shape[1] // 8 * 8])


def _quiet(a):
    a = a.copy()
    n = a.shape[1]
    a[:, n // 5: n // 5 + n // 10] = 0
    a[:, n // 2: n // 2 + n // 8] //= 512
    return a


def _features(oracle, seconds, D, seed=11, ch=1):
    """real features of dimension D (= 2 * chunk size) from quiet-spliced audio"""
    cs = D // 2
    pcm = _quiet(_audio(seconds, 44100, ch, seed))
    div = oracle.find_attenuation_divider(pcm, cs, 12)
    return np.ascontiguousarray(oracle.make_chunks(pcm, cs, 12, div)[3])


def _debug(ctx, flag, fn, *a):
    ctx.set_debug(flag)
    try:
        return fn(*a)
    finally:
        ctx.set_debug(0)


# ---- a plain restatement of the two contracts (no oracle code) ----------------------------------------------------
def np_nearest(x, C):
    """ANN order: d = 0; d = d + (x_k - c_k)^2 per dimension, left to right, float32, no FMA.  Strict < over
    ascending index: the lowest index wins ties, NaN rows never win; every row NaN -> (0, +inf)."""
    d = np.zeros(C.shape[0], np.float32)
    for k in range(C.shape[1]):
        t = np.float32(x[k]) - C[:, k]
        d = d + t * t
    d = np.where(np.isnan(d), np.float32(np.inf), d)
    j = int(np.argmin(d))
    return j, np.float32(d[j])


def np_knn_scan_reduce(X, c0, precision, max_passes):
    """enc:699-765: rate = float32(1 / sqrt(double(cnt))) with the counts of the previous pass, c + (x - c) * rate in
    float32, err the Double sum of sqrtf(d / D), stop when |err - prevErr| <= IntPower(10, -precision)."""
    X = np.asarray(X, np.float32)
    C = np.array(c0, np.float32, copy=True)
    N, D = X.shape
    K = C.shape[0]
    cnts = [np.ones(K, np.int64), np.ones(K, np.int64)]
    p = 1.0
    for _ in range(precision):
        p *= 10.0
    tol = 1.0 / p
    labels = np.zeros(N, np.int32)
    it, err = 0, 3.40282346638528860e+38
    while True:
        prev, err, odd = err, 0.0, it & 1
        for i in range(N):
            j, d = np_nearest(X[i], C)
            rate = np.float32(1.0 / math.sqrt(float(cnts[1 - odd][j])))
            C[j] = C[j] + (X[i] - C[j]) * rate
            labels[i] = j
            err += float(np.sqrt(d / np.float32(D)))
            cnts[odd][j] += 1
        cnts[1 - odd][:] = 1
        it += 1
        same = (err - prev <= tol) if err > prev else (prev - err <= tol)
        if same or it >= max_passes:
            return C, labels, it, err


def np_lloyd_exact(X, c0, iters):
    """Lloyd with exactly rounded member sums (math.fsum): every mean has a single rounding."""
    X = np.asarray(X, np.float32)
    C = np.array(c0, np.float32, copy=True)
    for _ in range(iters):
        lab = np.array([np_nearest(x, C)[0] for x in X])
        for c in np.unique(lab):
            m = X[lab == c].astype(np.float64)
            C[c] = [np.float32(math.fsum(m[:, k]) / len(m)) for k in range(X.shape[1])]
    return C, np.array([np_nearest(x, C)[0] for x in X], np.int32)


# ---- adversarial (points, start codebook) generators; every value within |x| <= 2^20 -------------------------------
def _lattice(oracle, D, K, N=3000, seed=1):
    rng = np.random.default_rng(seed)
    X = rng.integers(-3, 4, (N, D)).astype(np.float32)          # exact distances, ties everywhere
    return X, X[np.sort(rng.choice(N, K, replace=False))].copy()


def _dup_rows(oracle, D, K):
    X = _features(oracle, 0.3, D)[:3000]
    c0 = oracle.yakmo(X, K)[0]
    c0 = np.nan_to_num(c0, nan=0.0)
    rng = np.random.default_rng(2)
    idx = np.sort(rng.choice(K, 24, replace=False))
    c0[idx[:12]] = c0[idx[5]]                                   # exact duplicates at scattered indices
    base = c0[idx[20]].copy()
    for t, i in enumerate(idx[12:]):                            # near-duplicates: c0 descends as the index ascends
        c0[i] = base
        c0[i, 0] = base[0] + np.float32((len(idx) - 12 - t) * np.spacing(np.float32(max(abs(base[0]), 1e-3))))
    return X, c0


def _offset(oracle, D, K, all_dims):
    X = _features(oracle, 0.3, D, seed=5)[:3000]
    c0 = oracle.yakmo(X, K)[0]
    off = np.float32(2.0 ** 18) if all_dims else np.float32(2.0 ** 19)
    if all_dims:
        return X + off, c0 + off
    X, c0 = X.copy(), c0.copy()
    X[:, 0] += off
    c0[:, 0] += off
    return X, c0


def _scales(oracle, D, K, N=3000):
    rng = np.random.default_rng(4)
    X = np.concatenate([rng.normal(0, 1e-3, (N // 2, D)), 1e4 * rng.normal(0, 1, (N - N // 2, D)) + 3e4]).astype(np.float32)
    X = X[rng.permutation(N)]
    return X, X[np.sort(rng.choice(N, K, replace=False))].copy()


def _runs(oracle, D, K, N):
    """long runs of identical points, N = K + 1 or N < 32: whole batches pick one centroid"""
    rng = np.random.default_rng(6)
    rows = rng.integers(-2, 3, (max(3, N // 40), D)).astype(np.float32)
    X = np.repeat(rows, -(-N // len(rows)), axis=0)[:N].copy()
    X[N // 2] += 1.0
    c0 = X[np.sort(rng.choice(N, K, replace=False))].copy()
    c0[1::3] = rows[0]
    return X, c0


def _nan_rows(oracle, D, K, which):
    X = _features(oracle, 0.3, D, seed=9)[:3000]
    c0 = np.nan_to_num(oracle.yakmo(X, K)[0], nan=0.0)
    if which == "scattered":
        c0[[0, 3, K // 3, K // 2 + 1, K - 1]] = np.nan
    elif which == "cell":                                       # the 16 lowest c0: one whole cell of the sorted slots
        c0[np.argsort(c0[:, 0], kind="stable")[:16]] = np.nan
    elif which == "one_finite":
        keep = c0[K // 2].copy()
        c0[:] = np.nan
        c0[K // 2] = keep
    else:
        c0[:] = np.nan
    return X, c0


GENERATORS = {
    "lattice_d4_k300": lambda o: _lattice(o, 4, 300),
    "lattice_d8_k100": lambda o: _lattice(o, 8, 100),
    "lattice_d4_k64": lambda o: _lattice(o, 4, 64, N=1000, seed=3),
    "dup_rows_d8_k400": lambda o: _dup_rows(o, 8, 400),
    "dup_rows_d4_k200": lambda o: _dup_rows(o, 4, 200),
    "offset_dim0_d8_k300": lambda o: _offset(o, 8, 300, False),
    "offset_all_d4_k256": lambda o: _offset(o, 4, 256, True),
    "scales_d8_k300": lambda o: _scales(o, 8, 300),
    "scales_d4_k120": lambda o: _scales(o, 4, 120),
    "runs_n_k1_d8_k300": lambda o: _runs(o, 8, 300, 301),
    "runs_n_k1_d4_k40": lambda o: _runs(o, 4, 40, 41),
    "runs_n20_d8_k12": lambda o: _runs(o, 8, 12, 20),
    "nan_scattered_d8_k300": lambda o: _nan_rows(o, 8, 300, "scattered"),
    "nan_cell_d8_k512": lambda o: _nan_rows(o, 8, 512, "cell"),
    "nan_cell_d4_k200": lambda o: _nan_rows(o, 4, 200, "cell"),
    "nan_one_finite_d4_k300": lambda o: _nan_rows(o, 4, 300, "one_finite"),
    "nan_one_finite_d8_k64": lambda o: _nan_rows(o, 8, 64, "one_finite"),
    "nan_all_d8_k300": lambda o: _nan_rows(o, 8, 300, "all"),
    "nan_all_d4_k100": lambda o: _nan_rows(o, 4, 100, "all"),
}
GEN = sorted(GENERATORS)
PASSES = 5


@pytest.fixture(scope="module")
def adversarial(oracle):
    """every generator's (X, c0) with the oracle's references, computed in parallel"""
    def one(name):
        X, c0 = GENERATORS[name](oracle)
        X, c0 = np.ascontiguousarray(X, np.float32), np.ascontiguousarray(c0, np.float32)
        assert np.nanmax(np.abs(X)) <= 2.0 ** 20 and (np.isnan(c0).all() or np.nanmax(np.abs(c0)) <= 2.0 ** 20)
        return dict(X=X, c0=c0, scan=oracle.knn_scan_reduce(X, c0, 3, PASSES),
                    kdt=oracle.knn_scan_reduce_kdtree(X, c0, 3, PASSES), assign=oracle.assign(X, c0),
                    lloyd=oracle.lloyd(X, c0, 3), yakmo=oracle.yakmo(X, c0.shape[0]))
    with ThreadPoolExecutor(THREADS) as ex:
        return dict(zip(GEN, ex.map(one, GEN)))


def _same_scan(got, ref, what):
    assert got[2] == ref[2] and _same_err(got[3], ref[3]), (what, got[2:], ref[2:])
    assert np.array_equal(got[1], ref[1]), (what, int(np.argmax(got[1] != ref[1])))
    assert _same_f32(got[0], ref[0]), what


# ---- CPU: the restatement against the oracle ----------------------------------------------------------------------
SMALL = ["lattice_d4_k64", "lattice_d8_k100", "dup_rows_d4_k200", "runs_n_k1_d4_k40", "runs_n20_d8_k12", "nan_all_d4_k100",
         "nan_one_finite_d8_k64", "audio_d8_k128"]


def _small_case(oracle, name):
    if name == "audio_d8_k128":
        X = _features(oracle, 0.2, 8, seed=21)[:2500]
        return X, oracle.yakmo(X, 128)[0]
    X, c0 = GENERATORS[name](oracle)
    return np.ascontiguousarray(X[:3000], np.float32), np.ascontiguousarray(c0, np.float32)


@pytest.mark.parametrize("name", SMALL)
def test_numpy_restatement_equals_oracle(oracle, name):
    """The oracle and the kernels share an author; this restatement shares no code with either."""
    X, c0 = _small_case(oracle, name)
    lab, dist = oracle.assign(X, c0)
    for i in range(0, len(X), 7):
        j, d = np_nearest(X[i], c0)
        assert j == lab[i] and _same_f32(d, dist[i]), i
    ref = oracle.knn_scan_reduce(X, c0, 3, 3)
    mine = np_knn_scan_reduce(X, c0, 3, 3)
    _same_scan(mine, ref, name)


def test_numpy_lloyd_exact_sums_equal_oracle_on_lattice(oracle):
    X, c0 = _lattice(oracle, 4, 64, N=1000, seed=3)
    c_ref, l_ref = oracle.lloyd(X, c0, 3)
    c_np, l_np = np_lloyd_exact(X, c0, 3)
    assert _same_f32(c_np, c_ref) and np.array_equal(l_np, l_ref)


def test_all_nan_codebook_contract(oracle):
    """Every row NaN: centroid 0 at distance +inf (what the kernels report), so the error of a pass is +inf, not NaN."""
    X, c0 = _nan_rows(oracle, 8, 300, "all")
    lab, dist = oracle.assign(X[:50], c0)
    assert (lab == 0).all() and np.isposinf(dist).all()
    _, lab, it, err = oracle.knn_scan_reduce(X[:200], c0, 3, 3)
    assert (lab == 0).all() and it == 3 and np.isposinf(err)


# ---- CPU: every dispatched instantiation of the searched kernels has an exact test --------------------------------
# instantiation in libgsc_cuda.so -> the tests that run it and compare it bit for bit
COVERAGE = {
    "k_online<4,4,64>": "test_online_small_dictionary_both_kernels",     # D = 4, K <= 256, GSC_DBG_ONLINE_BATCHED
    "k_online<4,4,128>": "test_online_kmeans_bit_exact",
    "k_online<4,8,128>": "test_online_kmeans_bit_exact",
    "k_online<4,8,256>": "test_online_kmeans_bit_exact",
    "k_online<4,16,256>": "test_online_kmeans_bit_exact",
    "k_online<8,4,64>": "test_online_small_dictionary_both_kernels",
    "k_online<8,4,128>": "test_online_kmeans_bit_exact",
    "k_online<8,8,128>": "test_online_kmeans_bit_exact",
    "k_online<8,8,256>": "test_online_kmeans_bit_exact",
    "k_online<8,16,256>": "test_online_kmeans_bit_exact",
    "k_online_warp<4,1>": "test_online_small_dictionary_both_kernels",
    "k_online_warp<4,2>": "test_online_small_dictionary_both_kernels",
    "k_online_warp<8,1>": "test_online_small_dictionary_both_kernels",
    "k_online_warp<8,2>": "test_online_small_dictionary_both_kernels",
    **{f"k_assign<{d},{p}>": "test_assign_every_instantiation" for d in (4, 8, 16) for p in (2, 4, 8)},
    **{f"k_seed2<{d},{s}>": "test_yakmo_seeding_every_instantiation" for d in (4, 8, 16)
       for s in ("256,2", "256,3", "128,4", "128,6")},
    "k_knnfit_win<2>": "test_knnfit_adversarial_dictionary",
    "k_knnfit_win<4>": "test_knnfit_adversarial_dictionary",
    "k_knnfit_win<8>": "test_knnfit_adversarial_dictionary",
}
GUARDED = ("k_online", "k_online_warp", "k_assign", "k_seed2", "k_knnfit_win")


def kernel_instantiations(so):
    """demangled names of the guarded kernels in a built libgsc_cuda.so, as 'k_assign<4,8>'"""
    from soundchunks_b200 import build
    bindir = os.path.dirname(build.nvcc_path())
    dump = subprocess.run([os.path.join(bindir, "cuobjdump"), "-res-usage", so], capture_output=True, text=True, check=True)
    mangled = [ln.split("Function ", 1)[1].split(":")[0].strip() for ln in dump.stdout.splitlines() if "Function " in ln]
    filt = shutil.which("cu++filt") or os.path.join(bindir, "cu++filt")
    names = subprocess.run([filt], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout.split("\n")
    out = set()
    for n in names:
        n = n.strip().removeprefix("void ")
        head = n.split("<", 1)[0]
        if head in GUARDED and "<" in n:
            out.add(head + "<" + n.split("<", 1)[1].split(">", 1)[0].replace("(int)", "").replace(" ", "") + ">")
    return out


def test_every_search_kernel_instantiation_has_a_test(lib_built):
    """A new template instantiation of a pruned search kernel must come with an exact test (an entry above)."""
    found = kernel_instantiations(lib_built)
    assert {n.split("<")[0] for n in found} == set(GUARDED), found
    missing = sorted(found - set(COVERAGE))
    assert not missing, f"instantiations without an exact test: {missing}"
    sources = "".join(open(os.path.join(ROOT, "tests", f)).read() for f in os.listdir(os.path.join(ROOT, "tests")) if f.endswith(".py"))
    for inst, test in COVERAGE.items():
        assert f"def {test}(" in sources, (inst, test)


# ---- GPU: every instantiation -------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("P", [2, 4, 8])
@pytest.mark.parametrize("D", [4, 8, 16])
def test_assign_every_instantiation(ctx, oracle, D, P, monkeypatch):
    """k_assign<D, P>: codebook tiles of 512 (256 for D = 16) -> K at and either side of the tile edge; N is not a
    multiple of the 128 * P points of a CTA."""
    X = _features(oracle, 0.5 if D == 4 else 1.0, D, seed=30 + D, ch=2)[:5037]
    assert len(X) == 5037
    monkeypatch.setenv("GSC_ASSIGN_PTS", str(P))
    for K in (1, 255, 256, 257, 511, 512, 513, 4096):
        c0 = oracle.yakmo(X, K)[0] if K > 1 else X[17:18].copy()
        l_ref, d_ref = oracle.assign(X, c0)
        l_gpu, d_gpu = ctx.assign(X, c0)
        assert np.array_equal(l_gpu, l_ref), (K, int(np.argmax(l_gpu != l_ref)))
        assert _same_f32(d_gpu, d_ref), K


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["256x2", "256x3", "128x4", "128x6"])
@pytest.mark.parametrize("D", [4, 16])
def test_yakmo_seeding_every_instantiation(ctx, oracle, D, shape, monkeypatch):
    """k_seed2<D, threads, CTAs per SM> for D = 4 (-cs 2) and 16 (-cs 8): seeds, means and labels == the oracle and
    == the one-warp serial chain (GSC_DBG_SEED_SERIAL)."""
    X = _features(oracle, 0.4, D, seed=50 + D)
    K = 700
    c_ref, l_ref, s_ref = oracle.yakmo(X, K)
    monkeypatch.setenv("GSC_SEED_SHAPE", shape)
    c_gpu, l_gpu, s_gpu = ctx.yakmo(X, K)
    assert np.array_equal(s_gpu, s_ref), f"first divergence at seed {int(np.argmax(s_gpu != s_ref))}"
    assert _same_f32(c_gpu, c_ref) and np.array_equal(l_gpu, l_ref)
    if shape == "256x2":
        c2, l2, s2 = _debug(ctx, ctx.DBG_SEED_SERIAL, ctx.yakmo, X, K)
        assert np.array_equal(s2, s_ref) and _same_f32(c2, c_ref) and np.array_equal(l2, l_ref)


@pytest.mark.gpu
@pytest.mark.parametrize("D", [4, 8])
def test_online_pass_slices_and_precisions(ctx, oracle, D):
    """k_online runs in launches of 8 passes: max_passes either side of a slice edge; and every precision."""
    X = _features(oracle, 0.3, D, seed=70)
    K = 1025
    c0 = oracle.yakmo(X, K)[0]
    cases = [(3, p) for p in (1, 7, 8, 9, 16, 17)] + [(p, 100) for p in (1, 2, 4, 6)]
    with ThreadPoolExecutor(THREADS) as ex:
        refs = list(ex.map(lambda a: oracle.knn_scan_reduce(X, c0, *a), cases))
    for (prec, mp), ref in zip(cases, refs):
        _same_scan(ctx.knn_scan_reduce(X, c0, prec, mp), ref, (prec, mp))


# ---- GPU: the adversarial inputs through every search -------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", GEN)
def test_adversarial_online_kmeans(ctx, adversarial, name, monkeypatch):
    """knn_scan_reduce: one- and two-warp k_online_warp (K <= 256), the CTA-per-frame kernel with its filter and
    scoring every centroid exactly (GSC_DBG_ONLINE_EXACT)."""
    a = adversarial[name]
    X, c0 = a["X"], a["c0"]
    runs = [(0, "1"), (ctx.DBG_ONLINE_EXACT, "1")]
    if c0.shape[0] <= 256:
        runs += [(0, "2"), (ctx.DBG_ONLINE_BATCHED, "1"), (ctx.DBG_ONLINE_BATCHED | ctx.DBG_ONLINE_EXACT, "1")]
    for flag, warps in runs:
        monkeypatch.setenv("GSC_OW_WARPS", warps)
        _same_scan(_debug(ctx, flag, ctx.knn_scan_reduce, X, c0, 3, PASSES), a["scan"], (name, flag, warps))


@pytest.mark.gpu
@pytest.mark.parametrize("name", GEN)
def test_adversarial_kdtree(ctx, adversarial, name):
    a = adversarial[name]
    for flag in (0, ctx.DBG_KDTREE_SERIAL):
        _same_scan(_debug(ctx, flag, ctx.knn_scan_reduce_kdtree, a["X"], a["c0"], 3, PASSES), a["kdt"], (name, flag))


@pytest.mark.gpu
@pytest.mark.parametrize("name", GEN)
def test_adversarial_assign(ctx, adversarial, name, monkeypatch):
    a = adversarial[name]
    l_ref, d_ref = a["assign"]
    for P in ("2", "4", "8"):
        monkeypatch.setenv("GSC_ASSIGN_PTS", P)
        l_gpu, d_gpu = ctx.assign(a["X"], a["c0"])
        assert np.array_equal(l_gpu, l_ref) and _same_f32(d_gpu, d_ref), (name, P)


@pytest.mark.gpu
@pytest.mark.parametrize("name", GEN)
def test_adversarial_yakmo(ctx, adversarial, name):
    a = adversarial[name]
    c_ref, l_ref, s_ref = a["yakmo"]
    K = a["c0"].shape[0]
    for flag in (0, ctx.DBG_SEED_SERIAL):
        c, l, s = _debug(ctx, flag, ctx.yakmo, a["X"], K)
        assert np.array_equal(s, s_ref), (name, flag, int(np.argmax(s != s_ref)))
        assert _same_f32(c, c_ref) and np.array_equal(l, l_ref), (name, flag)


@pytest.mark.gpu
@pytest.mark.parametrize("name", GEN)
def test_adversarial_lloyd_owner(ctx, adversarial, name):
    """GSC_DBG_LLOYD_OWNER sums every cluster's rows in ascending point order in Double, the oracle's order: the
    result is oracle.lloyd bit for bit, labels included, NaN start rows included."""
    a = adversarial[name]
    c, l = _debug(ctx, ctx.DBG_LLOYD_OWNER, ctx.lloyd, a["X"], a["c0"], 3)
    assert _same_f32(c, a["lloyd"][0]) and np.array_equal(l, a["lloyd"][1]), name


@pytest.mark.gpu
@pytest.mark.parametrize("name", SMALL)
def test_numpy_restatement_equals_gpu(ctx, oracle, name):
    X, c0 = _small_case(oracle, name)
    lab, dist = ctx.assign(X, c0)
    for i in range(0, len(X), 7):
        j, d = np_nearest(X[i], c0)
        assert j == lab[i] and _same_f32(d, dist[i]), i
    _same_scan(ctx.knn_scan_reduce(X, c0, 3, 3), np_knn_scan_reduce(X, c0, 3, 3), name)


# ---- GPU: Lloyd -------------------------------------------------------------------------------------------------
def _ulps(a, b):
    a = np.asarray(a, np.float32).view(np.int32).astype(np.int64)
    b = np.asarray(b, np.float32).view(np.int32).astype(np.int64)
    return np.abs(a - b)


@pytest.mark.gpu
def test_lloyd_exact_sums_on_lattice(ctx, oracle):
    """Lattice points: every sum is exact, so the mean has one rounding whatever the order.  The default scatter
    path, the owner path, the oracle and the fsum restatement agree bit for bit."""
    X, c0 = _lattice(oracle, 8, 300, N=4000, seed=8)
    want = np_lloyd_exact(X, c0, 2)
    assert _same_f32(oracle.lloyd(X, c0, 2)[0], want[0])
    for flag in (0, ctx.DBG_LLOYD_OWNER):
        c, l = _debug(ctx, flag, ctx.lloyd, X, c0, 2)
        assert _same_f32(c, want[0]) and np.array_equal(l, want[1]), flag


@pytest.mark.gpu
def test_lloyd_audio_with_nan_start_rows(ctx, oracle):
    """A real mode-1 start (yakmo means, NaN for empty seed cells, not nan_to_num'ed): the owner path is the oracle
    bit for bit; the scatter path (atomic Double adds, any order) is within 1 ulp in a handful of coordinates."""
    from tests.golden_util import load_full
    pcm, sr, bits, K, *_ = load_full(os.path.join(ROOT, "tests", "golden", "full_60_f0_k4096_12.npz"))
    X = oracle.make_chunks(pcm, 4, bits, oracle.find_attenuation_divider(pcm, 4, bits))[3]
    c0 = oracle.yakmo(X, K)[0]
    assert np.isnan(c0).any()
    c_ref, l_ref = oracle.lloyd(X, c0, 1)
    c, l = _debug(ctx, ctx.DBG_LLOYD_OWNER, ctx.lloyd, X, c0, 1)
    assert _same_f32(c, c_ref) and np.array_equal(l, l_ref)
    c, l = ctx.lloyd(X, c0, 1)
    assert np.array_equal(np.isnan(c), np.isnan(c_ref))
    u = _ulps(np.nan_to_num(c), np.nan_to_num(c_ref))
    assert u.max() <= 1 and np.count_nonzero(u) <= 16, (u.max(), np.count_nonzero(u))


# ---- GPU: the caller-driven split API (gsc_split_begin / step / update / end) -------------------------------------
def _split_run(ctxs, parts, c0, iters):
    import torch
    K, D = c0.shape
    accs = [torch.zeros(K * (D + 1), dtype=torch.float64, device="cuda") for _ in ctxs]
    for c, X in zip(ctxs, parts):
        c.split_begin(X, c0)
    for _ in range(iters):
        for c, a in zip(ctxs, accs):
            c.split_step(a.data_ptr())
        total = accs[0] if len(accs) == 1 else accs[0] + accs[1]
        torch.cuda.synchronize()                     # the library's streams read the sum next
        for c in ctxs:
            c.split_update(total.data_ptr())
    outs = [c.split_end() for c in ctxs]
    return outs[0][0], np.concatenate([o[1] for o in outs])


@pytest.mark.gpu
@pytest.mark.parametrize("data", ["lattice", "audio"])
def test_split_api_one_and_two_contexts(ctx, oracle, data):
    import soundchunks_b200 as sc
    if data == "lattice":
        X, c0 = _lattice(oracle, 8, 256, N=6000, seed=12)
    else:
        X = _features(oracle, 0.5, 8, seed=14, ch=2)
        c0 = np.nan_to_num(oracle.yakmo(X, 512)[0], nan=0.0)
    iters = 3
    want = ctx.lloyd(X, c0, iters)
    one = _split_run([ctx], [X], c0, iters)
    assert _same_f32(one[0], want[0]) and np.array_equal(one[1], want[1])
    h = len(X) // 2 + 5
    with sc.Context(0) as a, sc.Context(0) as b:
        two = _split_run([a, b], [X[:h], X[h:]], c0, iters)
    if data == "lattice":
        assert _same_f32(two[0], want[0]) and np.array_equal(two[1], want[1])
    else:
        rel = np.max(np.abs(two[0] - want[0]) / np.maximum(np.abs(want[0]), 1e-6))
        assert rel <= 1e-4 and np.mean(two[1] != want[1]) < 1e-3


# ---- GPU: KNNFit on adversarial dictionaries ----------------------------------------------------------------------
def _clipped_pcm(seconds, sr, ch, seed):
    """audio with a clipped stretch, a square wave at full scale, a constant -32768 and a repeating 4-sample pattern"""
    a = _audio(seconds, sr, ch, seed).astype(np.int64)
    n = a.shape[1]
    a[:, : n // 5] = np.clip(a[:, : n // 5] * 16, -32768, 32767)
    sq = np.where((np.arange(n // 5) // 37) % 2 == 0, 32767, -32768)
    a[:, n // 5: 2 * n // 5] = sq
    a[:, 2 * n // 5: 3 * n // 5] = -32768
    a[:, 3 * n // 5: 4 * n // 5] = np.resize(np.array([32767, -32768, 1200, -5]), n // 5)
    return np.ascontiguousarray(a.astype(np.int16))


def _adversarial_dictionary(oracle, pcm, cs, bits, div, R):
    raw, attr, atten, feat, dst = oracle.make_chunks(pcm, cs, bits, div)
    labels = np.random.default_rng(cs).integers(0, R, len(feat)).astype(np.int32)
    d = oracle.build_dictionary(labels, raw, attr, R, bits, div)
    dic, datten = d["dict"].copy(), d["datten"].copy()
    pal = np.concatenate([np.arange(1, cs // 2 + 1), np.arange(cs // 2, 0, -1)]) * 301
    dic[[3, 40, R - 1]] = dic[17]; datten[[3, 40, R - 1]] = datten[17]       # duplicates, later and earlier
    dic[[5, 6, R // 2]] = 0                                                   # zero chunks
    dic[[7, R // 3]] = pal                                                    # palindromes: reversed == itself
    dic[8] = 32767; dic[9] = -32768; dic[10, ::2] = -32768; dic[10, 1::2] = 32767   # full scale, -32768 included
    datten[[8, 9, 10]] = 0
    return raw, dic, datten


@pytest.mark.gpu
@pytest.mark.parametrize("cs", [2, 4, 8])
def test_knnfit_adversarial_dictionary(ctx, oracle, cs):
    """k_knnfit_win<cs> (norm window + bisected band threshold) and the dense scan == oracle.knnfit's untruncated
    rule (best_all, band); the kd-tree path == oracle.knnfit_kdtree."""
    bits, R = 12, 512
    pcm = _clipped_pcm(0.4, 44100, 2, 80 + cs)
    div = oracle.find_attenuation_divider(pcm, cs, bits)
    raw, dic, datten = _adversarial_dictionary(oracle, pcm, cs, bits, div, R)
    ref = oracle.knnfit(dic, datten, raw, bits, div)
    for flag in (0, ctx.DBG_KNNFIT_DENSE):
        got = _debug(ctx, flag, ctx.knnfit, dic, datten, pcm, cs, bits, div)
        assert np.array_equal(got["band"], ref["band"]), (flag, int(np.argmax(got["band"] != ref["band"])))
        assert np.array_equal(got["best"], ref["best_all"]), flag
        assert np.array_equal(got["use"], np.bincount(ref["best_all"] >> 2, minlength=R)), flag
    kref = oracle.knnfit_kdtree(dic, datten, raw, bits, div)
    kgot = ctx.knnfit_kdtree(dic, datten, pcm, cs, bits, div)
    assert np.array_equal(kgot["best"], kref["best"]) and np.array_equal(kgot["use"], kref["use"])


# ---- GPU: chunk size 8 stage by stage, and whole frames of clipped / DC / square-wave PCM --------------------------
@pytest.mark.gpu
def test_chunk_size_8_stage_by_stage(ctx, oracle):
    """-cs 8 (Lloyd mode only): make_chunks, build_dictionary from the oracle's labels, knnfit and finalize bit for
    bit; then a whole mode-1 frame with the owner-ordered Lloyd sums, .gsc bytes included."""
    from soundchunks_b200 import host
    cs, bits, K = 8, 12, 256
    pcm = _quiet(_audio(0.3, 44100, 2, 90))
    div = oracle.find_attenuation_divider(pcm, cs, bits)
    assert ctx.find_attenuation_divider(pcm, cs, bits) == div
    raw, attr, atten, feat, dst = oracle.make_chunks(pcm, cs, bits, div)
    g_attr, g_atten, g_feat, g_dst = ctx.make_chunks(pcm, cs, bits, div)
    assert np.array_equal(g_attr, attr) and np.array_equal(g_atten, atten) and np.array_equal(g_dst, dst)
    assert _same_f32(g_feat, feat)
    c0 = oracle.yakmo(feat, K)[0]
    _, labels = oracle.lloyd(feat, c0, 3)
    ref = oracle.build_dictionary(labels, raw, attr, K, bits, div)
    gpu = ctx.build_dictionary(labels, pcm, attr, K, cs, bits, div)
    for k in ("counts", "order", "entry", "dict", "datten", "dattr"):
        assert np.array_equal(gpu[k], ref[k]), k
    assert _same_f32(gpu["means"], ref["means"])
    kf = oracle.knnfit(ref["dict"], ref["datten"], raw, bits, div)
    gk = ctx.knnfit(ref["dict"], ref["datten"], pcm, cs, bits, div)
    assert np.array_equal(gk["band"], kf["band"]) and np.array_equal(gk["best"], kf["best_all"])
    n_ref, remap_ref, order_ref = oracle.finalize_dictionary(gk["use"])
    n_gpu, remap_gpu, order_gpu = ctx.finalize_dictionary(gk["use"])
    assert n_gpu == n_ref and np.array_equal(remap_gpu, remap_ref) and np.array_equal(order_gpu, order_ref)
    kw = dict(chunk_size=cs, chunk_bit_depth=bits, chunks_per_frame=K, kmeans_mode=1, lloyd_iters=3)
    ctx.set_debug(ctx.DBG_LLOYD_OWNER)
    try:
        r = ctx.encode_frames([pcm], **kw)[0]
        blob, _ = ctx.fetch_stream(1, 44100)
    finally:
        ctx.set_debug(0)
    fr = oracle.encode_frame(pcm, band_all=1, **kw)
    assert (r.N, r.R, r.divider, r.overfull) == (fr.N, fr.R, fr.divider, fr.overfull)
    assert np.array_equal(r.dict, fr.dict) and np.array_equal(r.datten, fr.datten)
    assert np.array_equal(r.index, fr.index) and np.array_equal(r.attr, fr.attr)
    assert bytes(blob) == oracle.write_frame(fr, 2, cs, bits, 44100) == host.write_frame(r, 2, cs, bits, 44100)


def _full_scale_frame(kind, seconds=0.4, sr=44100):
    n = int(seconds * sr) // 8 * 8
    t = np.arange(n)
    if kind == "clipped":
        a = np.clip(_audio(seconds, sr, 2, 33)[:, :n].astype(np.int64) * 24, -32768, 32767)
    elif kind == "square":
        a = np.stack([np.where((t // 50) % 2 == 0, 32767, -32768), np.where((t // 7) % 2 == 0, -32768, 32767)])
    elif kind == "dc":
        a = np.stack([np.full(n, -32768), np.full(n, -32768)])
        a[1, n // 2:] = 32767
    else:   # a repeating 4-sample pattern on one channel, audio on the other
        a = np.stack([np.resize(np.array([32767, -32768, 0, -32768]), n), _audio(seconds, sr, 1, 34)[0, :n].astype(np.int64)])
    return np.ascontiguousarray(a.astype(np.int16))


FRAME_CASES = [(kind, mode, K) for kind in ("clipped", "square", "dc", "pattern4") for mode in (0, 3) for K in (256, 4096)]


@pytest.fixture(scope="module")
def full_scale_refs(oracle):
    def one(case):
        kind, mode, K = case
        kw = dict(band_all=1) if mode == 0 else {}
        return oracle.encode_frame(_full_scale_frame(kind), chunk_bit_depth=12, chunks_per_frame=K, kmeans_mode=mode, **kw)
    with ThreadPoolExecutor(THREADS) as ex:
        return dict(zip(FRAME_CASES, ex.map(one, FRAME_CASES)))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,mode,K", FRAME_CASES)
def test_full_scale_frames(ctx, oracle, full_scale_refs, kind, mode, K):
    """Whole frames through gsc_encode_frames (the seed cells give the k-means its first guesses) against
    oracle.encode_frame (mode 0 with the band over all rows, mode 3 through the kd-tree), .gsc bytes included."""
    pcm = _full_scale_frame(kind)
    ref = full_scale_refs[(kind, mode, K)]
    r = ctx.encode_frames([pcm], chunk_bit_depth=12, chunks_per_frame=K, kmeans_mode=mode)[0]
    assert (r.N, r.R, r.divider, r.passes, r.overfull) == (ref.N, ref.R, ref.divider, ref.passes, ref.overfull)
    assert _same_err(r.err, ref.err)
    assert np.array_equal(r.dict, ref.dict) and np.array_equal(r.datten, ref.datten)
    assert np.array_equal(r.index, ref.index) and np.array_equal(r.attr, ref.attr)
    blob, _ = ctx.fetch_stream(1, 44100)
    assert bytes(blob) == oracle.write_frame(ref, 2, 4, 12, 44100)


# ---- GPU: the packed stream follows the sample rate ---------------------------------------------------------------
@pytest.mark.gpu
def test_fetch_stream_repacks_for_another_sample_rate(ctx):
    """Every frame header carries the sample rate: fetching the same batch at 44100 and then at 48000 (and back)
    gives each rate's own bytes, for a one-lane and a two-lane batch."""
    from soundchunks_b200 import host
    for n in (2, 17):
        frames = [_quiet(_audio(0.05 + 0.01 * (i % 3), 44100, 2, 600 + i)) for i in range(n)]
        res = ctx.encode_frames(frames, chunk_bit_depth=12, chunks_per_frame=256)
        for sr in (44100, 48000, 44100):
            blob, sizes = ctx.fetch_stream(n, sr)
            want = [host.write_frame(r, 2, 4, 12, sr) for r in res]
            assert sizes.tolist() == [len(w) for w in want]
            assert bytes(blob) == b"".join(want), (n, sr)
