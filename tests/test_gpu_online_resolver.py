"""The resolver of the CTA-per-frame online k-means (k_online, phase 2 in gsc_online.cuh) on inputs made to drive each
of its paths, for every dispatched (D, K) shape, bit for bit against the CPU oracle.

Each case also asserts through the kernel's counters (ctx.online_counters) that the path it aims at ran:
  runs       runs of nearly identical points: most points of a batch want the same centroid, so rounds conflict and
             commit anywhere from one lane to a whole batch, and a centroid moves in two rounds of one batch
  crowded    48 near-copies of a few codebook rows next to the points: more than L = 32 candidates per point (full
             lists), which the resolver settles by re-filtering the point against the whole codebook
"""
import numpy as np
import pytest

PASSES = 4
# (D, K) of every k_online instantiation gsc_api.cu dispatches; K <= 256 runs it only under GSC_DBG_ONLINE_BATCHED
SHAPES = [(D, K) for D in (4, 8) for K in (200, 400, 1000, 2000, 4000)]


def _runs(D, K, seed):
    rng = np.random.default_rng(seed)
    N = K + 1200
    centers = rng.normal(0.0, 1.0, (N // 24 + 1, D)).astype(np.float32)
    lens = rng.integers(1, 48, len(centers))                    # runs of 1 .. 47 points
    X = np.repeat(centers, lens, axis=0)[:N]
    X = X + rng.normal(0.0, 1e-4, X.shape).astype(np.float32)   # nearly identical within a run
    if len(X) < N:
        X = np.concatenate([X, rng.normal(0.0, 1.0, (N - len(X), D)).astype(np.float32)])
    c0 = X[np.sort(rng.choice(N, K, replace=False))].copy()
    return X.astype(np.float32), c0


def _crowded(D, K, seed):
    rng = np.random.default_rng(seed)
    N = max(3000, K + 500)
    X = rng.normal(0.0, 1.0, (N, D)).astype(np.float32)
    c0 = X[np.sort(rng.choice(N, K, replace=False))].copy()
    hubs = rng.choice(N, 4, replace=False)
    slots = rng.choice(K, 4 * 48, replace=False).reshape(4, 48)
    for h, s in zip(hubs, slots):
        c0[s] = X[h] + rng.normal(0.0, 1e-5, (48, D)).astype(np.float32)
        X[h: h + 40] = X[h] + rng.normal(0.0, 1e-3, (min(40, N - h), D)).astype(np.float32)
    return X, c0


CASES = {"runs": _runs, "crowded": _crowded}


def _same_f32(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(a.view(np.uint32)[~na], b.view(np.uint32)[~nb])


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("D,K", SHAPES)
def test_resolver_paths_match_oracle(ctx, oracle, case, D, K):
    X, c0 = CASES[case](D, K, seed=1000 * D + K)
    X, c0 = np.ascontiguousarray(X, np.float32), np.ascontiguousarray(c0, np.float32)
    ref = oracle.knn_scan_reduce(X, c0, 3, PASSES)
    ctx.set_debug(ctx.DBG_ONLINE_BATCHED if K <= 256 else 0)
    try:
        got = ctx.knn_scan_reduce(X, c0, 3, PASSES)
        cn = ctx.online_counters(1)[0].astype(np.int64)
    finally:
        ctx.set_debug(0)
    assert got[2] == ref[2] and got[3] == ref[3], (got[2:], ref[2:])
    assert np.array_equal(got[1], ref[1]), int(np.argmax(got[1] != ref[1]))
    assert _same_f32(got[0], ref[0])
    batches, points, exhaustive, rounds, full, cands, again = (int(v) for v in cn[:7])
    assert points == len(X) * got[2] and batches > 0 and cands > 0, cn[:7]
    if case == "runs":
        assert rounds > batches, cn[:7]            # conflicting rounds
        assert again > 0, cn[:7]                   # a centroid committed in two rounds of one batch
    else:
        assert full > 0, cn[:7]                    # candidate lists overflowed
        assert exhaustive > 0, cn[:7]              # ... and their points were re-filtered
