"""The front stages on ragged page batches, every page against the oracle at the boundaries that keep pages apart.

Pages lie back to back in the packed candidate space (csrc/lanms.cu lanms_offsets_kernel), so a page boundary can fall
anywhere inside a warp, a 2048-key sort tile (csrc/sort.cu) or a CTA.  The batches here put pages of named, seeded
shapes next to each other -- sizes one off a power of two, exactly 4096 / 4097 kept boxes (the bitonic / radix switch
of lanms_sort_emit_kernel), runs of hot positions across a 2048-position round of lanms_accept_kernel, 1024 / 1025
accepted runs (lanms_build_clusters_kernel's shared-memory table), tied and signed-zero keys, a cluster cut by the page
end -- and compare every page of ms_lanms with oracle.cpu.locality_aware_nms of that page alone, bit for bit.

  * test_batch_pages_hit_their_boundaries (CPU): the oracle alone shows that each page is what its name claims.
  * Batch A: 27 pages at cap 20 483 (no multiple of 32, 128 or 2048) at thr 0, 0.2 and 0.5; the irregular page
    and its neighbours again at thr -1.
  * Batch B: 160 pages at cap 20 480 (10 sort tiles a page): fewer sort CTAs than tiles per page, so a CTA strides.
  * Both: a page alone gives the rows it gives in the batch, a permuted batch the permuted rows, a second call the
    same bits; an edge-buffer overflow is flagged on its own page only.
  * ms_east_boxes on a ragged batch (each page its own original size) against cpu.east_postprocess.
  * ms_test_np_sum_host: the pairwise sums of the area-anomaly filter against np.add.reduce, bit for bit.
"""
import concurrent.futures as cf
import ctypes as C
import multiprocessing
import os

import numpy as np
import pytest

import synthdata
from oracle import cpu

RECT = np.array([[0, 0], [1, 0], [1, 1], [0, 1]], float)
CAP_A = 20483
CAP_B = 20480
SORT_TILE = 2048        # csrc/sort.cu kTile
ACCEPT_ROUND = 2048     # csrc/lanms.cu kAcceptBatch
BUILD_RUNS = 1024       # csrc/lanms.cu kBuildRuns
SORT_MAX = 4096         # csrc/lanms.cu kSortMax
THRS_A = (0.0, 0.2, 0.5)
MS_FLAG_EDGE_OVERFLOW = 4


# ---- page generators: (rng) -> (n, 9) float32 candidate rows ---------------------------------------------------------
def _rows(quads, scores):
    q = np.asarray(quads, np.float64).reshape(-1, 8)
    return np.concatenate([q, np.asarray(scores, np.float64).reshape(-1, 1)], axis=1).astype(np.float32)


def _words(rng, n, x0=0.0, per_word=(1, 40)):
    """n candidates of words in one text line, words 90 px apart in x: the candidates of a word are its quad plus
    decode noise, so each word is contiguous in x0 order"""
    out, k = [], 0
    while sum(len(o) for o in out) < n:
        m = min(int(rng.integers(per_word[0], per_word[1] + 1)), n - sum(len(o) for o in out))
        w, h = rng.uniform(40, 70), rng.uniform(12, 24)
        base = RECT * [w, h] + [x0 + 90.0 * k, rng.uniform(0, 8)]
        q = base[None] + rng.normal(0, 0.4, (m, 4, 2))
        out.append(_rows(q, rng.uniform(0.6, 1.0, m)))
        k += 1
    return np.concatenate(out) if out else np.zeros((0, 9), np.float32)


def _clusters(rng, sizes, x0=0.0):
    """cluster c: sizes[c] near-identical quads (IoU ~0.95 with each other and with their running merge), clusters
    100 px apart in x (IoU 0 between clusters): cluster c holds sizes[c] - 1 hot positions and, if sizes[c] > 1, one
    accepted merge run -- at every threshold below ~0.9"""
    out = []
    for c, m in enumerate(sizes):
        base = RECT * [60, 20] + [x0 + 100.0 * c, 10.0]
        q = base[None] + rng.normal(0, 0.3, (m, 4, 2))
        out.append(_rows(q, rng.uniform(0.5, 1.0, m)))
    return np.concatenate(out)


def _grid(rng, k, scores):
    """k disjoint 30 x 12 boxes on a 64-column grid (10 / 8 px gaps): k clusters, all kept at every threshold"""
    i = np.arange(k)
    org = np.stack([(i % 64) * 40.0, (i // 64) * 20.0], -1)
    return _rows(RECT[None] * [30, 12] + org[:, None, :], scores)


def _tie_scores(rng, k):
    """equal scores and signed zeros: the kept order is the cluster index order within each tie"""
    return rng.choice(np.array([0.5, 0.25, 0.0, -0.0], np.float32), k)


def _banded(rng, x0s, n_bands=8):
    """one quad per x0, in random text bands 40 px apart, equal scores: consecutive quads of one band (IoU >= ~0.5)
    merge, others do not -- which quads are consecutive, and so the clusters and the order of the kept rows, is
    decided by the x0 order alone (ties: the original index)"""
    x0s = np.asarray(x0s, np.float32)
    n = len(x0s)
    band = rng.integers(0, n_bands, n)
    w = rng.uniform(40, 80, n)
    y = band * 40.0 + rng.normal(0, 0.3, n)
    q = np.zeros((n, 4, 2))
    q[:, :, 0] = np.abs(x0s.astype(np.float64))[:, None] + RECT[None, :, 0] * w[:, None]
    q[:, :, 1] = y[:, None] + RECT[None, :, 1] * 20.0
    rows = _rows(q, np.full(n, 0.7))
    rows[:, 0] = x0s  # x0 bit for bit (a signed zero stays signed)
    rows[:, 6] = x0s
    return rows


def gen_x0_all_equal(rng):
    return _banded(rng, np.full(5000, 100.0))  # 3 sort tiles of one key


def gen_x0_signed_zero(rng):
    z = np.where(rng.random(2500) < 0.5, np.float32(-0.0), np.float32(0.0))
    neg = _banded(rng, -rng.uniform(100, 500, 300).astype(np.float32))
    neg[:, 1::2] += 400  # other bands: the negative quads stay clear of the zero ones
    big = _banded(rng, rng.uniform(1e6, 1e6 + 2000, 300).astype(np.float32))
    rows = np.concatenate([_banded(rng, z), neg, big])
    return rows[rng.permutation(len(rows))]


def gen_dense(rng):
    """test_gpu_parity.test_lanms_dense_candidates: far more than 32 overlapping neighbours per cluster"""
    n = 3000
    c = rng.uniform(0, 260, (n, 1, 2))
    return _rows(c + RECT * rng.uniform(15, 45, (n, 1, 2)), rng.uniform(0.3, 1, n))


def gen_irregular(rng):
    """test_gpu_parity.test_lanms_hard_cases (c): clockwise, self-intersecting and degenerate quads among regular ones"""
    m = 600
    c = rng.uniform(0, 200, (m, 1, 2))
    quads = c + rng.uniform(-15, 15, (m, 4, 2))
    quads[:300] = c[:300] + RECT * rng.uniform(5, 30, (300, 1, 2))
    quads[300:330] = quads[300:330, ::-1]
    quads[330:340] = quads[330:340, :1]
    return _rows(quads, rng.uniform(0.3, 1, m))


def gen_nonfinite(rng):
    rows = _words(rng, 400)
    at = rng.choice(len(rows), 8, replace=False)
    rows[at[:4], 0] = np.nan        # NaN x0: sorted last, as numpy sorts
    rows[at[4], 0] = np.inf
    rows[at[5], 3] = np.nan
    rows[at[6], 5] = -np.inf
    rows[at[7], [0, 2]] = np.nan
    return rows


BAIT_QUAD = RECT * [60, 20] + [40000.0, 10.0]


def gen_bait_end(rng):
    """words, then a 300-candidate cluster of BAIT_QUAD at the largest x0: the page's last position lies inside it"""
    tail = _rows(BAIT_QUAD[None] + rng.normal(0, 0.3, (300, 4, 2)), rng.uniform(0.5, 1.0, 300))
    return np.concatenate([_words(rng, 700), tail])


def gen_bait_start(rng):
    """BAIT_QUAD (moved 1.5 px right, past the noise of gen_bait_end's copies) at the smallest x0, words to its right:
    it would merge with the previous page's last row if the pages were one list"""
    first = _rows(BAIT_QUAD[None] + [[1.5, 0.0]], [0.9])
    return np.concatenate([_words(rng, 500, x0=40100.0), first])


# name -> (generator, claims).  Claims hold at every threshold of THRS_A:
# n candidates, kept rows, hot positions (IoU with the x0 predecessor > thr), accepted runs (clusters of more than
# one candidate), "crossing": a run whose hot positions straddle a 2048-position round of the accept pass.
PAGES_A = {
    "empty": (lambda rng: np.zeros((0, 9), np.float32), dict(n=0, kept=0)),
    "one": (lambda rng: _words(rng, 1), dict(n=1, kept=1)),
    "two_same": (lambda rng: np.repeat(_words(rng, 1), 2, axis=0), dict(n=2, kept=1, hot=1, runs=1)),
    "n2047": (lambda rng: _words(rng, 2047), dict(n=2047)),
    "bait_end": (gen_bait_end, dict(n=1000, bait="end")),
    "bait_start": (gen_bait_start, dict(n=501, bait="start")),
    "n2048": (lambda rng: _words(rng, 2048), dict(n=2048)),
    "n2049": (lambda rng: _words(rng, 2049), dict(n=2049)),
    "x0_all_equal": (gen_x0_all_equal, dict(n=5000)),
    "kept1024": (lambda rng: _grid(rng, 1024, rng.uniform(0.1, 1, 1024)), dict(n=1024, kept=1024, hot=0)),
    "empty2": (lambda rng: np.zeros((0, 9), np.float32), dict(n=0, kept=0)),
    "kept1025_ties": (lambda rng: _grid(rng, 1025, _tie_scores(rng, 1025)), dict(n=1025, kept=1025, hot=0)),
    "n6149": (lambda rng: _words(rng, 3 * 2048 + 5), dict(n=3 * 2048 + 5)),
    "kept4096": (lambda rng: _grid(rng, 4096, rng.uniform(0.1, 1, 4096)), dict(n=4096, kept=4096, hot=0)),
    "kept4097_ties": (lambda rng: _grid(rng, 4097, _tie_scores(rng, 4097)), dict(n=4097, kept=4097, hot=0)),
    "x0_signed_zero": (gen_x0_signed_zero, dict(n=3100)),
    "hot2047": (lambda rng: _clusters(rng, [90] * 23), dict(n=2070, kept=23, hot=2047, runs=23)),
    "hot2048": (lambda rng: _clusters(rng, [65] * 32), dict(n=2080, kept=32, hot=2048, runs=32)),
    "hot2049": (lambda rng: _clusters(rng, [65] * 32 + [2]), dict(n=2082, kept=33, hot=2049, runs=33)),
    "hot4097": (lambda rng: _clusters(rng, [65] * 64 + [2]), dict(n=4162, kept=65, hot=4097, runs=65)),
    "run_across_round": (lambda rng: _clusters(rng, [101] * 20 + [150] + [11] * 5),
                         dict(n=2020 + 150 + 55, kept=26, hot=2199, runs=26, crossing=True)),
    "runs1024": (lambda rng: _clusters(rng, [2] * 1024), dict(n=2048, kept=1024, hot=1024, runs=1024)),
    "runs1025": (lambda rng: _clusters(rng, [2] * 1025), dict(n=2050, kept=1025, hot=1025, runs=1025)),
    "dense_redo": (gen_dense, dict(n=3000)),
    "irregular": (gen_irregular, dict(n=600)),
    "nonfinite": (gen_nonfinite, dict(n=400)),
    "n_cap": (lambda rng: _words(rng, CAP_A), dict(n=CAP_A)),
}
NAMES_A = list(PAGES_A)


def batch_a():
    return [PAGES_A[name][0](np.random.default_rng(1000 + i)) for i, name in enumerate(NAMES_A)]


DENSE_B = {7: (101, 1408, 800), 33: (102, 1344, 700), 64: (103, 1408, 900), 65: (104, 1472, 800),
           101: (105, 1344, 800), 150: (106, 1440, 700)}  # page -> synthdata (seed, page size, words)
N_PAGES_B = 160


def batch_b():
    rng = np.random.default_rng(2024)
    pages = []
    for p in range(N_PAGES_B):
        if p in DENSE_B:
            seed, size, words = DENSE_B[p]
            score, geo, _ = synthdata.make_maps(seed, size, words)
            pages.append(cpu.decode_quads_from_maps(score, geo, 0.6, 4.0, 1)[:CAP_B])
        else:
            n = 0 if p % 17 == 3 else int(rng.integers(1, 301))
            pages.append(_words(rng, n, x0=float(rng.uniform(0, 300)))[rng.permutation(n)])
    return pages


# ---- oracle --------------------------------------------------------------------------------------------------------
def _workers():
    return max(1, min(len(os.sched_getaffinity(0)), 32))


def oracle_lanms(jobs):
    """[(rows, thr)] -> [cpu.locality_aware_nms(rows, thr)], fanned out over host processes (largest first)"""
    order = sorted(range(len(jobs)), key=lambda j: -len(jobs[j][0]))
    out = [None] * len(jobs)
    with cf.ProcessPoolExecutor(_workers(), mp_context=multiprocessing.get_context("spawn")) as ex:
        futs = {ex.submit(cpu.locality_aware_nms, jobs[j][0], jobs[j][1]): j for j in order}
        for f in cf.as_completed(futs):
            out[futs[f]] = f.result()
    return out


def x0_order(rows):
    return np.argsort(rows[:, 0], kind="stable")  # NaN last


def hot_positions(rows, thr):
    """positions s (in stable x0 order) with polygon_iou(box_s, box_{s-1}) > thr -- lanms.py:180 for a fresh cluster"""
    s = rows[x0_order(rows)]
    if len(s) < 2:
        return np.zeros(0, np.int64)
    iou = cpu.polygon_iou_batch(s[1:, :8].reshape(-1, 4, 2), s[:-1, :8].reshape(-1, 4, 2))
    return np.nonzero(iou > thr)[0] + 1


def merge_scan(rows, thr):
    """lanms.py:166-192 restated on the oracle's primitives: (start position, size) of every cluster in x0 order"""
    s = rows[x0_order(rows)].astype(np.float64)
    clusters, last, wsum, start = [], None, 0.0, 0
    for i, r in enumerate(s):
        poly = r[:8].reshape(4, 2)
        if last is not None and cpu.should_merge(poly, last, thr):
            al = cpu.normalize_polygon(last, poly)
            tw = wsum + r[8]
            last = (last * wsum + al * r[8]) / tw
            wsum = tw
            continue
        if last is not None:
            clusters.append((start, i - start))
        last, wsum, start = poly.copy(), r[8], i
    if last is not None:
        clusters.append((start, len(s) - start))
    return clusters


# ---- 2. CPU: the pages are what their names claim ------------------------------------------------------------------------
def test_batch_pages_hit_their_boundaries():
    pages = batch_a()
    thrs = (0.0, 0.2, 0.5)
    want_kept = {name: c["kept"] for name, (_, c) in PAGES_A.items() if "kept" in c}
    kept_jobs = [(pages[NAMES_A.index(name)], thr) for name in want_kept for thr in thrs]
    kept = oracle_lanms(kept_jobs)
    for (name, thr), out in zip([(nm, t) for nm in want_kept for t in thrs], kept):
        assert len(out) == want_kept[name], (name, thr, len(out))
    for name, rows in zip(NAMES_A, pages):
        claims = PAGES_A[name][1]
        assert rows.shape == (claims["n"], 9) and rows.dtype == np.float32, (name, rows.shape)
        for thr in thrs:
            if "hot" in claims:
                assert len(hot_positions(rows, thr)) == claims["hot"], (name, thr)
            if "runs" in claims or claims.get("crossing"):
                cl = merge_scan(rows, thr)
                _, dbg = cpu.locality_aware_nms(rows, thr, debug=True)
                assert len(cl) == len(dbg["cluster_polys"]), (name, thr)  # the restated scan is the oracle's
                runs = [(a, m) for a, m in cl if m > 1]
                assert len(runs) == claims["runs"], (name, thr, len(runs))
                if claims.get("crossing"):
                    hot = hot_positions(rows, thr)
                    rank = {int(h): j for j, h in enumerate(hot)}
                    cross = [(a, m) for a, m in runs if rank[a + 1] < ACCEPT_ROUND <= rank[a + m - 1]]
                    assert len(cross) == 1, (name, thr)
    # the shapes of the switches: sizes one off the powers of two, tied and signed-zero keys across tiles
    n = {name: len(rows) for name, rows in zip(NAMES_A, pages)}
    assert {n["n2047"], n["n2048"], n["n2049"]} == {SORT_TILE - 1, SORT_TILE, SORT_TILE + 1}
    assert n["n_cap"] == CAP_A and CAP_A % 32 and CAP_A % 128 and CAP_A % SORT_TILE
    eq = pages[NAMES_A.index("x0_all_equal")]
    assert len(eq) > 2 * SORT_TILE and np.all(eq[:, 0] == eq[0, 0])
    sz = pages[NAMES_A.index("x0_signed_zero")][:, 0]
    zero = sz == 0
    assert np.signbit(sz[zero]).sum() > 500 and (~np.signbit(sz[zero])).sum() > 500
    assert (sz < 0).sum() > 100 and (sz >= 1e6).sum() > 100 and zero.sum() > SORT_TILE
    for name in ("kept1025_ties", "kept4097_ties"):
        sc = pages[NAMES_A.index(name)][:, 8]
        assert np.signbit(sc[sc == 0]).sum() > 100 and (~np.signbit(sc[sc == 0])).sum() > 100
    assert {want_kept["kept4096"], want_kept["kept4097_ties"]} == {SORT_MAX, SORT_MAX + 1}
    assert {PAGES_A["runs1024"][1]["runs"], PAGES_A["runs1025"][1]["runs"]} == {BUILD_RUNS, BUILD_RUNS + 1}
    nf = pages[NAMES_A.index("nonfinite")]
    assert np.isnan(nf[:, 0]).sum() >= 4 and not np.isfinite(nf[:, :8]).all(axis=1).all()
    # boundary bait: the last row (x0 order) of bait_end lies in a cluster of more than one candidate, and the first
    # row of bait_start would merge with it if the two pages were one list
    end, start = pages[NAMES_A.index("bait_end")], pages[NAMES_A.index("bait_start")]
    assert NAMES_A.index("bait_start") == NAMES_A.index("bait_end") + 1
    last, first = end[x0_order(end)[-1]], start[x0_order(start)[0]]
    assert first[0] >= last[0]  # adjacent in the x0 order of the two pages as one list
    for thr in thrs:
        a, m = merge_scan(end, thr)[-1]
        assert m > 100 and a + m == len(end)
        assert cpu.should_merge(first[:8].reshape(4, 2), last[:8].reshape(4, 2), thr)
    # Batch B: ten sort tiles a page; the dense pages hold more than eight tiles, so a CTA that strides over its
    # page's tiles (8 per page on a 148-SM B200) meets real keys on its second tile
    pb = batch_b()
    nb = [len(p) for p in pb]
    assert len(pb) == N_PAGES_B and -(-CAP_B // SORT_TILE) == 10
    assert all(15000 <= nb[p] <= CAP_B for p in DENSE_B)
    assert sum(nb[p] > 8 * SORT_TILE for p in DENSE_B) >= 3
    assert all(nb[p] <= 300 for p in range(N_PAGES_B) if p not in DENSE_B) and nb.count(0) >= 5


# ---- the device side -----------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch():
    import torch as t

    return t


@pytest.fixture(scope="module")
def ctx():
    import manuscript_b200 as mb

    return mb.Context(0)


def run_lanms(ctx, torch, pages, cap, thr, grow=True):
    """ms_lanms on device buffers as bench.py calls it: page-strided input, quads_out filled with NaN first.  With
    grow, an MS_FLAG_EDGE_OVERFLOW page makes the call run again with a larger edge factor (the header's policy).
    Returns (per-page rows, flags)."""
    from manuscript_b200._cabi import check

    P = len(pages)
    host = np.zeros((P, cap, 9), np.float32)
    for p, rows in enumerate(pages):
        host[p, :len(rows)] = rows
    q = torch.from_numpy(host).cuda()
    counts = torch.tensor([len(r) for r in pages], dtype=torch.int32, device="cuda")
    out = torch.empty((P, cap, 9), dtype=torch.float32, device="cuda")
    cnt = torch.empty(P, dtype=torch.int32, device="cuda")
    flags = torch.empty(P, dtype=torch.int32, device="cuda")
    while True:
        out.fill_(float("nan"))
        cnt.fill_(-1)
        flags.zero_()
        check(ctx.lib.ms_lanms(ctx.handle, q.data_ptr(), counts.data_ptr(), P, cap, float(thr), out.data_ptr(),
                               cnt.data_ptr(), flags.data_ptr(), None))
        torch.cuda.synchronize()
        f = flags.cpu().numpy()
        if not grow or not (f & MS_FLAG_EDGE_OVERFLOW).any() or not ctx.grow_edge_factor():
            break
    c = cnt.cpu().numpy()
    o = out.cpu().numpy()
    assert np.all(c >= 0) and np.all(c <= np.array([len(r) for r in pages]))
    return [o[p, :c[p]].copy() for p in range(P)], f


def assert_rows(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    np.testing.assert_array_equal(got, want, err_msg=str(what))
    fin = ~np.isnan(want)
    np.testing.assert_array_equal(np.signbit(got[fin]), np.signbit(want[fin]), err_msg=f"{what}: signed zeros")


def assert_same_bits(a, b, what):
    assert len(a) == len(b)
    for p, (x, y) in enumerate(zip(a, b)):
        assert x.shape == y.shape and x.tobytes() == y.tobytes(), (what, p)


@pytest.fixture(scope="module")
def pages_a():
    return batch_a()


@pytest.fixture(scope="module")
def want_a(pages_a):
    jobs = [(rows, thr) for thr in THRS_A for rows in pages_a]
    res = oracle_lanms(jobs)
    return {thr: res[i * len(pages_a):(i + 1) * len(pages_a)] for i, thr in enumerate(THRS_A)}


@pytest.mark.gpu
@pytest.mark.parametrize("thr", THRS_A)
def test_batch_a_every_page_matches_the_oracle(ctx, torch, pages_a, want_a, thr):
    got, flags = run_lanms(ctx, torch, pages_a, CAP_A, thr)
    assert not flags.any(), dict(zip(NAMES_A, flags))
    for name, g, w in zip(NAMES_A, got, want_a[thr]):
        assert_rows(g, w, (name, thr))


@pytest.mark.gpu
def test_irregular_page_at_negative_threshold(ctx, torch, pages_a):
    """thr < 0: IoU == 0 pairs merge too, and the NMS pairs every box with every other of its page (no prefilter)"""
    names = ["two_same", "irregular", "nonfinite", "empty", "n2047"]
    pages = [pages_a[NAMES_A.index(n)] for n in names]
    got, flags = run_lanms(ctx, torch, pages, CAP_A, -1.0)
    assert not flags.any()
    for n, g, w in zip(names, got, oracle_lanms([(rows, -1.0) for rows in pages])):
        assert_rows(g, w, n)


@pytest.mark.gpu
def test_batch_a_pages_alone_permuted_and_repeated(ctx, torch, pages_a, want_a):
    thr = 0.2
    got, _ = run_lanms(ctx, torch, pages_a, CAP_A, thr)
    again, _ = run_lanms(ctx, torch, pages_a, CAP_A, thr)
    assert_same_bits(got, again, "second call")
    for p, rows in enumerate(pages_a):
        alone, _ = run_lanms(ctx, torch, [rows], CAP_A, thr)
        assert alone[0].tobytes() == got[p].tobytes(), NAMES_A[p]
    perm = np.random.default_rng(5).permutation(len(pages_a))
    pg, _ = run_lanms(ctx, torch, [pages_a[i] for i in perm], CAP_A, thr)
    assert_same_bits(pg, [got[i] for i in perm], "permuted batch")
    for name, g, w in zip(NAMES_A, got, want_a[thr]):
        assert_rows(g, w, name)


@pytest.fixture(scope="module")
def pages_b():
    return batch_b()


SMALL_B = 6000  # thr 0.0 and 0.5 are compared on the pages below this many candidates (oracle time)


@pytest.fixture(scope="module")
def want_b(pages_b):
    jobs = [(rows, 0.2) for rows in pages_b] + [(rows, thr) for thr in (0.0, 0.5) for rows in pages_b
                                               if len(rows) < SMALL_B]
    res = iter(oracle_lanms(jobs))
    want = {0.2: [next(res) for _ in pages_b]}
    for thr in (0.0, 0.5):
        want[thr] = [next(res) if len(rows) < SMALL_B else None for rows in pages_b]
    return want


@pytest.mark.gpu
@pytest.mark.parametrize("thr", [0.2, 0.0, 0.5])
def test_batch_b_every_page_matches_the_oracle(ctx, torch, pages_b, want_b, thr):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    tiles = -(-CAP_B // SORT_TILE)
    gx = min(tiles, -(-8 * sms // N_PAGES_B))  # csrc/sort.cu msk_sort_pages (and lanms_build_clusters: 80 -> gx)
    assert gx < tiles, (sms, gx)  # a CTA of seg_hist / seg_scatter sorts more than one tile of a dense page
    got, flags = run_lanms(ctx, torch, pages_b, CAP_B, thr)
    assert not flags.any()
    compared = 0
    for p, (g, w) in enumerate(zip(got, want_b[thr])):
        if w is not None:
            assert_rows(g, w, (p, len(pages_b[p]), thr))
            compared += 1
    assert compared >= N_PAGES_B - len(DENSE_B)


@pytest.mark.gpu
def test_batch_b_pages_alone_permuted_and_repeated(ctx, torch, pages_b, want_b):
    thr = 0.2
    got, _ = run_lanms(ctx, torch, pages_b, CAP_B, thr)
    again, _ = run_lanms(ctx, torch, pages_b, CAP_B, thr)
    assert_same_bits(got, again, "second call")
    for p, rows in enumerate(pages_b):
        alone, _ = run_lanms(ctx, torch, [rows], CAP_B, thr)
        assert alone[0].tobytes() == got[p].tobytes(), p
    perm = np.random.default_rng(6).permutation(N_PAGES_B)
    pg, _ = run_lanms(ctx, torch, [pages_b[i] for i in perm], CAP_B, thr)
    assert_same_bits(pg, [got[i] for i in perm], "permuted batch")


@pytest.mark.gpu
def test_edge_overflow_stays_on_its_page(torch, pages_a, want_a):
    """edge factor 1: the dense page overflows its neighbour-pair buffer and is the only page flagged; every other page
    is still the oracle's; after the edge factor is raised (x4, as the header asks) the dense page is too"""
    import manuscript_b200 as mb

    c = mb.Context(0)
    try:
        names = ["n2047", "kept1024", "hot2048", "dense_redo", "runs1024", "n6149", "one"]
        pages = [pages_a[NAMES_A.index(n)] for n in names]
        want = [want_a[0.2][NAMES_A.index(n)] for n in names]
        c.edge_factor = 1
        got, flags = run_lanms(c, torch, pages, CAP_A, 0.2, grow=False)
        d = names.index("dense_redo")
        assert flags[d] & MS_FLAG_EDGE_OVERFLOW and not np.delete(flags, d).any(), dict(zip(names, flags))
        for i, (g, w) in enumerate(zip(got, want)):
            if i != d:
                assert_rows(g, w, names[i])
        while flags[d] & MS_FLAG_EDGE_OVERFLOW:
            assert c.grow_edge_factor()
            got, flags = run_lanms(c, torch, pages, CAP_A, 0.2, grow=False)
        assert not flags.any() and c.edge_factor > 1
        for n, g, w in zip(names, got, want):
            assert_rows(g, w, n)
    finally:
        c.close()


# ---- 3. ms_east_boxes on a ragged batch -----------------------------------------------------------------------------------
CAP_E = 5003
TARGET = 1280


def _disjoint(rng, k, size=(14, 40)):
    """k disjoint boxes inside the target square (LANMS keeps all of them), varied sizes and scores"""
    cols = max(1, int(np.ceil(np.sqrt(k * 3))))
    pitch = TARGET / cols
    i = np.arange(k)
    org = np.stack([(i % cols) * pitch, (i // cols) * pitch / 3], -1) + 1.0
    wh = np.stack([rng.uniform(0.3, 0.9, k) * pitch, rng.uniform(0.2, 0.3, k) * pitch], -1)
    return _rows(org[:, None, :] + RECT[None] * wh[:, None, :], rng.uniform(0.6, 1, k))


def _nested(rng):
    """boxes with boxes inside them (IoU <= 0.1: LANMS keeps both) and a few area outliers"""
    outer = _disjoint(rng, 200)
    q = outer[:80, :8].reshape(80, 4, 2).astype(np.float64)
    ctr = q.mean(1, keepdims=True)
    inner = _rows(ctr + (q - ctr) * 0.3, rng.uniform(0.6, 1, 80))
    big = _rows(RECT[None] * [400, 300] + rng.uniform(0, 800, (3, 1, 2)), [0.99, 0.98, 0.97])
    return np.concatenate([outer, inner, big])


def _same_min_corner(rng):
    """12 boxes sharing their min corner (pairwise IoU <= 1/6: none merges): one grid cell holds the whole page"""
    wh = np.array([(w, h) for w in (10, 60, 360, 2160) for h in (5, 30, 180)], float) * 0.5
    return _rows(np.array([100.0, 100.0]) + RECT[None] * wh[:, None, :], rng.uniform(0.6, 1, len(wh)))


def _nonfinite_boxes(rng):
    rows = _disjoint(rng, 60)
    rows[7, 2] = np.nan
    rows[30, 1] = np.inf
    return rows


EAST_PAGES = [(f"k{k}", (lambda k: lambda rng: _disjoint(rng, k))(k), k)
              for k in (0, 1, 7, 8, 9, 127, 128, 129)]
EAST_PAGES += [("nonfinite", _nonfinite_boxes, None), ("k136", lambda rng: _disjoint(rng, 136), 136),
               ("k137", lambda rng: _disjoint(rng, 137), 137), ("nested", _nested, None),
               ("k1024", lambda rng: _disjoint(rng, 1024), 1024), ("same_min_corner", _same_min_corner, 12),
               ("k1025", lambda rng: _disjoint(rng, 1025), 1025), ("k5000", lambda rng: _disjoint(rng, 5000), 5000)]
ORIG_HW = [(900, 700), (1600, 1100), (640, 2000), (1280, 960), (3000, 1500), (500, 480), (720, 1280), (2048, 1536),
           (1100, 1700), (333, 777), (1400, 600), (2500, 3100), (801, 1279), (1281, 1900), (960, 540), (4000, 3000)]


@pytest.fixture(scope="module")
def east_inputs():
    """the oracle's LANMS output of every page (thr 0.2), as the EAST path hands it to the box filters"""
    pages = [gen(np.random.default_rng(3000 + i)) for i, (_, gen, _) in enumerate(EAST_PAGES)]
    return oracle_lanms([(rows, 0.2) for rows in pages])


def test_east_pages_hit_their_sizes(east_inputs):
    """(CPU) the LANMS outputs have the box counts the pairwise-sum leaf rule and its 8-accumulator loop turn on"""
    for (name, _, k), rows in zip(EAST_PAGES, east_inputs):
        if k is not None:
            assert len(rows) == k, (name, len(rows))
    assert len(east_inputs[-1]) > 4096 and len(EAST_PAGES) == len(ORIG_HW)
    assert not np.isfinite(east_inputs[[n for n, _, _ in EAST_PAGES].index("nonfinite")]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("expand", [0.9, 0.0])
@pytest.mark.parametrize("axis_aligned", [True, False])
def test_east_boxes_ragged_batch(ctx, torch, east_inputs, axis_aligned, expand):
    import manuscript_b200 as mb
    from manuscript_b200._cabi import check

    P = len(east_inputs)
    host = np.zeros((P, CAP_E, 9), np.float32)
    for p, rows in enumerate(east_inputs):
        host[p, :len(rows)] = rows
    q = torch.from_numpy(host).cuda()
    counts = torch.tensor([len(r) for r in east_inputs], dtype=torch.int32, device="cuda")
    hw = torch.tensor(ORIG_HW, dtype=torch.int32, device="cuda")
    out = torch.full((P, CAP_E, 9), float("nan"), dtype=torch.float32, device="cuda")
    cnt = torch.full((P,), -1, dtype=torch.int32, device="cuda")
    params = mb.EastParams.default(target_size=TARGET, axis_aligned_output=int(axis_aligned),
                                   expand_ratio_w=expand, expand_ratio_h=expand)
    check(ctx.lib.ms_east_boxes(ctx.handle, q.data_ptr(), counts.data_ptr(), P, CAP_E, C.byref(params), hw.data_ptr(),
                                out.data_ptr(), cnt.data_ptr(), None))
    torch.cuda.synchronize()
    o, c = out.cpu().numpy(), cnt.cpu().numpy()
    removed = 0
    for p, ((name, _, _), rows) in enumerate(zip(EAST_PAGES, east_inputs)):
        want = cpu.east_postprocess(rows, ORIG_HW[p], target_size=TARGET, expand_w=expand, expand_h=expand,
                                    axis_aligned=axis_aligned)
        assert_rows(o[p, :c[p]], want, (name, ORIG_HW[p]))
        removed += len(rows) - len(want)
    assert removed > 50  # contained-box removal and the anomaly filter both took rows out


# ---- 4. the pairwise sums of the area-anomaly filter -------------------------------------------------------------------
def _sum_vectors(rng, lengths):
    """order-sensitive float32 values: mixed signs, magnitudes 1e-3 .. 1e6, runs of equal values"""
    out = []
    for n in lengths:
        mag = 10.0 ** rng.uniform(-3, 6, n)
        v = mag * rng.choice([-1.0, 1.0], n)
        if n > 16:
            for _ in range(3):
                a = int(rng.integers(0, n))
                v[a:a + int(rng.integers(2, 40))] = v[a]
        out.append(v.astype(np.float32))
    return out


def np_sum_device(ctx, vectors):
    from manuscript_b200._cabi import check

    lengths = np.array([len(v) for v in vectors], np.int32)
    offsets = np.concatenate([[0], np.cumsum(lengths[:-1], dtype=np.int64)]).astype(np.int64)
    values = np.ascontiguousarray(np.concatenate(vectors), np.float32)
    serial = np.empty(len(vectors), np.float32)
    cta = np.empty(len(vectors), np.float32)
    check(ctx.lib.ms_test_np_sum_host(ctx.handle, values.ctypes.data, offsets.ctypes.data, lengths.ctypes.data,
                                      len(vectors), serial.ctypes.data, cta.ctypes.data))
    return serial, cta


def _split_lengths():
    ls = set(range(1, 4097))
    for k in (513, 1000, 1025, 2048, 4096, 8191):
        ls.update({8 * k - 1, 8 * k + 1})
    for k in range(12):
        ls.update({128 * 2 ** k - 8, 128 * 2 ** k + 8})
    ls.update({131072 + 1, 140000, 200003, 262144 - 1, 299993, 300000})  # more than 1024 leaves: one thread
    return sorted(v for v in ls if v > 0)


@pytest.mark.gpu
def test_np_pairwise_sums_on_the_device(ctx):
    rng = np.random.default_rng(71)
    lengths = _split_lengths()
    vectors = _sum_vectors(rng, lengths)
    serial, cta = np_sum_device(ctx, vectors)
    want = np.array([np.add.reduce(v) for v in vectors], np.float32)
    lib = cpu.lib()
    model = np.array([lib.orc_np_sum_f32(v, len(v)) for v in vectors], np.float32)
    np.testing.assert_array_equal(model.view(np.uint32), want.view(np.uint32))  # the oracle's model is numpy's
    for name, got in (("serial", serial), ("cta", cta)):
        bad = np.nonzero(got.view(np.uint32) != want.view(np.uint32))[0]
        assert len(bad) == 0, (name, [(lengths[i], got[i], want[i]) for i in bad[:5]])
    assert max(lengths) > 1024 * 256  # the one-thread fallback of np_pairwise_f32_cta ran


@pytest.mark.gpu
def test_anomaly_mean_and_std_on_the_device(ctx):
    """infer.py:222-224 mean / std of float32 areas (as east_finish_kernel and oracle.c compute them) == np.mean /
    np.std, with the device sums"""
    rng = np.random.default_rng(72)
    ks = [31, 127, 128, 129, 1000, 1025, 4097, 20000, 150000]
    areas = []
    for k in ks:
        a = rng.uniform(50, 5000, k) * rng.choice([1.0, 1.0, 1.0, 30.0], k)
        areas.append(a.astype(np.float32))
    sums, sums_cta = np_sum_device(ctx, areas)
    np.testing.assert_array_equal(sums.view(np.uint32), sums_cta.view(np.uint32))
    mean = np.array([s / np.float32(k) for s, k in zip(sums, ks)], np.float32)
    devs = [np.square(a - m) for a, m in zip(areas, mean)]
    dsum, dsum_cta = np_sum_device(ctx, devs)
    np.testing.assert_array_equal(dsum.view(np.uint32), dsum_cta.view(np.uint32))
    std = np.array([np.sqrt(d / np.float32(k)) for d, k in zip(dsum, ks)], np.float32)
    lib = cpu.lib()
    for i, a in enumerate(areas):
        assert mean[i].tobytes() == np.float32(np.mean(a)).tobytes(), ks[i]
        assert std[i].tobytes() == np.float32(np.std(a)).tobytes(), ks[i]
        assert sums[i] == lib.orc_np_sum_f32(a, len(a)) and dsum[i] == lib.orc_np_sum_f32(devs[i], len(devs[i]))
