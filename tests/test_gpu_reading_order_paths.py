"""Both reading-order kernels on the paths of the page routine they share: every case runs once in a default context
(pages of up to 4096 boxes and 28 672 intersecting pairs take the shared-memory kernel) and once in a context created
with MS_B200_RO_FORCE_LARGE=1 (every page takes the global-memory kernel).  Pages go through the device entry point
ms_reading_order, must come back unflagged, and must give the order of host_word_order, the host restatement pinned to
the reference goldens."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", params=["shared", "global"])
def ctx(request):
    import manuscript_b200 as mb

    os.environ.pop("MS_B200_RO_FORCE_LARGE", None)
    if request.param == "global":
        os.environ["MS_B200_RO_FORCE_LARGE"] = "1"
    try:
        c = mb._cabi.Context(0)
    finally:
        os.environ.pop("MS_B200_RO_FORCE_LARGE", None)
    yield c
    c.close()


def _polys(boxes):
    b = np.asarray(boxes, np.float32).reshape(-1, 4)
    x0, y0, x1, y1 = b[:, 0], b[:, 1], b[:, 2], b[:, 3]
    return np.stack([x0, y0, x1, y0, x1, y1, x0, y1], axis=1)


def _random_boxes(rng, n, side, w=(1, 90), h=(1, 40)):
    x0, y0 = rng.integers(0, side, n), rng.integers(0, side, n)
    return np.stack([x0, y0, x0 + rng.integers(*w, n), y0 + rng.integers(*h, n)], axis=1).reshape(n, 4)


def _staircase(n):
    """Box k meets boxes k - 1 and k + 1 only: the pairs form one chain of n - 1 dependency levels.  The staircase climbs
    to the right, so the lines, and with them the order, depend on the heights the sweeps leave."""
    k = np.arange(n)
    y = 3 * (n - 1 - k)
    return np.stack([10 * k, y, 10 * k + 15, y + 20], axis=1)


def _n_pairs(bx):
    b = np.asarray(bx, np.int64)
    inter = ~((b[:, None, 2] <= b[None, :, 0]) | (b[None, :, 2] <= b[:, None, 0]) |
              (b[:, None, 3] <= b[None, :, 1]) | (b[None, :, 3] <= b[:, None, 1]))
    return (int(inter.sum()) - len(b)) // 2


def _check_pages(ctx, pages):
    """All pages in one ms_reading_order call; order and reordered rows of every page against the host restatement."""
    import torch

    import manuscript_b200 as mb
    from manuscript_b200.reading_order import host_word_order

    P, cap = len(pages), max(1, max(len(b) for b in pages))
    rows = np.zeros((P, cap, 9), np.float32)
    cnts = np.array([len(b) for b in pages], np.int32)
    for pg, bx in enumerate(pages):
        if len(bx):
            rows[pg, : len(bx), :8] = _polys(bx)
            rows[pg, : len(bx), 8] = np.arange(len(bx))
    d_rows, d_cnt = torch.from_numpy(rows).cuda(), torch.from_numpy(cnts).cuda()
    d_ord = torch.full((P, cap), -1, dtype=torch.int32, device="cuda")
    d_out = torch.zeros_like(d_rows)
    d_flags = torch.zeros((P,), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    mb._cabi.check(ctx.lib.ms_reading_order(ctx.handle, d_rows.data_ptr(), d_cnt.data_ptr(), P, cap, d_ord.data_ptr(),
                                            d_out.data_ptr(), d_flags.data_ptr(), C.c_void_p(0)))
    torch.cuda.synchronize()
    assert d_flags.cpu().tolist() == [0] * P
    ords, outs = d_ord.cpu().numpy(), d_out.cpu().numpy()
    for pg, bx in enumerate(pages):
        n = len(bx)
        want = host_word_order(rows[pg, :n, :8]) if n else np.zeros(0, np.int32)
        assert ords[pg, :n].tolist() == want.tolist(), f"page {pg} ({n} boxes)"
        np.testing.assert_array_equal(outs[pg, :n], rows[pg, want], err_msg=f"page {pg}")


def _with_duplicates(bx):
    d, m = bx.copy(), len(bx) // 7
    d[m:2 * m] = d[3 * m:4 * m]                                       # exact duplicates
    d[4 * m:4 * m + m // 2, 2:] = d[5 * m:5 * m + m // 2, 2:]          # boxes that share a corner with another one
    d[:, 2] = np.maximum(d[:, 2], d[:, 0] + 1)  # the integer boxes are min / max hulls: x0 < x1, y0 < y1
    d[:, 3] = np.maximum(d[:, 3], d[:, 1] + 1)
    return d


def test_duplicates_and_shared_corners(ctx):
    """The dict (last box of equal compressed coordinates) and first-match quirks, on the grid and all-pairs paths."""
    rng = np.random.default_rng(21)
    _check_pages(ctx, [_with_duplicates(_random_boxes(rng, 700, 900)), _with_duplicates(_random_boxes(rng, 140, 300))])


def test_zero_height_boxes(ctx):
    """avg_h == 0: the horizontal condition is never true and every box is its own line."""
    rng = np.random.default_rng(22)
    pages = []
    for n, side in ((700, 900), (90, 200)):
        bx = _random_boxes(rng, n, side)
        bx[:, 3] = bx[:, 1]
        pages.append(bx)
    _check_pages(ctx, pages)


def test_page_wide_box(ctx):
    """One box over more than 64 grid cells: the pair search tests all pairs instead of the grid."""
    bx = _random_boxes(np.random.default_rng(23), 700, 900)
    bx[5] = (0, 0, 900, 900)
    _check_pages(ctx, [bx])


def test_fewer_than_256_boxes(ctx):
    """Below 256 boxes the shared-memory kernel tests all pairs without a grid."""
    rng = np.random.default_rng(24)
    _check_pages(ctx, [_random_boxes(rng, n, side) for n, side in ((1, 50), (2, 30), (3, 40), (100, 300), (255, 500))])


def test_staircase_of_300_boxes(ctx):
    """A chain of 299 levels: more than the shared-memory kernel's 255 (one-thread sweeps), fewer than the global-memory
    kernel's 4095 (parallel sweeps over level buckets)."""
    bx = _staircase(300)
    assert _n_pairs(bx) == 299
    _check_pages(ctx, [bx])


def test_staircase_of_5000_boxes(ctx):
    """A chain of 4999 levels: more than the global-memory kernel's 4095 (one-thread sweeps)."""
    _check_pages(ctx, [_staircase(5000)])


def test_batch_mixing_both_kernels(ctx):
    """One call over small and empty pages, pages of more than 4096 boxes and a page of fewer boxes but more than 28 672
    intersecting pairs: both kernels in a default context, more pages than the global-memory kernel has scratch slots
    when every page goes there."""
    rng = np.random.default_rng(25)
    dense = _random_boxes(rng, 3000, 800, w=(20, 80), h=(10, 40))
    assert _n_pairs(dense) > 28672
    pages = [_random_boxes(rng, 150, 400), _with_duplicates(_random_boxes(rng, 700, 900)), np.zeros((0, 4), np.int64),
             _random_boxes(rng, 5000, 3000), _staircase(300), dense, _random_boxes(rng, 2500, 1500)]
    pages += [_random_boxes(rng, int(n), 1500) for n in rng.integers(4097, 4600, 2)]
    pages += [_random_boxes(rng, int(n), 1000) for n in rng.integers(0, 2000, 3)]
    _check_pages(ctx, pages)
