"""The host-buffer entry points' capacity retry and the CUDA-graph key of the device page batch.

Retry: with the NMS neighbour-pair capacity set to 1 pair per candidate, ms_page_batch_host (several upload chunks),
ms_page_batch_ragged_host and ms_standard_nms_host overflow it, grow it and run again inside the call; what they return
must be bit for bit what a fresh context at the default capacity returns.

Graph key: two calls on the same buffers that differ in one argument are two graphs; alternating them past the capture
must give what direct launches (MS_B200_NO_GRAPHS=1) give."""
import numpy as np
import pytest

import synthdata
from oracle import cpu

pytestmark = pytest.mark.gpu

MAP, PAGE = 64, 256  # 64 x 64 maps of a 256-pixel detector input (scale 4)


@pytest.fixture(scope="module")
def mb():
    import manuscript_b200 as m

    return m


def dense_maps(n_pages, seed, q=2):
    """Every quantisation cell is a candidate (1024 per page) whose box depends only on its column and on its row mod 4:
    in x0 order, neighbours lie in different bands and never merge, while each box overlaps about two dozen others of
    its band -- about 12 suppression pairs per candidate (the default capacity is 16)."""
    rng = np.random.default_rng(seed)
    score = rng.uniform(0.7, 0.99, (n_pages, MAP, MAP)).astype(np.float32)
    geo = np.zeros((n_pages, 8, MAP, MAP), np.float32)
    c = np.arange(MAP // q)
    cy, cx = np.meshgrid(c, c, indexing="ij")
    y, x = cy * q + q // 2, cx * q + q // 2
    x0 = cx * q + rng.uniform(0, 0.5, (n_pages, 1, 1))
    y0 = (cy % 4) * 16 + 2 + rng.uniform(0, 0.5, (n_pages, 1, 1))
    for k, (vx, vy) in enumerate([(x0, y0), (x0 + 6, y0), (x0 + 6, y0 + 8), (x0, y0 + 8)]):  # TL, TR, BR, BL
        geo[:, 2 * k, y, x] = vx - x
        geo[:, 2 * k + 1, y, x] = vy - y
    return score, geo


def host_result(res):
    """Copies of a host-form PageBatchResult (its arrays are views of the runner's reused buffers)."""
    n = int(res.n_crops[0])
    counts = res.box_counts.copy()
    boxes = [res.boxes[p, : counts[p]].copy() for p in range(len(counts))]
    return counts, boxes, res.crops[:n].copy(), res.batch[:n].cpu().numpy(), res.flags.copy()


def assert_same(got, want):
    for a, b in zip(got[:1] + got[2:], want[:1] + want[2:]):
        np.testing.assert_array_equal(a, b)
    for a, b in zip(got[1], want[1]):
        np.testing.assert_array_equal(a, b)


def runner(mb, edge_factor=None):
    r = mb.PageBatch(device=0, params=mb.EastParams.default(target_size=PAGE), cap_boxes=1024)
    if edge_factor is not None:
        r.ctx.edge_factor = edge_factor
    return r


@pytest.mark.parametrize("ragged", [False, True])
def test_host_page_batch_grows_the_pair_capacity(mb, ragged):
    n_pages = 9  # five upload chunks of the uniform host form
    score, geo = dense_maps(n_pages, 5)
    rng = np.random.default_rng(6)
    if ragged:
        sizes = [(PAGE, PAGE), (300, 280), (256, 320)]
        imgs = [rng.integers(0, 256, sizes[p % 3] + (3,), dtype=np.uint8) for p in range(n_pages)]
        run = lambda r: r.run_host_ragged(score, geo, imgs)  # noqa: E731
    else:
        imgs = rng.integers(0, 256, (n_pages, PAGE, PAGE, 3), dtype=np.uint8)
        run = lambda r: r.run_host(score, geo, imgs)  # noqa: E731
    want = host_result(run(runner(mb)))
    grown = runner(mb, edge_factor=1)
    got = host_result(run(grown))
    assert grown.ctx.edge_factor > 1, "the call did not overflow the pair capacity"
    assert_same(got, want)
    assert not want[4].any() and all(len(b) > 20 for b in want[1]) and len(want[2]) > 100


def test_standard_nms_host_grows_the_pair_capacity(mb):
    rng = np.random.default_rng(17)
    n = 1000
    rect = np.array([[0, 0], [1, 0], [1, 1], [0, 1]], float)
    polys = rng.uniform(0, 260, (n, 1, 2)) + rect * rng.uniform(15, 45, (n, 1, 2))
    scores = rng.uniform(0.3, 1, n)
    want = mb.standard_nms(polys, scores, 0.1, return_index=True, ctx=mb.Context(0))
    ctx = mb.Context(0)
    ctx.edge_factor = 1
    got = mb.standard_nms(polys, scores, 0.1, return_index=True, ctx=ctx)
    assert ctx.edge_factor > 1, "the call did not overflow the pair capacity"
    np.testing.assert_array_equal(got, want)
    np.testing.assert_array_equal(got, cpu.standard_nms(polys, scores, 0.1, return_index=True))


@pytest.mark.parametrize("field,a,b", [("min_text_size", 5, 100), ("score_thresh", 0.6, 0.8)])
def test_graph_key_tells_calls_apart(mb, monkeypatch, field, a, b):
    import torch

    score, geo, imgs = synthdata.make_batch([71, 72], 512, 60)
    s, g, im = (torch.from_numpy(t).cuda() for t in (score, geo, imgs))

    def call(r, v):
        if field == "min_text_size":
            r.min_text_size = v
        else:
            r.params.score_thresh = v
        res = r.run(s, g, im)
        n = int(res.n_crops.cpu()[0])
        counts = res.box_counts.cpu().numpy()
        boxes = res.boxes.cpu().numpy()
        return (counts, np.concatenate([boxes[p, : counts[p]] for p in range(len(counts))]),
                res.crops[:n].cpu().numpy(), res.batch[:n].cpu().numpy(), res.flags.cpu().numpy())

    def make():
        return mb.PageBatch(device=0, params=mb.EastParams.default(target_size=512), cap_boxes=512)

    monkeypatch.setenv("MS_B200_NO_GRAPHS", "1")
    direct = make()
    monkeypatch.delenv("MS_B200_NO_GRAPHS")
    want = {v: call(direct, v) for v in (a, b)}
    if all(np.array_equal(w, x) for w, x in zip(want[a], want[b])):
        pytest.fail(f"{field} = {a} and {b} give the same results: the test cannot tell the graphs apart")
    cached = make()
    for v in (a, b) * 3:  # direct launches, capture, then replays of each
        for w, x in zip(call(cached, v), want[v]):
            np.testing.assert_array_equal(w, x)
