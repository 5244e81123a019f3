"""Page batches whose crop stage is the rectified crop of every final quad (ms_page_batch_quads,
ms_page_batch_ragged_quads, PageBatch(crops="quads")) and Pipeline(rotated_crops=True) on the fused routes.

The crop list and every crop row are checked against the standalone ms_quad_crop_resize_pad_ex of the same quads, the
boxes against ms_page_batch_ragged_ex, and a sample of rows against the oracle."""
import ctypes as C

import numpy as np
import pytest

import synthdata
from oracle import cpu

pytestmark = pytest.mark.gpu

T = 512          # detector target size: maps are (T/4, T/4)
OUT_H, OUT_W = 32, 128
MIN_TEXT = 5
CAP_BOXES = 512
# a 2048-wide page (rows a multiple of 16 bytes, aligned base: the staged kernel), widths that are not a multiple of
# 16, a long thin page, and one page at an odd address
SHAPES = [(700, 2048), (333, 517), (900, 640), (1031, 777), (512, 512), (64, 1500), (1200, 1000), (450, 1111), (800, 600)]
STAGED = 0
UNALIGNED = 6
SENTINEL = -7


@pytest.fixture(scope="module")
def mb():
    import manuscript_b200 as m

    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t

    assert t.cuda.is_available()
    return t


@pytest.fixture(scope="module")
def ctx(mb):
    return mb.Context(0)


def stream_of(torch):
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


@pytest.fixture(scope="module")
def data(torch):
    maps = [synthdata.make_maps(500 + i, T, 70) for i in range(len(SHAPES))]
    score = torch.from_numpy(np.stack([m[0] for m in maps])).cuda()
    geo = torch.from_numpy(np.stack([m[1] for m in maps])).cuda()
    imgs = [synthdata.make_page_image(600 + i, max(h, w))[:h, :w].copy() for i, (h, w) in enumerate(SHAPES)]
    keep, ptrs = [], []
    for i, img in enumerate(imgs):
        off = 3 if i == UNALIGNED else 0
        buf = torch.zeros(img.nbytes + off + 16, dtype=torch.uint8, device="cuda")
        buf[off:off + img.nbytes].copy_(torch.from_numpy(img.reshape(-1)))
        keep.append(buf)
        ptrs.append(buf.data_ptr() + off)
    assert ptrs[UNALIGNED] % 16 != 0 and ptrs[STAGED] % 16 == 0
    d_ptrs = torch.tensor(ptrs, dtype=torch.int64, device="cuda")
    d_hw = torch.tensor([list(s) for s in SHAPES], dtype=torch.int32, device="cuda")
    return dict(score=score, geo=geo, imgs=imgs, keep=keep, ptrs=ptrs, d_ptrs=d_ptrs, d_hw=d_hw)


def params(mb):
    return mb.EastParams.default(target_size=T, axis_aligned_output=0, sort_reading_order=1)


class Out:
    """Output buffers of one page-batch call, filled with sentinels"""

    def __init__(self, mb, torch, n_pages, rows, dtype, canvas=False):
        self.dtype_code = mb.batch_dtype_code(dtype if dtype is not None else torch.float32)
        self.boxes = torch.full((n_pages, CAP_BOXES, 9), -1.0, dtype=torch.float32, device="cuda")
        self.counts = torch.zeros((n_pages,), dtype=torch.int32, device="cuda")
        self.crops = torch.full((rows, 5), SENTINEL, dtype=torch.int32, device="cuda")
        self.n = torch.full((1,), SENTINEL, dtype=torch.int32, device="cuda")
        self.batch = torch.full((rows, 3, OUT_H, OUT_W), SENTINEL, dtype=dtype, device="cuda") if dtype else None
        self.canvas = torch.full((rows, OUT_H, OUT_W, 3), 201, dtype=torch.uint8, device="cuda") if canvas else None
        self.flags = torch.full((n_pages,), SENTINEL, dtype=torch.int32, device="cuda")

    def tail(self, cap):
        """the arguments from out_h on, without the stream"""
        return (OUT_H, OUT_W, CAP_BOXES, self.boxes.data_ptr(), self.counts.data_ptr(), self.crops.data_ptr(), cap,
                self.n.data_ptr(), self.batch.data_ptr() if self.batch is not None else None, self.dtype_code,
                self.canvas.data_ptr() if self.canvas is not None else None, self.flags.data_ptr())


def page_views(d):
    """the pages as (h, w, 3) CUDA tensors (views of the test's buffers)"""
    return [d["keep"][i][(3 if i == UNALIGNED else 0):][:img.nbytes].view(img.shape) for i, img in enumerate(d["imgs"])]


def ragged_quads(mb, torch, ctx, d, border=(0, 0), dtype="f32", cap=None, rows=None, canvas=False):
    """dtype None: no batch (the u8 canvas only)"""
    dtype = torch.float32 if dtype == "f32" else dtype
    P = len(SHAPES)
    cap = P * CAP_BOXES if cap is None else cap
    o = Out(mb, torch, P, rows or cap, dtype, canvas)
    rc = ctx.lib.ms_page_batch_ragged_quads(ctx.handle, d["score"].data_ptr(), d["geo"].data_ptr(),
                                            d["d_ptrs"].data_ptr(), d["d_hw"].data_ptr(), P, T // 4, T // 4,
                                            C.byref(params(mb)), MIN_TEXT, border[0], border[1],
                                            *o.tail(cap), stream_of(torch))
    assert rc == 0, mb._cabi.last_error()
    torch.cuda.synchronize()
    return o


def host(o):
    n = int(o.n.cpu()[0])
    return o.counts.cpu().numpy(), o.boxes.cpu().numpy(), o.crops.cpu().numpy(), n


def standalone(mb, torch, ctx, d, p, quads, border, dtype=None, canvas=False):
    """ms_quad_crop_resize_pad_ex of one page's quads (rows of 9 floats)"""
    dtype = torch.float32 if dtype is None else dtype
    h, w = SHAPES[p]
    n = len(quads)
    q = torch.from_numpy(np.ascontiguousarray(quads, dtype=np.float32)).cuda()
    batch = torch.zeros((n, 3, OUT_H, OUT_W), dtype=dtype, device="cuda")
    can = torch.zeros((n, OUT_H, OUT_W, 3), dtype=torch.uint8, device="cuda") if canvas else None
    sizes = torch.zeros((n, 2), dtype=torch.int32, device="cuda")
    rc = ctx.lib.ms_quad_crop_resize_pad_ex(ctx.handle, d["ptrs"][p], 1, h, w, q.data_ptr(), 9, None, n, MIN_TEXT,
                                            border[0], border[1], OUT_H, OUT_W, batch.data_ptr(),
                                            mb.batch_dtype_code(dtype), can.data_ptr() if canvas else None,
                                            sizes.data_ptr(), stream_of(torch))
    assert rc == 0, mb._cabi.last_error()
    torch.cuda.synchronize()
    return batch, can, sizes.cpu().numpy()


def expected_list(counts, boxes):
    rows = []
    for p in range(len(SHAPES)):
        for b in range(int(counts[p])):
            w, h = cpu.quad_patch_size(boxes[p, b, :8])
            if w >= max(2, MIN_TEXT) and h >= max(2, MIN_TEXT):
                rows.append((p, b, w, h, 0))
    return np.array(rows, np.int32).reshape(-1, 5)


@pytest.mark.parametrize("border", [(0, 0), (1, 0), (0, 77)])
def test_ragged_quads_against_standalone_and_oracle(mb, torch, ctx, data, border):
    d = data
    o = ragged_quads(mb, torch, ctx, d, border)
    staged = (C.c_int32 * 2)()
    assert ctx.lib.ms_quad_crop_last_counts(ctx.handle, staged) == 0
    counts, boxes, crops, n = host(o)
    assert not o.flags.cpu().numpy().any()
    # the front stages are those of the rectangle page batch: same bits
    ref = mb.PageBatch(device=0, params=params(mb), cap_boxes=CAP_BOXES, out_hw=(OUT_H, OUT_W),
                       min_text_size=MIN_TEXT).run_ragged(d["score"], d["geo"], page_views(d))
    torch.cuda.synchronize()
    np.testing.assert_array_equal(counts, ref.box_counts.cpu().numpy())
    for p in range(len(SHAPES)):
        np.testing.assert_array_equal(boxes[p, :counts[p]], ref.boxes[p, :counts[p]].cpu().numpy())
    # the list: every quad with a patch (the synthetic quads are never singular), in (page, box) order
    want = expected_list(counts, boxes)
    assert n == len(want) and n > 200
    np.testing.assert_array_equal(crops[:n], want)
    assert (crops[n:] == SENTINEL).all()
    assert staged[0] > 0 and staged[0] + staged[1] >= n  # the 2048-wide page is served by the staged kernel
    batch = o.batch[:n]
    for p in range(len(SHAPES)):
        mine = np.flatnonzero(crops[:n, 0] == p)
        if not len(mine):
            continue
        sb, _, sizes = standalone(mb, torch, ctx, d, p, boxes[p, :counts[p]], border)
        bx = crops[mine, 1]
        np.testing.assert_array_equal(sizes[bx], crops[mine, 2:4])
        assert torch.equal(batch[torch.from_numpy(mine).cuda()], sb[torch.from_numpy(bx).cuda()]), f"page {p}"
        for j in mine[:: max(1, len(mine) // 4)][:4]:  # a sample against the oracle
            _, chw = cpu.quad_crop_resize_pad(d["imgs"][p], boxes[p, crops[j, 1], :8], OUT_H, OUT_W, MIN_TEXT,
                                              "replicate" if border[0] else "constant", border[1])
            np.testing.assert_array_equal(batch[j].cpu().numpy(), chw, err_msg=f"page {p} row {j}")
    assert (o.batch[n:].cpu().numpy() == SENTINEL).all()  # rows past the list are not written


def test_uniform_equals_ragged(mb, torch, ctx):
    P, H, W = 4, 600, 800
    maps = [synthdata.make_maps(700 + i, T, 70) for i in range(P)]
    score = torch.from_numpy(np.stack([m[0] for m in maps])).cuda()
    geo = torch.from_numpy(np.stack([m[1] for m in maps])).cuda()
    pages = torch.from_numpy(np.stack([synthdata.make_page_image(710 + i, W)[:H, :W] for i in range(P)])).cuda()
    cap = P * CAP_BOXES
    outs = []
    for uniform in (True, False):
        o = Out(mb, torch, P, cap, torch.float32, canvas=True)
        if uniform:
            rc = ctx.lib.ms_page_batch_quads(ctx.handle, score.data_ptr(), geo.data_ptr(), pages.data_ptr(), P, T // 4,
                                             T // 4, H, W, C.byref(params(mb)), MIN_TEXT, 1, 0,
                                             *o.tail(cap), stream_of(torch))
        else:
            ptrs = torch.tensor([pages[i].data_ptr() for i in range(P)], dtype=torch.int64, device="cuda")
            hw = torch.tensor([[H, W]] * P, dtype=torch.int32, device="cuda")
            rc = ctx.lib.ms_page_batch_ragged_quads(ctx.handle, score.data_ptr(), geo.data_ptr(), ptrs.data_ptr(),
                                                    hw.data_ptr(), P, T // 4, T // 4, C.byref(params(mb)), MIN_TEXT,
                                                    1, 0, *o.tail(cap), stream_of(torch))
        assert rc == 0, mb._cabi.last_error()
        torch.cuda.synchronize()
        outs.append(o)
    a, b = outs
    n = int(a.n.cpu()[0])
    assert n == int(b.n.cpu()[0]) and n > 100
    for x, y in ((a.counts, b.counts), (a.crops, b.crops), (a.batch, b.batch), (a.canvas, b.canvas), (a.flags, b.flags)):
        assert torch.equal(x, y)
    for p in range(P):
        k = int(a.counts[p])
        assert torch.equal(a.boxes[p, :k], b.boxes[p, :k])


@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
def test_16bit_batch_is_f32_cast_and_u8_canvas(mb, torch, ctx, data, dtype):
    dt = getattr(torch, dtype)
    ref = ragged_quads(mb, torch, ctx, data, (0, 0), canvas=True)
    got = ragged_quads(mb, torch, ctx, data, (0, 0), dtype=dt, canvas=True)
    n = int(ref.n.cpu()[0])
    assert torch.equal(got.crops, ref.crops) and int(got.n.cpu()[0]) == n
    assert torch.equal(got.batch[:n].view(torch.int16), ref.batch[:n].to(dt).view(torch.int16))
    assert torch.equal(got.canvas, ref.canvas)
    # the canvases are those of the standalone call
    counts, boxes, crops, _ = host(ref)
    for p in (STAGED, UNALIGNED):
        mine = np.flatnonzero(crops[:n, 0] == p)
        _, can, _ = standalone(mb, torch, ctx, data, p, boxes[p, :counts[p]], (0, 0), canvas=True)
        assert torch.equal(ref.canvas[torch.from_numpy(mine).cuda()], can[torch.from_numpy(crops[mine, 1]).cuda()])
    # u8 canvas only (no batch)
    only = ragged_quads(mb, torch, ctx, data, (0, 0), dtype=None, canvas=True)
    assert torch.equal(only.canvas, ref.canvas)


def test_crops_cap_below_the_list(mb, torch, ctx, data):
    full = ragged_quads(mb, torch, ctx, data, (0, 0))
    n = int(full.n.cpu()[0])
    cap = n // 2 + 3
    o = ragged_quads(mb, torch, ctx, data, (0, 0), cap=cap, rows=n)
    assert int(o.n.cpu()[0]) == cap
    assert torch.equal(o.crops[:cap], full.crops[:cap])
    assert (o.crops[cap:].cpu().numpy() == SENTINEL).all()
    assert torch.equal(o.batch[:cap], full.batch[:cap])
    assert (o.batch[cap:].cpu().numpy() == SENTINEL).all()


def test_repeated_call_replays_a_graph_keyed_by_crop_mode_and_border(mb, torch, data):
    d = data
    pages = page_views(d)

    def runner(**kw):
        return mb.PageBatch(device=0, params=params(mb), cap_boxes=CAP_BOXES, out_hw=(OUT_H, OUT_W),
                            min_text_size=MIN_TEXT, **kw)

    r = runner(crops="quads")

    def snapshot(**kw):
        for k, v in kw.items():
            setattr(r, k, v)
        res = r.run_ragged(d["score"], d["geo"], pages)
        torch.cuda.synchronize()
        n = int(res.n_crops.cpu()[0])
        return res.box_counts.cpu().numpy().copy(), res.crops[:n].cpu().numpy().copy(), res.batch[:n].clone()

    l0 = r.ctx.launches
    first = snapshot()
    per_call = r.ctx.launches - l0
    second = snapshot()
    third = snapshot()
    assert r.ctx.launches - l0 == 3 * per_call and per_call > 20
    for a, b, c in zip(first, second, third):
        assert np.array_equal(a, b) if isinstance(a, np.ndarray) else torch.equal(a, b)
        assert np.array_equal(a, c) if isinstance(a, np.ndarray) else torch.equal(a, c)
    # the same buffers with another border, then as rectangles: each is its own call, not a replay of the other's graph
    for kw, fresh_kw in ((dict(border_mode=0, border_value=77), dict(crops="quads", border_value=77)),
                         (dict(border_mode=1, border_value=0), dict(crops="quads", border_mode=1)),
                         (dict(crops="rects", border_mode=0), dict(crops="rects"))):
        for _ in range(3):
            got = snapshot(**kw)
        f = runner(**fresh_kw).run_ragged(d["score"], d["geo"], pages)
        torch.cuda.synchronize()
        n = int(f.n_crops.cpu()[0])
        np.testing.assert_array_equal(got[1], f.crops[:n].cpu().numpy())
        assert torch.equal(got[2], f.batch[:n])
    assert not np.array_equal(got[1], first[1])


def test_invalid_arguments(mb, torch, ctx, data):
    d = data
    P = len(SHAPES)
    o = Out(mb, torch, P, 16, torch.float32)
    lib, h, s = ctx.lib, ctx.handle, stream_of(torch)
    prm = C.byref(params(mb))

    def ragged(ptrs, hw, bm, bv, dtype=0):
        t = list(o.tail(16))
        t[9] = dtype
        return lib.ms_page_batch_ragged_quads(h, d["score"].data_ptr(), d["geo"].data_ptr(), ptrs, hw, P, T // 4,
                                              T // 4, prm, MIN_TEXT, bm, bv, *t, s)

    P_, HW = d["d_ptrs"].data_ptr(), d["d_hw"].data_ptr()
    bad = [(P_, HW, 2, 0), (P_, HW, -1, 0), (P_, HW, 0, 256), (P_, HW, 0, -1), (None, HW, 0, 0), (P_, None, 0, 0),
           (P_, HW, 0, 0, 7)]
    for args in bad:
        assert ragged(*args) == mb._cabi.MS_ERR_INVALID, args
    big = torch.zeros((16,), dtype=torch.uint8, device="cuda")
    for ih, iw in ((40000, 100), (100, 40000), (0, 100)):
        rc = lib.ms_page_batch_quads(h, d["score"].data_ptr(), d["geo"].data_ptr(), big.data_ptr(), 1, T // 4, T // 4,
                                     ih, iw, prm, MIN_TEXT, 0, 0, *o.tail(16), s)
        assert rc == mb._cabi.MS_ERR_INVALID, (ih, iw)
    assert ragged(P_, HW, 0, 0) == 0
    torch.cuda.synchronize()


# ---- Pipeline(rotated_crops=True) on the fused routes ---------------------------------------------------------------
from test_gpu_batch_pipeline import T as PT  # noqa: E402
from test_gpu_batch_pipeline import StubEAST, StubTRBA, page_fields, page_images  # noqa: E402


class NotEAST:
    """A detector that is not this package's EAST (so Pipeline takes the per-image route) and answers with the words
    the wrapped EAST finds."""

    def __init__(self, det):
        self.det = det

    def predict(self, image, vis=False, profile=False):
        return self.det.predict(image, vis=vis, profile=profile)


def rotated_pipe(mb, torch, per_image=False, batch_dtype=None, batch_size=24):
    net = StubEAST(torch, torch.float32)
    det = mb.EAST(model=net, target_size=PT, axis_aligned_output=False)
    rec_net = StubTRBA()
    rec = mb.TRBA(model=rec_net, img_h=32, img_w=128, batch_size=batch_size, batch_dtype=batch_dtype)
    pipe = mb.Pipeline(detector=NotEAST(det) if per_image else det, recognizer=rec, rotated_crops=True)
    return pipe, det, rec_net


@pytest.fixture(scope="module")
def per_image_ref(mb, torch):
    imgs = page_images()
    pipe, _, rec_net = rotated_pipe(mb, torch, per_image=True)
    pages = [pipe.predict(img) for img in imgs]
    assert pipe.last_route == "rotated_crops"
    return imgs, [page_fields(p) for p in pages], torch.cat(rec_net.batches)


def test_pipeline_predict_fused_rotated(mb, torch, per_image_ref):
    imgs, want, want_rows = per_image_ref
    pipe, det, rec_net = rotated_pipe(mb, torch)
    uploads = []
    orig = det.upload
    det.upload = lambda img: (uploads.append(1), orig(img))[1]
    got = []
    for img in imgs:
        got.append(page_fields(pipe.predict(img)))
        assert pipe.last_route == "fused_rotated"
    assert got == want
    assert len(uploads) == len(imgs)
    assert torch.equal(torch.cat(rec_net.batches), want_rows)
    assert sum(len(b) for b in got[2]) == 0 and any(w[2] for b in got[0] for w in b)  # a blank page; texts


def test_pipeline_process_batch_fused_rotated(mb, torch, per_image_ref):
    imgs, want, want_rows = per_image_ref
    pipe, det, rec_net = rotated_pipe(mb, torch)
    uploads = []
    orig = det.upload_batch
    det.upload = None  # the batched route never uploads page by page
    det.upload_batch = lambda images: (uploads.append(len(images)), orig(images))[1]
    got = pipe.process_batch(imgs, max_pages=4)
    assert pipe.last_route == "fused_batch_rotated"
    assert [page_fields(p) for p in got] == want
    assert uploads == [4, 2]
    assert all(len(b) <= 24 for b in rec_net.batches)
    assert torch.equal(torch.cat(rec_net.batches), want_rows)
    again = pipe.process_batch(imgs, max_pages=4)  # replayed page batch
    assert [page_fields(p) for p in again] == want


def test_pipeline_rotated_crop_buffer_growth(mb, torch, per_image_ref, monkeypatch):
    import manuscript_b200.pipeline as pl

    imgs, want, _ = per_image_ref
    monkeypatch.setattr(pl, "_BATCH_CROPS_CAP0", 8)
    pipe, _, _ = rotated_pipe(mb, torch)
    assert [page_fields(p) for p in pipe.process_batch(imgs, max_pages=4)] == want
    cap = pipe._fused_runner(batch=True).crops_cap
    assert cap > 8 and cap & (cap - 1) == 0
    assert [page_fields(p) for p in pipe.process_batch(imgs[:3], max_pages=4)] == want[:3]


def test_pipeline_rotated_page_ordered_on_the_host(mb, torch, per_image_ref, monkeypatch):
    """a page flagged MS_FLAG_ORDER_OVERFLOW: its rows are dropped and it is finished on the host from the page already
    on the device"""
    from manuscript_b200.batch import PageBatchResult

    imgs, want, _ = per_image_ref
    pipe, _, _ = rotated_pipe(mb, torch)
    orig = PageBatchResult.order_overflow_pages
    monkeypatch.setattr(PageBatchResult, "order_overflow_pages",
                        lambda self: np.array([1]) if len(self.flags) > 1 else orig(self))
    dev_pages = []
    orig_rot = pipe._recognise_rotated
    pipe._recognise_rotated = lambda a, w, page_dev=None: (dev_pages.append(page_dev), orig_rot(a, w, page_dev))[1]
    got = pipe.process_batch(imgs, max_pages=4)
    assert pipe.last_route == "fused_batch_rotated"
    assert [page_fields(p) for p in got] == want
    # page 1 of each of the two chunks, each cut from its upload (no second upload)
    assert len(dev_pages) == 2 and all(p is not None for p in dev_pages)


def test_pipeline_rotated_16bit_batch(mb, torch):
    imgs = page_images()[:4]
    ref, _, ref_net = rotated_pipe(mb, torch, per_image=True, batch_dtype=torch.float16)
    want = [page_fields(ref.predict(img)) for img in imgs]
    pipe, _, rec_net = rotated_pipe(mb, torch, batch_dtype=torch.float16)
    assert [page_fields(p) for p in pipe.process_batch(imgs)] == want
    assert rec_net.batches[0].dtype == torch.float16
    assert torch.equal(torch.cat(rec_net.batches).view(torch.int16), torch.cat(ref_net.batches).view(torch.int16))
