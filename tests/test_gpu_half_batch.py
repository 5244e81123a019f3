"""The recogniser batch in float16 / bfloat16 (an extension): every crop route, the batched entry points, the CUDA-graph
cache and the classes write exactly the float32 batch cast with .to(dtype) -- compared bit for bit on the int16 view
against the float32 result of the same call."""
import ctypes as C

import numpy as np
import pytest

import synthdata

pytestmark = pytest.mark.gpu

DTYPES = ["float16", "bfloat16"]


@pytest.fixture(scope="module")
def mb():
    import manuscript_b200 as m

    return m


@pytest.fixture(scope="module")
def torch():
    import torch as t

    return t


@pytest.fixture(scope="module")
def ctx(mb):
    return mb.Context(0)


def assert_cast(got, ref32, dtype):
    """got (16-bit tensor) == ref32.to(dtype), bit for bit"""
    import torch

    want = ref32.to(dtype)
    assert got.dtype == dtype and got.shape == want.shape
    bad = (got.contiguous().view(torch.int16) != want.view(torch.int16)).sum().item()
    assert bad == 0, f"{bad} values differ from the float32 batch cast to {dtype}"


def stream_of(torch):
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


# ---- the axis-aligned crop kernels through ms_crop_resize_pad_ex ----------------------------------------------------
def route_rects(rng, H, W):
    """[x1, y1, x2, y2) rectangles that take every route at a 32 x 128 canvas (and a spread at the others)"""
    r = [
        (5, 7, 155, 57),      # shrink factor < 2: 3-tap INTER_AREA (persistent kernel)
        (3, 4, 303, 84),      # shrink factor 2.5: 4-tap INTER_AREA
        (10, 20, 266, 84),    # exactly 2 x 2: integer-ratio routine of the persistent kernel
        (40, 30, 70, 40),     # INTER_LINEAR upscale (generic kernel)
        (11, 13, 111, 45),    # same size: copy
        (1, 2, 471, 172),     # shrink factor 5.3: long tables (generic kernel)
        (2, 3, 386, 99),      # exactly 3 x 3 integer ratio (generic kernel)
        (0, 5, 450, 45),      # rows too long for the staging ring (generic kernel)
        (50, 50, 50, 90),     # empty: invalid
        (W - 10, 5, W + 20, 40),  # outside the page: invalid
    ]
    for _ in range(120):
        h = int(rng.integers(6, 150))
        w = int(rng.integers(6, 420))
        x, y = int(rng.integers(0, W - w)), int(rng.integers(0, H - h))
        r.append((x, y, x + w, y + h))
    return np.array(r, np.int32)


def crop_call(mb, torch, ctx, pages, crops, out_h, out_w, dtype, canvas=False, offset=0):
    n = len(crops)
    d_crops = torch.from_numpy(crops).cuda()
    n_dev = torch.tensor([n], dtype=torch.int32, device="cuda")
    buf = torch.zeros(n * 3 * out_h * out_w + offset, dtype=dtype, device="cuda")
    batch = buf[offset:].view(n, 3, out_h, out_w)
    can = torch.zeros((n, out_h, out_w, 3), dtype=torch.uint8, device="cuda") if canvas else None
    rc = ctx.lib.ms_crop_resize_pad_ex(ctx.handle, pages.data_ptr(), int(pages.shape[0]), int(pages.shape[1]),
                                       int(pages.shape[2]), d_crops.data_ptr(), n_dev.data_ptr(), n, out_h, out_w,
                                       batch.data_ptr(), mb._cabi.batch_dtype_code(dtype),
                                       can.data_ptr() if canvas else None, stream_of(torch))
    assert rc == 0, mb._cabi.last_error()
    torch.cuda.synchronize()
    return batch, can


@pytest.mark.parametrize("dt", DTYPES)
def test_crop_kernels_every_route(mb, torch, ctx, dt):
    dtype = getattr(torch, dt)
    rng = np.random.default_rng(11)
    # page rows of 1536 bytes (a multiple of 16) and of 1503 bytes (not: every staged row has its own misalignment)
    for W in (512, 501):
        H = 400
        imgs = rng.integers(0, 256, (2, H, W, 3), dtype=np.uint8)
        pages = torch.from_numpy(imgs).cuda()
        rects = route_rects(rng, H, W)
        crops = np.zeros((len(rects), 5), np.int32)
        crops[:, 0] = rng.integers(0, 2, len(rects))
        crops[:, 1:] = rects
        crops[12, 0] = 7  # page out of range: invalid
        for out_h, out_w in ((32, 128), (64, 256), (30, 100)):  # 100 % 8 != 0: scalar padding for 16-bit elements
            ref, ref_can = crop_call(mb, torch, ctx, pages, crops, out_h, out_w, torch.float32, canvas=True)
            got, _ = crop_call(mb, torch, ctx, pages, crops, out_h, out_w, dtype)
            assert_cast(got, ref, dtype)
            # with the u8 canvas beside it: the same batch, the float32 run's canvas
            got, can = crop_call(mb, torch, ctx, pages, crops, out_h, out_w, dtype, canvas=True)
            assert_cast(got, ref, dtype)
            assert torch.equal(can, ref_can)
        # a batch one element past a 16-byte boundary: the padding writer's unaligned path
        ref, _ = crop_call(mb, torch, ctx, pages, crops, 32, 128, torch.float32)
        got, _ = crop_call(mb, torch, ctx, pages, crops, 32, 128, dtype, offset=1)
        assert_cast(got, ref, dtype)


# ---- rotated quads through ms_quad_crop_resize_pad_ex -----------------------------------------------------------------
def rotated_quads(rng, n, H, W):
    q = []
    for i in range(n):
        big = i % 10 == 0  # a patch too large for the staged kernel's bands
        ww = rng.uniform(300, 600) if big else rng.uniform(30, 220)
        hh = rng.uniform(60, 120) if big else rng.uniform(18, 70)
        cx, cy = rng.uniform(ww / 2 + 20, W - ww / 2 - 20), rng.uniform(hh / 2 + 20, H - hh / 2 - 20)
        a = rng.uniform(-0.15, 0.15)
        c, s = np.cos(a), np.sin(a)
        p = np.array([[-ww / 2, -hh / 2], [ww / 2, -hh / 2], [ww / 2, hh / 2], [-ww / 2, hh / 2]]) @ np.array(
            [[c, s], [-s, c]]) + [cx, cy]
        q.append(p.reshape(-1))
    return np.array(q, np.float32)


@pytest.mark.parametrize("dt", DTYPES)
def test_rotated_quads_staged_and_generic(mb, torch, ctx, dt):
    dtype = getattr(torch, dt)
    rng = np.random.default_rng(21)
    H, W = 600, 1024  # rows of 3072 bytes: 16-byte aligned, the staged kernel takes the quads it can
    pages = torch.from_numpy(rng.integers(0, 256, (2, H, W, 3), dtype=np.uint8)).cuda()
    n = 300
    quads = torch.from_numpy(rotated_quads(rng, n, H, W)).cuda()
    page_of = torch.from_numpy(rng.integers(0, 2, n).astype(np.int32)).cuda()

    def run(dtype, canvas):
        batch = torch.zeros((n, 3, 32, 128), dtype=dtype, device="cuda")
        can = torch.zeros((n, 32, 128, 3), dtype=torch.uint8, device="cuda") if canvas else None
        sizes = torch.zeros((n, 2), dtype=torch.int32, device="cuda")
        rc = ctx.lib.ms_quad_crop_resize_pad_ex(ctx.handle, pages.data_ptr(), 2, H, W, quads.data_ptr(), 8,
                                                page_of.data_ptr(), n, 5, 0, 0, 32, 128, batch.data_ptr(),
                                                mb._cabi.batch_dtype_code(dtype), can.data_ptr() if canvas else None,
                                                sizes.data_ptr(), stream_of(torch))
        assert rc == 0, mb._cabi.last_error()
        counts = (C.c_int32 * 2)()
        assert ctx.lib.ms_quad_crop_last_counts(ctx.handle, counts) == 0
        torch.cuda.synchronize()
        return batch, can, sizes, tuple(counts)

    ref, ref_can, ref_sizes, ref_counts = run(torch.float32, True)
    for canvas in (False, True):
        got, can, sizes, counts = run(dtype, canvas)
        assert counts == ref_counts and counts[0] > 0 and counts[1] > 0  # both kernels served quads
        assert torch.equal(sizes, ref_sizes)
        assert_cast(got, ref, dtype)
        if canvas:
            assert torch.equal(can, ref_can)


# ---- the batched entry points (PageBatch's four run methods) on three pages of the benchmark corpus ----------------------
@pytest.fixture(scope="module")
def corpus3():
    score, geo, imgs = synthdata.make_batch([0, 1, 2], 2048, 2000)
    return score, geo, imgs


def same_results(res, ref, n, dtype):
    import torch

    as_t = (lambda a: (a if isinstance(a, torch.Tensor) else torch.from_numpy(np.asarray(a))).cpu())
    for name in ("box_counts", "flags"):
        assert torch.equal(as_t(getattr(res, name)), as_t(getattr(ref, name))), name
    for p, k in enumerate(as_t(ref.box_counts).tolist()):  # rows past a page's count are not written
        assert torch.equal(as_t(res.boxes)[p, :k], as_t(ref.boxes)[p, :k])
    assert int(as_t(res.n_crops).reshape(-1)[0]) == n
    assert torch.equal(as_t(res.crops).cpu()[:n], as_t(ref.crops).cpu()[:n])
    assert_cast(res.batch[:n], ref.batch[:n], dtype)


@pytest.mark.parametrize("dt", DTYPES)
def test_page_batch_four_run_methods(mb, torch, corpus3, dt):
    dtype = getattr(torch, dt)
    score, geo, imgs = corpus3
    params = mb.EastParams.default(target_size=2048)
    kw = dict(device=0, params=params, cap_boxes=4096, crops_cap=3 * 2600, out_hw=(32, 128))
    ref_r, half_r = mb.PageBatch(**kw), mb.PageBatch(batch_dtype=dtype, **kw)
    d_score, d_geo, d_pages = (torch.from_numpy(x).cuda() for x in (score, geo, imgs))
    # ms_page_batch_ex: the benchmark's pages, most crops taken by the persistent TMA kernel
    ref = ref_r.run(d_score, d_geo, d_pages, sync=True)
    n = int(ref.n_crops.item())
    assert n > 3000
    res = half_r.run(d_score, d_geo, d_pages, sync=True)
    assert res.batch.dtype == dtype
    same_results(res, ref, n, dtype)
    # ms_page_batch_ragged_ex: the same pages as images of their own (here equal) sizes
    pages_list = [d_pages[i] for i in range(3)]
    ref = ref_r.run_ragged(d_score, d_geo, pages_list, sync=True)
    res = half_r.run_ragged(d_score, d_geo, pages_list, sync=True)
    same_results(res, ref, n, dtype)
    # ms_page_batch_host_ex / ms_page_batch_ragged_host_ex: host buffers in, the batch in the runner's device tensor
    ref = ref_r.run_host(score, geo, imgs)
    res = half_r.run_host(score, geo, imgs)
    same_results(res, ref, n, dtype)
    ref = ref_r.run_host_ragged(score, geo, list(imgs))
    res = half_r.run_host_ragged(score, geo, list(imgs))
    same_results(res, ref, n, dtype)


@pytest.mark.parametrize("dt", DTYPES)
def test_page_batch_host_ex_downloads_16_bit(mb, torch, dt):
    """ms_page_batch_host_ex with a host batch and the library-owned device batch, both in 16 bits"""
    dtype = getattr(torch, dt)
    score, geo, imgs = synthdata.make_batch([4, 5], 1024, 400)
    ctx = mb.Context(0)
    params = mb.EastParams.default(target_size=1024)
    P, M = 2, 256
    cap_boxes, crops_cap = 1024, 900

    def run(dtype):
        boxes = np.zeros((P, cap_boxes, 9), np.float32)
        counts, flags = np.zeros(P, np.int32), np.zeros(P, np.int32)
        crops, nc = np.zeros((crops_cap, 5), np.int32), np.zeros(1, np.int32)
        host = torch.zeros((crops_cap, 3, 32, 128), dtype=dtype)
        dev = C.c_void_p(None)  # NULL on entry: the library's own device batch
        rc = ctx.lib.ms_page_batch_host_ex(ctx.handle, score.ctypes.data, geo.ctypes.data, imgs.ctypes.data, P, M, M,
                                           1024, 1024, C.byref(params), 5, 32, 128, cap_boxes, boxes.ctypes.data,
                                           counts.ctypes.data, crops.ctypes.data, crops_cap, nc.ctypes.data,
                                           host.data_ptr(), mb._cabi.batch_dtype_code(dtype), C.byref(dev),
                                           flags.ctypes.data)
        assert rc == 0, mb._cabi.last_error()
        n = int(nc[0])
        assert dev.value  # the library-owned device batch the host copy came from
        return boxes, counts, crops[:n], host[:n]

    rb, rc_, rcr, rbatch = run(torch.float32)
    hb, hc, hcr, hbatch = run(dtype)
    assert len(rcr) > 200
    np.testing.assert_array_equal(hc, rc_)
    for p, k in enumerate(rc_):
        np.testing.assert_array_equal(hb[p, :k], rb[p, :k])
    np.testing.assert_array_equal(hcr, rcr)
    assert_cast(hbatch, rbatch, dtype)


def test_graph_cache_keys_on_the_dtype(mb, torch):
    """One byte buffer, the same arguments, the dtype alternating: each dtype is recorded, captured and replayed as
    its own graph, and every call writes its own format."""
    score, geo, imgs = synthdata.make_batch([6, 7], 1024, 400)
    d_score, d_geo, d_pages = (torch.from_numpy(x).cuda() for x in (score, geo, imgs))
    params = mb.EastParams.default(target_size=1024)
    ref_r = mb.PageBatch(device=0, params=params, cap_boxes=1024, crops_cap=900)
    ref = ref_r.run(d_score, d_geo, d_pages, sync=True)
    n = int(ref.n_crops.item())
    assert n > 200
    ctx = mb.Context(0)
    P, M, cap = 2, 256, 900
    buf = torch.zeros(cap * 3 * 32 * 128 * 4, dtype=torch.uint8, device="cuda")
    boxes = torch.zeros((P, 1024, 9), dtype=torch.float32, device="cuda")
    counts, flags = torch.zeros(P, dtype=torch.int32, device="cuda"), torch.zeros(P, dtype=torch.int32, device="cuda")
    crops, nc = torch.zeros((cap, 5), dtype=torch.int32, device="cuda"), torch.zeros(1, dtype=torch.int32, device="cuda")
    for dtype in [torch.float32, torch.float16, torch.bfloat16] * 4:
        buf.fill_(0xAB)
        rc = ctx.lib.ms_page_batch_ex(ctx.handle, d_score.data_ptr(), d_geo.data_ptr(), d_pages.data_ptr(), P, M, M,
                                      1024, 1024, C.byref(params), 5, 32, 128, 1024, boxes.data_ptr(), counts.data_ptr(),
                                      crops.data_ptr(), cap, nc.data_ptr(), buf.data_ptr(),
                                      mb._cabi.batch_dtype_code(dtype), None, flags.data_ptr(), stream_of(torch))
        assert rc == 0, mb._cabi.last_error()
        torch.cuda.synchronize()
        assert int(nc.item()) == n and torch.equal(crops[:n], ref.crops[:n]) and int(flags.abs().sum()) == 0
        size = torch.empty(0, dtype=dtype).element_size()
        got = buf[: n * 3 * 32 * 128 * size].view(dtype).view(n, 3, 32, 128)
        if dtype == torch.float32:
            assert torch.equal(got, ref.batch[:n])
        else:
            assert_cast(got, ref.batch[:n], dtype)


def test_unknown_dtype_is_invalid(mb, torch, ctx):
    lib, h = ctx.lib, ctx.handle
    z = None
    params = C.byref(mb.EastParams.default())

    def invalid(rc):
        assert rc == -1 and "dtype" in mb._cabi.last_error()

    invalid(lib.ms_crop_resize_pad_ex(h, z, 1, 8, 8, z, z, 1, 32, 128, z, 3, z, z))
    invalid(lib.ms_quad_crop_resize_pad_ex(h, z, 1, 8, 8, z, 8, z, 1, 5, 0, 0, 32, 128, z, 3, z, z, z))
    invalid(lib.ms_page_batch_ex(h, z, z, z, 1, 8, 8, 8, 8, params, 5, 32, 128, 8, z, z, z, 1, z, z, -1, z, z, z))
    invalid(lib.ms_page_batch_ragged_ex(h, z, z, z, z, 1, 8, 8, params, 5, 32, 128, 8, z, z, z, 1, z, z, 7, z, z, z))
    invalid(lib.ms_page_batch_host_ex(h, z, z, z, 1, 8, 8, 8, 8, params, 5, 32, 128, 8, z, z, z, 1, z, z, 3, z, z))
    invalid(lib.ms_page_batch_ragged_host_ex(h, z, z, z, z, 1, 8, 8, params, 5, 32, 128, 8, z, z, z, 1, z, z, 3, z, z))
    for bad in (torch.float64, torch.int16, torch.uint8, "float16"):
        with pytest.raises(ValueError):
            mb.batch_dtype_code(bad)
    with pytest.raises(ValueError):
        mb.TRBA(model=None, batch_dtype=torch.float64)
    with pytest.raises(ValueError):
        mb.PageBatch(device=0, batch_dtype=torch.int32)


# ---- the classes --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dt", DTYPES)
def test_trba_preprocess(mb, torch, dt):
    dtype = getattr(torch, dt)
    rng = np.random.default_rng(2)
    crops = [rng.integers(0, 256, (int(h), int(w), 3), dtype=np.uint8)
             for h, w in [(20, 60), (64, 256), (70, 300), (10, 10), (33, 500), (5, 7), (128, 64), (44, 130)]]
    for ih, iw in ((32, 128), (64, 256)):
        ref = mb.TRBA(model=None, img_h=ih, img_w=iw).preprocess(crops)
        got = mb.TRBA(model=None, img_h=ih, img_w=iw, batch_dtype=dtype).preprocess(crops)
        assert_cast(got, ref, dtype)
    assert mb.TRBA(model=None, batch_dtype=dtype).preprocess([]).dtype == dtype


class Recorder:
    """a recogniser network: records the dtype and the rows it is given, names each row by its position"""

    def __init__(self):
        self.dtypes, self.rows = [], []

    def __call__(self, batch):
        self.dtypes.append(batch.dtype)
        start = sum(len(r) for r in self.rows)
        self.rows.append(batch.clone())
        return [(f"w{start + i}", 0.5) for i in range(len(batch))]


def _det(mb, torch, target, score, geo):
    class Net:
        def __call__(self, x):
            return {"score": torch.from_numpy(score)[None, None].cuda(), "geometry": torch.from_numpy(geo)[None].cuda()}

    return mb.EAST(model=Net(), target_size=target)


@pytest.mark.parametrize("dt", DTYPES)
def test_pipeline_routes_feed_the_16_bit_batch(mb, torch, dt):
    dtype = getattr(torch, dt)
    target = 512
    score, geo, _ = synthdata.make_maps(5, target, 60)
    img = synthdata.make_page_image(5, 700)[:600, :700].copy()

    def predict(batch_dtype, route, **kw):
        rec_net = Recorder()
        rec = mb.TRBA(model=rec_net, img_h=32, img_w=128, batch_dtype=batch_dtype)
        det = _det(mb, torch, target, score, geo)
        if route == "fused":
            pipe = mb.Pipeline(detector=det, recognizer=rec)
        else:  # the same words from a detector that is not this package's EAST
            words = [w for b in mb.pipeline._page_of(det.predict(img)).blocks for w in b.words]

            class Fixed:
                def predict(self, image, vis=False, profile=False):
                    return {"page": mb.Page(blocks=[mb.Block(words=[w.model_copy() for w in words])])}

            pipe = mb.Pipeline(detector=Fixed(), recognizer=rec, **kw)
        page = pipe.predict(img)
        assert pipe.last_route == route
        texts = [(tuple(map(tuple, w.polygon)), w.text) for b in page.blocks for w in b.words]
        return texts, rec_net

    for route, kw in (("fused", {}), ("device_crops", {}), ("rotated_crops", {"rotated_crops": True})):
        ref_texts, ref_net = predict(torch.float32, route, **kw)
        texts, net = predict(dtype, route, **kw)
        assert texts == ref_texts and any(t for _, t in texts)
        assert set(net.dtypes) == {dtype} and set(ref_net.dtypes) == {torch.float32}
        assert_cast(torch.cat(net.rows), torch.cat(ref_net.rows), dtype)

    # a foreign recogniser still gets uint8 slices
    class Foreign:
        def predict(self, images):
            self.images = images
            return [{"text": "p", "confidence": 1.0} for _ in images]

    rec = Foreign()
    det = _det(mb, torch, target, score, geo)
    mb.Pipeline(detector=det, recognizer=rec).predict(img)
    assert rec.images and all(im.dtype == np.uint8 for im in rec.images)
