"""Detector maps in float16, bfloat16 and at any strides (ms_maps): every output of the decode, the four page-batch
entry points and the fused Pipeline routes equals, bit for bit, that of the same call on the float32 dense copies of
the maps (.float().contiguous()), with no copy of the maps made."""
import ctypes as C
import zlib

import numpy as np
import pytest

import synthdata

pytestmark = pytest.mark.gpu

DTYPES = ["float32", "float16", "bfloat16"]
# NCHW; channels_last geometry; the score / geometry channels of a fused (P, 9, H, W) head, NCHW and channels_last
LAYOUTS = ["nchw", "channels_last", "head", "head_channels_last"]


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


def as_layout(torch, score, geo, layout):
    """score (P, H, W), geo (P, 8, H, W) CUDA tensors -> the same values in `layout`"""
    if layout == "nchw":
        return score.contiguous(), geo.contiguous()
    if layout == "channels_last":
        return score.contiguous(), geo.contiguous(memory_format=torch.channels_last)
    head = torch.cat([score[:, None], geo], 1)
    if layout == "head_channels_last":
        head = head.contiguous(memory_format=torch.channels_last)
    return head[:, 0], head[:, 1:]


def dense_f32(s, g):
    return s.float().contiguous(), g.float().contiguous()


def bits(t):
    """a tensor's bits as numpy integers (NaN payloads compared too)"""
    import torch

    t = t.contiguous()
    return (t.view(torch.int32) if t.element_size() == 4 else t.view(torch.int16)).cpu().numpy()


def neighbours16(torch, dt, v):
    """v rounded to dt and its two neighbours in dt, as float32 values"""
    x = torch.tensor([v], dtype=torch.float32).to(dt).view(torch.int16)
    return torch.cat([x - 1, x, x + 1]).view(dt).float().tolist()


def special_maps(torch, dt, P, H, W, thr, seed):
    """Seeded word maps (P, H, W) / (P, 8, H, W) in dt, with NaNs (several payloads), infinities, subnormals and scores
    at the dt neighbours of thr scattered over both maps"""
    rng = np.random.default_rng(seed)
    M = max(H, W)
    score, geo, _ = synthdata.make_batch(list(range(seed, seed + P)), 4 * M, 12, with_images=False)
    s = torch.from_numpy(np.ascontiguousarray(score[:, :H, :W])).cuda().to(dt)
    g = torch.from_numpy(np.ascontiguousarray(geo[:, :, :H, :W])).cuda().to(dt)
    if dt == torch.float32:
        nans = [0x7F800001, 0x7FC00000, 0xFFC12345, 0x7FBFFFFF]
        subn = [1e-40, -3e-39, 1e-45]
        near = [float(np.nextafter(np.float32(thr), np.float32(d))) for d in (-1, 1)] + [float(np.float32(thr))]
        iview = torch.int32
    else:
        nans = [0x7C01, 0x7E00, 0xFE55, 0x7DFF] if dt == torch.float16 else [0x7F81, 0x7FC0, 0xFFC1, 0x7FFF]
        subn = [1e-6, -3e-7, 6e-8] if dt == torch.float16 else [1e-39, -5e-40, 1e-40]
        near = neighbours16(torch, dt, thr)
        iview = torch.int16

    def scatter(t, values, n, as_bits):
        flat = t.view(-1)
        idx = torch.from_numpy(rng.integers(0, flat.numel(), n)).cuda()
        vals = torch.tensor([values[i % len(values)] for i in range(n)])
        if as_bits:
            vals = vals.to(torch.int64)
            vals = torch.where(vals >= 2 ** (8 * t.element_size() - 1), vals - 2 ** (8 * t.element_size()), vals)
            flat.view(iview)[idx] = vals.to(iview).cuda()
        else:
            flat[idx] = vals.to(t.dtype).cuda()

    n = H * W * P
    for t in (s, g):
        scatter(t, nans, max(4, n // 200), True)
        scatter(t, [float("inf"), float("-inf")], max(2, n // 300), False)
        scatter(t, subn, max(3, n // 200), False)
    scatter(s, near, max(3, n // 50), False)
    return s, g


def decode(mb, ctx, torch, s, g, q, thr, cap, fill=-7.0):
    P, H, W = s.shape
    out = torch.full((P * cap, 9), fill, dtype=torch.float32, device="cuda")
    counts = torch.full((P,), -1, dtype=torch.int32, device="cuda")
    flags = torch.zeros((P,), dtype=torch.int32, device="cuda")
    maps = mb._cabi.maps_descriptor(s, g)
    rc = ctx.lib.ms_decode_quads_maps(ctx.handle, C.byref(maps), P, H, W, thr, 4.0, q, out.data_ptr(), cap,
                                      counts.data_ptr(), flags.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, mb._cabi.last_error()
    torch.cuda.synchronize()
    return bits(out), counts.cpu().numpy(), flags.cpu().numpy()


@pytest.mark.parametrize("W", [64, 61])
@pytest.mark.parametrize("q", [1, 2, 3])
@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("dtype", DTYPES)
def test_decode_equals_dense_f32(mb, ctx, torch, dtype, layout, q, W):
    dt = getattr(torch, dtype)
    thr = 0.6
    s0, g0 = special_maps(torch, dt, 3, 61, W, thr, seed=7 + q)
    s0[1, -1, :] = 0.9  # the last row, a partial cell for q > 1: its centre is outside the map -> MS_FLAG_INDEX_ERROR
    s, g = as_layout(torch, s0, g0, layout)
    assert s.dtype == dt and g.dtype == dt
    cap = -(-61 // q) * -(-W // q)
    for c in (cap, 25):  # every cell fits; MS_FLAG_CAND_OVERFLOW
        got = decode(mb, ctx, torch, s, g, q, thr, c)
        want = decode(mb, ctx, torch, *dense_f32(s, g), q, thr, c)
        for a, b in zip(got, want):
            np.testing.assert_array_equal(a, b)
        assert want[1].min() > 0
        if c == 25:
            assert (want[2] & mb._cabi.MS_FLAG_CAND_OVERFLOW).any()
    if q > 1:
        assert want[2][1] & mb._cabi.MS_FLAG_INDEX_ERROR


def page_batch_inputs(torch, P=16, page=512, seed=300):
    score, geo, imgs = synthdata.make_batch(list(range(seed, seed + P)), page, 50)
    return (torch.from_numpy(score).cuda(), torch.from_numpy(geo).cuda(), torch.from_numpy(imgs).cuda())


def snapshot(torch, r):
    torch.cuda.synchronize()
    counts = r.box_counts.cpu().numpy().copy()
    boxes = r.boxes.cpu().numpy()
    n = int(r.n_crops.cpu()[0])
    out = [counts, r.flags.cpu().numpy().copy(), r.crops[:n].cpu().numpy().copy()]
    out += [bits(r.boxes[p, : min(int(counts[p]), boxes.shape[1])]) for p in range(len(counts))]
    if r.batch is not None:
        out.append(bits(r.batch[:n]))
    return out


def assert_same(a, b):
    assert len(a) == len(b)
    for x, y in zip(a, b):
        np.testing.assert_array_equal(x, y)


@pytest.mark.parametrize("crops", ["rects", "quads"])
@pytest.mark.parametrize("ragged", [False, True])
@pytest.mark.parametrize("sort", [0, 1])
@pytest.mark.parametrize("layout", ["nchw", "channels_last", "head_channels_last"])
@pytest.mark.parametrize("dtype", DTYPES)
def test_page_batch_entries_equal_dense_f32(mb, torch, dtype, layout, sort, ragged, crops):
    """ms_page_batch_maps / _ragged_maps / _quads_maps / _ragged_quads_maps on 16 pages (two concurrent front halves)"""
    dt = getattr(torch, dtype)
    score, geo, imgs = page_batch_inputs(torch)
    s, g = as_layout(torch, score.to(dt), geo.to(dt), layout)
    batch_dtype = torch.bfloat16 if sort else torch.float32
    runner = mb.PageBatch(device=0, params=mb.EastParams.default(target_size=512, sort_reading_order=sort),
                          cap_boxes=512, crops=crops, batch_dtype=batch_dtype)
    pages = [imgs[i] for i in range(len(imgs))] if ragged else imgs
    run = (lambda a, b: runner.run_ragged(a, b, pages)) if ragged else (lambda a, b: runner.run(a, b, pages))
    got = snapshot(torch, run(s, g))
    want = snapshot(torch, run(*dense_f32(s, g)))
    assert_same(got, want)
    assert len(want[2]) > 0 and not want[1].any()


def test_maps_call_replays_a_graph_and_the_dtype_is_part_of_the_call(mb, torch):
    """A repeated call with the same bfloat16 map tensors replays the graph of its second occurrence (same results, same
    launch accounting, new data in the same tensors honoured); the same addresses and strides read as float16 are
    another call, with float16 results."""
    score, geo, imgs = page_batch_inputs(torch, seed=400)
    s, g = as_layout(torch, score.to(torch.bfloat16), geo.to(torch.bfloat16), "channels_last")
    runner = mb.PageBatch(device=0, params=mb.EastParams.default(target_size=512), cap_boxes=512)
    ref = mb.PageBatch(device=0, params=mb.EastParams.default(target_size=512), cap_boxes=512)
    l0 = runner.ctx.launches
    first = snapshot(torch, runner.run(s, g, imgs))
    per_call = runner.ctx.launches - l0
    second = snapshot(torch, runner.run(s, g, imgs))
    third = snapshot(torch, runner.run(s, g, imgs))
    assert runner.ctx.launches - l0 == 3 * per_call and per_call > 20
    assert_same(first, second)
    assert_same(first, third)
    assert_same(first, snapshot(torch, ref.run(*dense_f32(s, g), imgs)))
    score2, geo2, _ = page_batch_inputs(torch, seed=500)
    s.copy_(score2.to(torch.bfloat16)), g.copy_(geo2.to(torch.bfloat16))
    fourth = snapshot(torch, runner.run(s, g, imgs))
    assert not all(np.array_equal(x, y) for x, y in zip(first[3:], fourth[3:]))
    assert_same(fourth, snapshot(torch, ref.run(*dense_f32(s, g), imgs)))
    # only the dtype changes: float16 results, not a replay of the bfloat16 graph
    sh, gh = s.view(torch.float16), g.view(torch.float16)
    assert sh.data_ptr() == s.data_ptr() and gh.stride() == g.stride()
    for _ in range(3):
        assert_same(snapshot(torch, runner.run(sh, gh, imgs)), snapshot(torch, ref.run(*dense_f32(sh, gh), imgs)))
    assert_same(snapshot(torch, runner.run(s, g, imgs)), fourth)


def test_dense_f32_descriptor_is_the_ex_call(mb, torch, ctx):
    """ms_page_batch_ex and ms_page_batch_maps on the same dense float32 maps: the same results, the u8 canvas included"""
    score, geo, imgs = page_batch_inputs(torch, P=4, seed=600)
    P, H, W = score.shape
    p = mb.EastParams.default(target_size=512)
    cap, crops_cap, oh, ow = 512, 2048, 32, 128
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(use_maps):
        boxes = torch.full((P, cap, 9), -1.0, device="cuda")
        counts = torch.zeros(P, dtype=torch.int32, device="cuda")
        crops = torch.zeros((crops_cap, 5), dtype=torch.int32, device="cuda")
        n = torch.zeros(1, dtype=torch.int32, device="cuda")
        batch = torch.zeros((crops_cap, 3, oh, ow), dtype=torch.float16, device="cuda")
        canvas = torch.zeros((crops_cap, oh, ow, 3), dtype=torch.uint8, device="cuda")
        flags = torch.zeros(P, dtype=torch.int32, device="cuda")
        tail = (imgs.data_ptr(), P, H, W, 512, 512, C.byref(p), 5, oh, ow, cap, boxes.data_ptr(), counts.data_ptr(),
                crops.data_ptr(), crops_cap, n.data_ptr(), batch.data_ptr(), mb._cabi.MS_DTYPE_F16, canvas.data_ptr(),
                flags.data_ptr(), st)
        if use_maps:
            maps = mb._cabi.maps_descriptor(score, geo)
            rc = ctx.lib.ms_page_batch_maps(ctx.handle, C.byref(maps), *tail)
        else:
            rc = ctx.lib.ms_page_batch_ex(ctx.handle, score.data_ptr(), geo.data_ptr(), *tail)
        assert rc == 0, mb._cabi.last_error()
        torch.cuda.synchronize()
        return [bits(boxes), counts.cpu().numpy(), bits(crops), n.cpu().numpy(), bits(batch), canvas.cpu().numpy(),
                flags.cpu().numpy()]

    want = call(False)
    assert want[3][0] > 0
    for use_maps in (True, False, True, True):
        assert_same(call(use_maps), want)


def test_invalid_descriptors(mb, torch, ctx):
    score, geo, imgs = page_batch_inputs(torch, P=2, seed=700)
    P, H, W = score.shape
    p = mb.EastParams.default(target_size=512)
    boxes = torch.empty((P, 64, 9), device="cuda")
    counts, n_crops, flags = (torch.zeros(n, dtype=torch.int32, device="cuda") for n in (P, 1, P))
    crops = torch.zeros((64, 5), dtype=torch.int32, device="cuda")
    ptrs = torch.tensor([imgs[0].data_ptr(), imgs[1].data_ptr()], dtype=torch.int64, device="cuda")
    hw = torch.tensor([[512, 512]] * 2, dtype=torch.int32, device="cuda")
    B, I, CR, PT, HW = boxes.data_ptr(), imgs.data_ptr(), crops.data_ptr(), ptrs.data_ptr(), hw.data_ptr()
    N, NC, F = counts.data_ptr(), n_crops.data_ptr(), flags.data_ptr()
    lib, h = ctx.lib, ctx.handle
    calls = {
        "ms_decode_quads_maps": lambda m: lib.ms_decode_quads_maps(h, m, P, H, W, 0.6, 4.0, 2, B, 64, N, F, None),
        "ms_page_batch_maps": lambda m: lib.ms_page_batch_maps(h, m, I, P, H, W, 512, 512, C.byref(p), 5, 32, 128, 64,
                                                               B, N, CR, 64, NC, None, 0, None, F, None),
        "ms_page_batch_ragged_maps": lambda m: lib.ms_page_batch_ragged_maps(h, m, PT, HW, P, H, W, C.byref(p), 5, 32,
                                                                             128, 64, B, N, CR, 64, NC, None, 0, None,
                                                                             F, None),
        "ms_page_batch_quads_maps": lambda m: lib.ms_page_batch_quads_maps(h, m, I, P, H, W, 512, 512, C.byref(p), 5,
                                                                           0, 0, 32, 128, 64, B, N, CR, 64, NC, None, 0,
                                                                           None, F, None),
        "ms_page_batch_ragged_quads_maps": lambda m: lib.ms_page_batch_ragged_quads_maps(
            h, m, PT, HW, P, H, W, C.byref(p), 5, 0, 0, 32, 128, 64, B, N, CR, 64, NC, None, 0, None, F, None),
    }
    for name, call in calls.items():
        good = mb._cabi.maps_descriptor(score, geo)
        assert call(C.byref(good)) == 0, (name, mb._cabi.last_error())
        torch.cuda.synchronize()
        assert call(None) == mb._cabi.MS_ERR_INVALID, name
        for field, value in [("dtype", 3), ("dtype", -1), ("score", None), ("geo", None)]:
            m = mb._cabi.maps_descriptor(score, geo)
            setattr(m, field, value)
            assert call(C.byref(m)) == mb._cabi.MS_ERR_INVALID, (name, field, value)
        for arr, i in [("score_strides", 0), ("score_strides", 2), ("geo_strides", 1), ("geo_strides", 3)]:
            m = mb._cabi.maps_descriptor(score, geo)
            getattr(m, arr)[i] = -1
            assert call(C.byref(m)) == mb._cabi.MS_ERR_INVALID, (name, arr, i)


def test_boxes_from_maps_takes_16bit_maps_in_place(mb, torch):
    score, geo, _ = synthdata.make_batch([800], 512, 60, with_images=False)
    det = mb.EAST(model=None, target_size=512)
    want = det.boxes_from_maps(score[0], geo[0], (512, 512))
    assert len(want) > 0
    for dt in (torch.float16, torch.bfloat16):
        s16 = torch.from_numpy(score[0]).cuda().to(dt)
        g16 = torch.from_numpy(geo[0]).cuda().to(dt)[None].contiguous(memory_format=torch.channels_last)[0]
        got = det.boxes_from_maps(s16, g16, (512, 512))
        np.testing.assert_array_equal(got, det.boxes_from_maps(s16.float().cpu().numpy(), g16.float().cpu().numpy(),
                                                               (512, 512)))


# ---- Pipeline: the network's own maps go to the page batch ----------------------------------------------------------
T = 512


class StubEAST:
    """Detector network: each input row gets its own seeded maps, keyed by the signs of that row's values; a blank
    page gets no words.  Maps are bfloat16 values, returned in out_dtype, the geometry optionally channels_last."""

    def __init__(self, torch, out_dtype, channels_last=False):
        self.torch, self.out_dtype, self.channels_last, self._maps = torch, out_dtype, channels_last, {}
        self.outputs = []

    def _row_maps(self, row):
        if row.min().item() == row.max().item():
            return np.zeros((T // 4, T // 4), np.float32), np.zeros((8, T // 4, T // 4), np.float32)
        key = zlib.crc32((row > 0).cpu().numpy().tobytes())
        if key not in self._maps:
            score, geo, _ = synthdata.make_maps(key % 9973, T, 60)
            self._maps[key] = score, geo
        return self._maps[key]

    def __call__(self, x):
        torch = self.torch
        maps = [self._row_maps(x[i]) for i in range(x.shape[0])]
        score = torch.from_numpy(np.stack([m[0] for m in maps]))[:, None].cuda().to(torch.bfloat16).to(self.out_dtype)
        geo = torch.from_numpy(np.stack([m[1] for m in maps])).cuda().to(torch.bfloat16).to(self.out_dtype)
        if self.channels_last:
            geo = geo.contiguous(memory_format=torch.channels_last)
        self.outputs.append((score, geo))
        return {"score": score, "geometry": geo}


class StubTRBA:
    def __call__(self, batch):
        rows = batch.float().cpu().numpy()
        return [(f"t{zlib.crc32(r.tobytes()):08x}", float(np.float32(r.mean() * 0.25 + 0.5))) for r in rows]


def page_images():
    imgs = [synthdata.make_page_image(60 + i, 1100)[:h, :w].copy()
            for i, (h, w) in enumerate([(600, 700), (900, 640), (512, 512), (1000, 1100)])]
    imgs.insert(2, np.full((480, 360, 3), 255, np.uint8))
    return imgs


def page_fields(page):
    return [[(w.polygon, w.detection_confidence, w.text, w.recognition_confidence) for w in b.words]
            for b in page.blocks]


@pytest.mark.parametrize("rotated", [False, True])
@pytest.mark.parametrize("channels_last", [False, True])
def test_pipeline_hands_the_networks_maps_to_the_page_batch(mb, torch, rotated, channels_last):
    imgs = page_images()

    def make(out_dtype, cl):
        net = StubEAST(torch, out_dtype, cl)
        det = mb.EAST(model=net, target_size=T, input_dtype=torch.bfloat16)
        rec = mb.TRBA(model=StubTRBA(), img_h=32, img_w=128, batch_size=16)
        return mb.Pipeline(detector=det, recognizer=rec, rotated_crops=rotated), net

    ref, _ = make(torch.float32, False)
    want_single = [page_fields(ref.predict(img)) for img in imgs[:2]]
    want_batch = [page_fields(p) for p in ref.process_batch(imgs, max_pages=3)]
    assert sum(len(w) for w in want_batch[0]) > 0

    pipe, net = make(torch.bfloat16, channels_last)
    seen = []
    for runner_batch in (False, True):
        runner = pipe._fused_runner(batch=runner_batch)
        orig = runner.run_ragged

        def spy(score, geo, pages, _orig=orig, **kw):
            if not kw.get("sync"):  # (a sync=True call runs itself again with sync=False)
                seen.append((score, geo))
            return _orig(score, geo, pages, **kw)

        runner.run_ragged = spy
    got_single = [page_fields(pipe.predict(img)) for img in imgs[:2]]
    assert pipe.last_route == ("fused_rotated" if rotated else "fused")
    got_batch = [page_fields(p) for p in pipe.process_batch(imgs, max_pages=3)]
    assert pipe.last_route == ("fused_batch_rotated" if rotated else "fused_batch")
    assert got_single == want_single and got_batch == want_batch
    assert len(seen) == len(net.outputs) == 4
    for (score, geo), (s_net, g_net) in zip(seen, net.outputs):
        assert score.dtype == geo.dtype == torch.bfloat16
        assert score.data_ptr() == s_net.data_ptr() and geo.data_ptr() == g_net.data_ptr()
        assert geo.stride()[-3:] == g_net.stride()[-3:]
    # the documented default of maps_from_device_page(s) stays float32
    pages_dev = pipe.detector.upload_batch(imgs[:2])
    s32, g32 = pipe.detector.maps_from_device_pages(pages_dev)
    assert s32.dtype == g32.dtype == torch.float32
    s1, g1 = pipe.detector.maps_from_device_page(pages_dev[0])
    assert s1.dtype == g1.dtype == torch.float32
    sn, gn = pipe.detector.maps_from_device_pages(pages_dev, dtype=None)
    assert sn.dtype == gn.dtype == torch.bfloat16
