"""Batched detector input (ms_detector_input_batch, EAST.upload_batch / network_inputs) and Pipeline.process_batch on the
fused route: every page bit for bit what the one-page calls give, in float32 and in 16 bits."""
import ctypes as C
import zlib

import numpy as np
import pytest

import synthdata

pytestmark = pytest.mark.gpu


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


def stream_of(torch):
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def cv2_input(img, th, tw):
    """infer.py:301-305: cv2.resize(img, (tw, th)) -> ToTensor -> Normalize(0.5, 0.5), (3, th, tw) float32"""
    import cv2
    import torch

    tt = torch.from_numpy(cv2.resize(img, (tw, th))).permute(2, 0, 1).float().div(255.0)
    return ((tt - 0.5) / 0.5).numpy()


# shrinking, enlarging, exactly 2x, same size (as the first target), a long thin page, one page placed at an odd address
PAGE_SHAPES = [(333, 517), (100, 180), (512, 512), (256, 256), (64, 2000), (1031, 777), (700, 900), (200, 300), (57, 61)]
UNALIGNED = 6  # index of the page whose base address is not 16-byte aligned
# square; non-square with a width that is a multiple of 4 but not of 8; a width that is not a multiple of 4
TARGETS = [(256, 256), (200, 300), (190, 250)]


@pytest.fixture(scope="module")
def ragged(torch):
    rng = np.random.default_rng(21)
    imgs = [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in PAGE_SHAPES]
    keep, ptrs = [], []
    for i, img in enumerate(imgs):
        off = 3 if i == UNALIGNED else 0
        buf = torch.zeros(img.nbytes + off, dtype=torch.uint8, device="cuda")
        buf[off:].copy_(torch.from_numpy(img.reshape(-1)))
        keep.append(buf)
        ptrs.append(buf.data_ptr() + off)
    assert ptrs[UNALIGNED] % 16 != 0
    d_ptrs = torch.tensor(ptrs, dtype=torch.int64, device="cuda")
    d_hw = torch.tensor([list(s) for s in PAGE_SHAPES], dtype=torch.int32, device="cuda")
    return imgs, keep, ptrs, d_ptrs, d_hw


def batch_call(mb, torch, ctx, d_ptrs, d_hw, n, th, tw, dtype, offset=0):
    buf = torch.full((n * 3 * th * tw + offset,), 7.0, dtype=dtype, device="cuda")
    out = buf[offset:].view(n, 3, th, tw)
    rc = ctx.lib.ms_detector_input_batch(ctx.handle, d_ptrs.data_ptr(), d_hw.data_ptr(), n, th, tw, out.data_ptr(),
                                         mb.batch_dtype_code(dtype), stream_of(torch))
    assert rc == 0, mb._cabi.last_error()
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("th,tw", TARGETS)
def test_batch_input_matches_single_pages_and_cv2(mb, torch, ctx, ragged, th, tw):
    imgs, _, ptrs, d_ptrs, d_hw = ragged
    out = batch_call(mb, torch, ctx, d_ptrs, d_hw, len(imgs), th, tw, torch.float32)
    single = torch.empty((3, th, tw), dtype=torch.float32, device="cuda")
    for i, img in enumerate(imgs):
        h, w = img.shape[:2]
        rc = ctx.lib.ms_detector_input(ctx.handle, ptrs[i], h, w, th, tw, single.data_ptr(), None, stream_of(torch))
        assert rc == 0, mb._cabi.last_error()
        got = out[i].cpu().numpy()
        np.testing.assert_array_equal(got, single.cpu().numpy(), err_msg=f"page {i} {(h, w)} -> {(th, tw)}")
        np.testing.assert_array_equal(got, cv2_input(img, th, tw), err_msg=f"page {i} {(h, w)} -> {(th, tw)}")


def test_batch_input_empty_page_is_zeros(mb, torch, ctx, ragged):
    """page sizes are device data: a page of zero height or width is not read and its input is all zeros"""
    imgs, _, ptrs, _, _ = ragged
    d_ptrs = torch.tensor([ptrs[0], 0, ptrs[1]], dtype=torch.int64, device="cuda")
    d_hw = torch.tensor([list(imgs[0].shape[:2]), [0, 40], [imgs[1].shape[0], -3]], dtype=torch.int32, device="cuda")
    out = batch_call(mb, torch, ctx, d_ptrs, d_hw, 3, 64, 96, torch.float32)
    np.testing.assert_array_equal(out[0].cpu().numpy(), cv2_input(imgs[0], 64, 96))
    assert not out[1:].any().item()


@pytest.mark.parametrize("dtype", ["float16", "bfloat16"])
@pytest.mark.parametrize("th,tw", TARGETS)
def test_batch_input_16bit_is_f32_cast(mb, torch, ctx, ragged, th, tw, dtype):
    _, _, _, d_ptrs, d_hw = ragged
    dt = getattr(torch, dtype)
    ref = batch_call(mb, torch, ctx, d_ptrs, d_hw, len(PAGE_SHAPES), th, tw, torch.float32)
    for offset in (0, 1):  # a 16-byte-aligned output and one that is not (scalar stores)
        got = batch_call(mb, torch, ctx, d_ptrs, d_hw, len(PAGE_SHAPES), th, tw, dt, offset=offset)
        assert torch.equal(got.view(torch.int16), ref.to(dt).view(torch.int16))


def test_batch_input_invalid_arguments(mb, torch, ctx, ragged):
    _, _, _, d_ptrs, d_hw = ragged
    out = torch.empty((2, 3, 32, 32), dtype=torch.float32, device="cuda")
    lib, h, s = ctx.lib, ctx.handle, stream_of(torch)
    P, O, HW = d_ptrs.data_ptr(), out.data_ptr(), d_hw.data_ptr()
    bad = [(P, HW, 2, 32, 32, O, 7), (P, HW, 2, 32, 32, O, -1), (None, HW, 2, 32, 32, O, 0), (P, None, 2, 32, 32, O, 0),
           (P, HW, 2, 32, 32, None, 0), (P, HW, 0, 32, 32, O, 0), (P, HW, -2, 32, 32, O, 0), (P, HW, 2, 0, 32, O, 0),
           (P, HW, 2, 32, -5, O, 0)]
    for args in bad:
        assert lib.ms_detector_input_batch(h, *args, s) == mb._cabi.MS_ERR_INVALID, args
    assert lib.ms_detector_input_batch(None, P, HW, 2, 32, 32, O, 0, s) == mb._cabi.MS_ERR_INVALID


# ---- Pipeline.process_batch ------------------------------------------------------------------------------------------
T = 512


class StubEAST:
    """Detector network: each input row gets its own seeded maps, keyed by the signs of that row's values (the same
    for a row in a batch, alone, or cast to 16 bits); a blank page (a constant row) gets no words.  Maps are rounded to
    bfloat16 values, so the float32 and the bfloat16 routes see the same maps."""

    def __init__(self, torch, out_dtype):
        self.torch, self.out_dtype, self.inputs, self._maps = torch, out_dtype, [], {}

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
        self.inputs.append(x.clone())
        maps = [self._row_maps(x[i]) for i in range(x.shape[0])]
        score = torch.from_numpy(np.stack([m[0] for m in maps]))[:, None].cuda().to(torch.bfloat16)
        geo = torch.from_numpy(np.stack([m[1] for m in maps])).cuda().to(torch.bfloat16)
        return {"score": score.to(self.out_dtype), "geometry": geo.to(self.out_dtype)}


class StubTRBA:
    """Recogniser network: text and confidence from each row's own contents; records every batch it is given."""

    def __init__(self):
        self.batches = []

    def __call__(self, batch):
        self.batches.append(batch.clone())
        rows = batch.float().cpu().numpy()
        return [(f"t{zlib.crc32(r.tobytes()):08x}", float(np.float32(r.mean() * 0.25 + 0.5))) for r in rows]


def page_images():
    imgs = [synthdata.make_page_image(40 + i, 1100)[:h, :w].copy()
            for i, (h, w) in enumerate([(600, 700), (900, 640), (512, 512), (1000, 1100), (333, 517)])]
    imgs.insert(2, np.full((480, 360, 3), 255, np.uint8))  # a blank page: no words
    return imgs


def make_pipe(mb, torch, input_dtype=None, batch_size=32):
    net = StubEAST(torch, torch.float32 if input_dtype is None else input_dtype)
    det = mb.EAST(model=net, target_size=T, input_dtype=input_dtype)
    rec_net = StubTRBA()
    rec = mb.TRBA(model=rec_net, img_h=32, img_w=128, batch_size=batch_size)
    return mb.Pipeline(detector=det, recognizer=rec), net, rec_net


def page_fields(page):
    return [[(w.polygon, w.detection_confidence, w.text, w.recognition_confidence) for w in b.words]
            for b in page.blocks]


def test_process_batch_equals_predict_loop(mb, torch):
    imgs = page_images()
    pipe, net, rec_net = make_pipe(mb, torch, batch_size=24)
    want = [pipe.predict(img) for img in imgs]
    assert pipe.last_route == "fused"
    single_inputs = torch.cat(net.inputs)
    single_rows = torch.cat(rec_net.batches)
    n_single_calls = len(rec_net.batches)
    net.inputs.clear()
    rec_net.batches.clear()
    uploads = []
    det = pipe.detector
    orig = det.upload_batch
    det.upload = None  # the batched route never uploads page by page
    det.upload_batch = lambda images: (uploads.append(len(images)), orig(images))[1]
    got = pipe.process_batch(imgs, max_pages=4)
    assert pipe.last_route == "fused_batch"
    assert [page_fields(p) for p in got] == [page_fields(p) for p in want]
    assert sum(len(b.words) for b in got[2].blocks) == 0 and sum(len(b.words) for b in got[0].blocks) > 0
    assert uploads == [4, 2]  # one upload per page
    # one network call per chunk, on the stacked single-page inputs
    assert [tuple(x.shape) for x in net.inputs] == [(4, 3, T, T), (2, 3, T, T)]
    assert torch.equal(torch.cat(net.inputs), single_inputs)
    # recogniser chunks of at most batch_size rows that span pages, rows equal to predict's crops
    assert all(len(b) <= 24 for b in rec_net.batches) and len(rec_net.batches) <= n_single_calls
    assert torch.equal(torch.cat(rec_net.batches), single_rows)
    # a repeated call (same shapes: same device buffers, the page batch replays its graph) gives the same pages
    views = [v.data_ptr() for v in det.upload_batch(imgs[:4])]
    again = pipe.process_batch(imgs, max_pages=4)
    assert [v.data_ptr() for v in det.upload_batch(imgs[:4])] == views
    assert [page_fields(p) for p in again] == [page_fields(p) for p in want]
    # vis=True keeps returning Pages only
    assert all(isinstance(p, mb.Page) for p in pipe.process_batch(imgs[:2], vis=True))


def test_process_batch_bfloat16_detector_input(mb, torch):
    imgs = page_images()[:4]
    ref_pipe, ref_net, _ = make_pipe(mb, torch)
    want = ref_pipe.process_batch(imgs)
    pipe, net, _ = make_pipe(mb, torch, input_dtype=torch.bfloat16)
    got = pipe.process_batch(imgs)
    assert pipe.last_route == "fused_batch"
    assert net.inputs[0].dtype == torch.bfloat16
    assert torch.equal(net.inputs[0].view(torch.int16), ref_net.inputs[0].to(torch.bfloat16).view(torch.int16))
    assert [page_fields(p) for p in got] == [page_fields(p) for p in want]
    # the single-page route takes the same dtype
    net.inputs.clear()
    assert page_fields(pipe.predict(imgs[0])) == page_fields(want[0])
    assert net.inputs[0].dtype == torch.bfloat16 and tuple(net.inputs[0].shape) == (1, 3, T, T)


def test_process_batch_foreign_recogniser_keeps_the_loop(mb, torch):
    imgs = page_images()[:2]
    net = StubEAST(torch, torch.float32)
    det = mb.EAST(model=net, target_size=T)
    seen = []

    class Foreign:
        def predict(self, crops):
            seen.append(len(crops))
            return [{"text": "x", "confidence": 0.5} for _ in crops]

    pipe = mb.Pipeline(detector=det, recognizer=Foreign())
    pages = pipe.process_batch(imgs)
    assert pipe.last_route == "host_crops" and len(pages) == 2 and len(seen) == 2
    assert all(tuple(x.shape) == (1, 3, T, T) for x in net.inputs)


def test_detector_input_u8_only(mb, torch, ctx, ragged):
    """ms_detector_input with only the u8 output (out_f32 = NULL) writes the same resized image as with both outputs"""
    imgs, _, ptrs, _, _ = ragged
    for i in (0, 1, 3, UNALIGNED):
        h, w = imgs[i].shape[:2]
        both_f = torch.empty((3, 200, 300), dtype=torch.float32, device="cuda")
        both_u = torch.zeros((200, 300, 3), dtype=torch.uint8, device="cuda")
        only_u = torch.zeros((200, 300, 3), dtype=torch.uint8, device="cuda")
        for f, u in ((both_f.data_ptr(), both_u), (None, only_u)):
            rc = ctx.lib.ms_detector_input(ctx.handle, ptrs[i], h, w, 200, 300, f, u.data_ptr(), stream_of(torch))
            assert rc == 0, mb._cabi.last_error()
        torch.cuda.synchronize()
        assert torch.equal(only_u, both_u)
        import cv2

        np.testing.assert_array_equal(only_u.cpu().numpy(), cv2.resize(imgs[i], (300, 200)))


def test_process_batch_crop_buffer_is_bounded(mb, torch, monkeypatch):
    """The batched route's crop buffer holds what a chunk needs, not cap_boxes per page: it starts small, grows to a
    power of two when a chunk needs more (and the chunk is run again), and at most two chunk sizes keep buffers."""
    import manuscript_b200.pipeline as pl

    monkeypatch.setattr(pl, "_BATCH_CROPS_CAP0", 8)
    imgs = page_images()
    pipe, _, _ = make_pipe(mb, torch, batch_size=24)
    want = [page_fields(pipe.predict(img)) for img in imgs]
    assert [page_fields(p) for p in pipe.process_batch(imgs, max_pages=4)] == want
    runner = pipe._fused_runner(batch=True)
    cap = runner.crops_cap
    assert cap > 8 and cap & (cap - 1) == 0 and cap < 4 * pipe.detector.cap_boxes
    for n in (1, 2, 3, 5, 6, 4):
        assert [page_fields(p) for p in pipe.process_batch(imgs[:n], max_pages=4)] == want[:n]
        assert len(runner._bufs) <= 2
        assert all(b["batch"].shape[0] == runner.crops_cap for b in runner._bufs.values())


def test_process_batch_page_ordered_on_the_host(mb, torch, monkeypatch):
    """A page of a chunk flagged MS_FLAG_ORDER_OVERFLOW is finished on the host (reading order, its own crops), the
    other pages' rows are taken out of the crop batch; the Pages still equal the per-image loop's."""
    from manuscript_b200.batch import PageBatchResult

    imgs = page_images()
    pipe, _, rec_net = make_pipe(mb, torch, batch_size=24)
    want = [page_fields(pipe.predict(img)) for img in imgs]
    orig = PageBatchResult.order_overflow_pages
    monkeypatch.setattr(PageBatchResult, "order_overflow_pages",
                        lambda self: np.array([1]) if len(self.flags) > 1 else orig(self))
    rec_net.batches.clear()
    got = pipe.process_batch(imgs, max_pages=4)
    assert pipe.last_route == "fused_batch"
    assert [page_fields(p) for p in got] == want
    assert all(len(b) <= 24 for b in rec_net.batches)
