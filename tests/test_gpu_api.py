"""The reference-facing classes (EAST / TRBA / Pipeline mirrors) on the GPU: the duck-typed contract pinned by the
reference's tests/test_pipeline_api_compatibility.py:15-238, plus parity of what flows through them."""
import os

import numpy as np
import pytest

import synthdata
from oracle import cpu

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mb():
    import manuscript_b200 as m

    return m


def three_words(mb):
    W = mb.Word
    return [W(polygon=[[10.0, 10.0], [100.0, 10.0], [100.0, 50.0], [10.0, 50.0]], detection_confidence=0.95),
            W(polygon=[[110.0, 10.0], [200.0, 10.0], [200.0, 50.0], [110.0, 50.0]], detection_confidence=0.92),
            W(polygon=[[210.0, 10.0], [300.0, 10.0], [300.0, 50.0], [210.0, 50.0]], detection_confidence=0.88)]


class DummyDetector:
    def __init__(self, mb, return_type="dict", words=None):
        self.mb, self.return_type, self.words = mb, return_type, words

    def predict(self, image, vis=False, profile=False):
        page = self.mb.Page(blocks=[self.mb.Block(words=self.words or three_words(self.mb))])
        if self.return_type == "dict":
            return {"page": page, "vis_image": None, "score_map": None, "geo_map": None}
        if self.return_type == "tuple":
            return (page, None)
        return page


class DummyRecognizer:
    def __init__(self):
        self.call_count = 0
        self.seen = None

    def predict(self, images):
        self.call_count += 1
        self.seen = images
        return [{"text": f"word{i + 1}", "confidence": 0.9 - i * 0.05} for i, _ in enumerate(images)]


@pytest.mark.parametrize("rt", ["dict", "tuple", "page"])
def test_pipeline_duck_typed_detector_and_recognizer(mb, rt):
    rec = DummyRecognizer()
    pipe = mb.Pipeline(detector=DummyDetector(mb, rt), recognizer=rec)
    img = np.random.default_rng(0).integers(0, 256, (100, 400, 3), dtype=np.uint8)
    page = pipe.predict(img, recognize_text=True, vis=False)
    assert isinstance(page, mb.Page) and len(page.blocks[0].words) == 3
    assert [w.text for w in page.blocks[0].words] == ["word1", "word2", "word3"]
    assert rec.call_count == 1 and len(rec.seen) == 3
    # the crops are the reference's slices image[y1:y2, x1:x2] in reading order (_pipeline.py:204-221)
    np.testing.assert_array_equal(rec.seen[0], img[10:50, 10:100])
    np.testing.assert_array_equal(rec.seen[2], img[10:50, 210:300])
    assert "word1 word2 word3" == pipe.get_text(page)
    assert isinstance(pipe.predict(img, recognize_text=False), mb.Page)


def test_pipeline_min_text_size_filter(mb):
    small = [mb.Word(polygon=[[10.0, 10.0], [12.0, 10.0], [12.0, 12.0], [10.0, 12.0]], detection_confidence=0.95)]
    rec = DummyRecognizer()
    pipe = mb.Pipeline(detector=DummyDetector(mb, "dict", small), recognizer=rec, min_text_size=5)
    pipe.predict(np.zeros((100, 400, 3), np.uint8))
    assert rec.call_count == 0


def test_pipeline_errors(mb):
    class NoPage:
        def predict(self, image, vis=False, profile=False):
            return {"page": None}

    with pytest.raises(RuntimeError):
        mb.Pipeline(detector=NoPage(), recognizer=DummyRecognizer()).predict(np.zeros((10, 10, 3), np.uint8))
    with pytest.raises(TypeError):
        mb.read_image(123)
    with pytest.raises(FileNotFoundError):
        mb.read_image("/nonexistent/file.png")


def test_east_predict_from_maps_golden(mb, golden_dir):
    g = np.load(os.path.join(golden_dir, "page_s2.npz"))
    seed, page, words = int(g["seed"]), int(g["page"]), int(g["words"])
    score, geo, _ = synthdata.make_maps(seed, page, words)
    det = mb.EAST(target_size=page)
    orig_hw = tuple(int(v) for v in g["orig_hw"])
    boxes = det.boxes_from_maps(score, geo, orig_hw)
    np.testing.assert_array_equal(boxes, g["aligned"])
    pg = det.predict_from_maps(score, geo, orig_hw)
    assert len(pg.blocks) == 1 and len(pg.blocks[0].words) == len(g["aligned"])
    w0 = pg.blocks[0].words[0]
    assert w0.polygon[0] == (float(g["aligned"][0, 0]), float(g["aligned"][0, 1]))
    assert w0.detection_confidence == float(g["aligned"][0, 8])
    # non-default kwargs reach the kernels
    det2 = mb.EAST(target_size=page, expand_ratio_w=0.3, expand_ratio_h=0.7, axis_aligned_output=False, iou_threshold=0.5)
    q = cpu.decode_quads_from_maps(score, geo, 0.6, 4.0, 2)
    want = cpu.east_postprocess(cpu.locality_aware_nms(q, 0.5), orig_hw, target_size=page, expand_w=0.3, expand_h=0.7,
                                axis_aligned=False)
    np.testing.assert_array_equal(det2.boxes_from_maps(score, geo, orig_hw), want)


def test_east_predict_with_a_stub_network(mb):
    """EAST.predict end to end with a stand-in network that replays synthetic maps (the real ResNet is outside
    the path): result dict keys and Page contents as the reference's (infer.py:395-400)."""
    import torch

    page, words = 512, 60
    score, geo, _ = synthdata.make_maps(5, page, words)

    class Net:
        def __call__(self, x):
            assert x.shape == (1, 3, page, page) and x.is_cuda
            return {"score": torch.from_numpy(score)[None, None].cuda(), "geometry": torch.from_numpy(geo)[None].cuda()}

    det = mb.EAST(model=Net(), target_size=page)
    img = synthdata.make_page_image(5, 700)[:600, :700]
    out = det.predict(img, return_maps=True, sort_reading_order=True)
    assert set(out) == {"page", "vis_image", "score_map", "geo_map"}
    np.testing.assert_array_equal(out["score_map"], score)
    q = cpu.decode_quads_from_maps(score, geo, 0.6, 4.0, 2)
    want = cpu.east_postprocess(cpu.locality_aware_nms(q, 0.2), (600, 700), target_size=page)
    got = sorted(tuple(np.float32(v) for pt in w.polygon for v in pt) for w in out["page"].blocks[0].words)
    assert got == sorted(tuple(r[:8]) for r in want)
    with pytest.raises(RuntimeError):
        mb.EAST(target_size=page).predict(img)


def test_trba_preprocess_matches_oracle(mb):
    rng = np.random.default_rng(2)
    crops = [rng.integers(0, 256, (int(h), int(w), 3), dtype=np.uint8)
             for h, w in [(20, 60), (64, 256), (70, 300), (10, 10), (33, 500), (5, 7), (128, 64)]]
    for ih, iw in [(64, 256), (32, 128)]:
        rec = mb.TRBA(model=lambda b: [{"text": "x", "confidence": 0.5}] * len(b), img_h=ih, img_w=iw)
        batch = rec.preprocess(crops).cpu().numpy()
        for i, c in enumerate(crops):
            _, chw = cpu.crop_resize_pad(c, np.array([0, 0, c.shape[1], c.shape[0]], np.int32), ih, iw)
            np.testing.assert_array_equal(batch[i], chw)
        res = rec.predict(crops, batch_size=3)
        assert len(res) == len(crops) and res[0] == {"text": "x", "confidence": 0.5}
    grey = rng.integers(0, 256, (20, 50), dtype=np.uint8)
    b = mb.TRBA(model=None).preprocess([grey]).cpu().numpy()
    _, chw = cpu.crop_resize_pad(np.repeat(grey[:, :, None], 3, 2), np.array([0, 0, 50, 20], np.int32), 64, 256)
    np.testing.assert_array_equal(b[0], chw)


def test_pipeline_with_b200_trba_feeds_device_batch(mb):
    seen = {}

    def model(batch):
        seen["shape"], seen["cuda"] = tuple(batch.shape), batch.is_cuda
        seen["batch"] = batch.cpu().numpy()
        return [(f"t{i}", 0.5) for i in range(len(batch))]

    rec = mb.TRBA(model=model, img_h=32, img_w=128)
    pipe = mb.Pipeline(detector=DummyDetector(mb, "dict"), recognizer=rec)
    img = np.random.default_rng(1).integers(0, 256, (100, 400, 3), dtype=np.uint8)
    page = pipe.predict(img)
    assert seen["shape"] == (3, 3, 32, 128) and seen["cuda"]
    _, chw = cpu.crop_resize_pad(img, np.array([110, 10, 200, 50], np.int32), 32, 128)
    np.testing.assert_array_equal(seen["batch"][1], chw)
    assert [w.text for w in page.blocks[0].words] == ["t0", "t1", "t2"]
    assert page.blocks[0].words[0].recognition_confidence == 0.5


def _boxes_to_polys(boxes):
    b = np.asarray(boxes, np.float32).reshape(-1, 4)
    x0, y0, x1, y1 = b[:, 0], b[:, 1], b[:, 2], b[:, 3]
    return np.stack([x0, y0, x1, y0, x1, y1, x0, y1], axis=1)


def _host_order(mb, boxes):
    """Pipeline.predict's sort + re-match (host restatement pinned to the reference goldens) as word indices."""
    keys = [tuple(int(v) for v in bx) for bx in boxes]
    first = {}
    for i, k in enumerate(keys):
        first.setdefault(k, i)
    return [first[tuple(int(v) for v in bx)] for bx in mb.sort_boxes_reading_order_with_resolutions(keys)]


def test_reading_order_device_matches_reference_goldens(mb, golden_dir):
    g = np.load(os.path.join(golden_dir, "reading_order.npz"))
    for i in range(int(g["n_cases"])):
        boxes = g[f"boxes_{i}"]
        got = mb.word_reading_order(_boxes_to_polys(boxes))
        # the golden holds the reference's sorted boxes; compare box sequences, then exact word indices vs the host mirror
        np.testing.assert_array_equal(boxes[got].reshape(-1, 4), g[f"sorted_res_{i}"], err_msg=f"case {i}")
        assert list(got) == _host_order(mb, boxes), f"case {i}"


def test_reading_order_device_on_detector_output(mb):
    """Expanded (heavily overlapping) detector boxes of a synthetic page, fractional coordinates included."""
    page, words = 1280, 500
    score, geo, _ = synthdata.make_maps(9, page, words)
    q = cpu.decode_quads_from_maps(score, geo, 0.6, 4.0, 2)
    boxes = cpu.east_postprocess(cpu.locality_aware_nms(q, 0.2), (page, page), target_size=page)
    got = mb.word_reading_order(boxes[:, :8])
    ib = []
    for b in boxes[:, :8]:
        xs, ys = np.trunc(b[0::2]).astype(np.int64), np.trunc(b[1::2]).astype(np.int64)
        ib.append((int(xs.min()), int(ys.min()), int(xs.max()), int(ys.max())))
    assert list(got) == _host_order(mb, ib)
    assert sorted(set(got.tolist())) == sorted(set(range(len(boxes)))) or len(set(ib)) < len(ib)
    # through the batched path: boxes come out in reading order and crops follow them
    import torch

    imgs = synthdata.make_page_image(9, page)[None]
    params = mb.EastParams.default(target_size=page, sort_reading_order=1)
    runner = mb.PageBatch(device=0, params=params, cap_boxes=1024)
    res = runner.run(torch.from_numpy(score[None]).cuda(), torch.from_numpy(geo[None]).cuda(), torch.from_numpy(imgs).cuda())
    torch.cuda.synchronize()
    n = int(res.box_counts.cpu()[0])
    assert n == len(boxes) and int(res.flags.cpu()[0]) == 0
    np.testing.assert_array_equal(res.boxes[0, :n].cpu().numpy(), boxes[got])
    rects, valid = cpu.word_rects(boxes[got], page, page, 5)
    nc = int(res.n_crops.cpu()[0])
    np.testing.assert_array_equal(res.crops[:nc].cpu().numpy()[:, 1:], rects[valid])


# ---- SURVEY 8f-4 (extension): rotated crops through the Pipeline and the device entry point ---------------------------
def test_pipeline_rotated_crops(mb):
    W = mb.Word
    words = [W(polygon=[[20.0, 30.0], [110.0, 18.0], [114.0, 48.0], [24.0, 60.0]], detection_confidence=0.9),
             W(polygon=[[150.0, 20.0], [153.0, 20.0], [153.0, 23.0], [150.0, 23.0]], detection_confidence=0.9),  # 3 px
             W(polygon=[[200.0, 40.0], [330.0, 60.0], [326.0, 90.0], [196.0, 70.0]], detection_confidence=0.9)]
    img = np.random.default_rng(5).integers(0, 256, (120, 400, 3), dtype=np.uint8)
    seen = {}

    def model(batch):
        seen["batch"] = batch.cpu().numpy()
        return [(f"t{i}", 0.5) for i in range(len(batch))]

    pipe = mb.Pipeline(detector=DummyDetector(mb, "dict", words), recognizer=mb.TRBA(model=model, img_h=32, img_w=128),
                       rotated_crops=True)
    page = pipe.predict(img)
    got = {tuple(w.polygon[0]): w.text for w in page.blocks[0].words}
    assert seen["batch"].shape == (2, 3, 32, 128)
    assert got[(150.0, 20.0)] is None and {got[(20.0, 30.0)], got[(200.0, 40.0)]} == {"t0", "t1"}
    first = [w for w in page.blocks[0].words if w.text == "t0"][0]
    _, chw = cpu.quad_crop_resize_pad(img, np.array(first.polygon, np.float32).reshape(-1), 32, 128)
    np.testing.assert_array_equal(seen["batch"][0], chw)

    # a foreign recogniser receives the rectified uint8 patches
    class Rec:
        def predict(self, images):
            self.images = images
            return [{"text": "p", "confidence": 1.0} for _ in images]

    rec = Rec()
    mb.Pipeline(detector=DummyDetector(mb, "dict", words), recognizer=rec, rotated_crops=True).predict(img)
    assert len(rec.images) == 2
    np.testing.assert_array_equal(rec.images[0], cpu.warp_quad(img, np.array(first.polygon, np.float32).reshape(-1)))


def test_quad_crop_device_entry(mb):
    """ms_quad_crop_resize_pad on device buffers: two pages, box rows of 9 floats (quad + score) as the detector
    stage leaves them, page_of per quad, launched on a torch stream."""
    import ctypes as C

    import torch

    rng = np.random.default_rng(9)
    pages = rng.integers(0, 256, (2, 300, 500, 3), dtype=np.uint8)
    n = 50
    rows = np.zeros((n, 9), np.float32)
    for i in range(n):
        cx, cy, ww, hh, a = rng.uniform(50, 450), rng.uniform(40, 260), rng.uniform(20, 150), rng.uniform(6, 50), \
            rng.uniform(-0.4, 0.4)
        c, s = np.cos(a), np.sin(a)
        q = np.array([[-ww / 2, -hh / 2], [ww / 2, -hh / 2], [ww / 2, hh / 2], [-ww / 2, hh / 2]]) @ np.array(
            [[c, s], [-s, c]]) + [cx, cy]
        rows[i, :8] = q.reshape(-1)
        rows[i, 8] = 0.9
    page_of = rng.integers(0, 2, n).astype(np.int32)
    page_of[3] = 7  # out of range: no patch
    d_pages, d_rows, d_po = torch.from_numpy(pages).cuda(), torch.from_numpy(rows).cuda(), torch.from_numpy(page_of).cuda()
    batch = torch.empty((n, 3, 32, 128), dtype=torch.float32, device="cuda")
    sizes = torch.zeros((n, 2), dtype=torch.int32, device="cuda")
    ctx = mb.Context(0)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        before = ctx.launches
        rc = ctx.lib.ms_quad_crop_resize_pad(ctx.handle, d_pages.data_ptr(), 2, 300, 500, d_rows.data_ptr(), 9,
                                             d_po.data_ptr(), n, 5, 1, 0, 32, 128, batch.data_ptr(), None,
                                             sizes.data_ptr(), C.c_void_p(stream.cuda_stream))
        assert rc == 0, mb._cabi.last_error()
        assert ctx.launches - before == 3  # plan, fallback list, generic kernel (1500-byte rows are not 16-byte aligned: no staged kernel)
    stream.synchronize()
    got, sz = batch.cpu().numpy(), sizes.cpu().numpy()
    for i in range(n):
        if page_of[i] > 1:
            assert tuple(sz[i]) == (0, 0) and (got[i] == 1.0).all()
            continue
        assert tuple(sz[i]) == cpu.quad_patch_size(rows[i, :8])
        _, chw = cpu.quad_crop_resize_pad(pages[page_of[i]], rows[i, :8], 32, 128, 5, "replicate")
        if chw is None:
            assert tuple(sz[i]) == (0, 0)
        else:
            np.testing.assert_array_equal(got[i], chw)


# ---- the rest of the reference's Pipeline surface (tests/test_pipeline_api_compatibility.py:95-238, case by case) ------
def test_pipeline_non_tuple_recognizer_confidence(mb):
    pipe = mb.Pipeline(detector=DummyDetector(mb), recognizer=DummyRecognizer())
    page = pipe.predict(np.zeros((100, 400, 3), np.uint8), recognize_text=True, vis=False)
    assert page.blocks[0].words[0].text == "word1" and page.blocks[0].words[0].recognition_confidence == 0.9


def test_pipeline_without_recognition(mb):
    rec = DummyRecognizer()
    page = mb.Pipeline(detector=DummyDetector(mb), recognizer=rec).predict(np.zeros((100, 400, 3), np.uint8),
                                                                          recognize_text=False, vis=False)
    assert rec.call_count == 0 and page.blocks[0].words[0].text is None


def test_pipeline_with_visualization(mb):
    """reference test :177-188: vis=True returns (Page, PIL.Image); also with recognize_text=False (_pipeline.py:81-87)
    and from EAST.predict (infer.py:390)."""
    from PIL import Image

    pipe = mb.Pipeline(detector=DummyDetector(mb), recognizer=DummyRecognizer())
    img = np.zeros((100, 400, 3), np.uint8)
    page, vis_img = pipe.predict(img, recognize_text=True, vis=True)
    assert isinstance(page, mb.Page) and isinstance(vis_img, Image.Image) and vis_img.size == (400, 100)
    assert np.asarray(vis_img).any()  # something was drawn
    page2, vis2 = pipe.predict(img, recognize_text=False, vis=True)
    assert isinstance(page2, mb.Page) and isinstance(vis2, Image.Image)


def test_pipeline_get_text_and_process_batch(mb):
    pipe = mb.Pipeline(detector=DummyDetector(mb), recognizer=DummyRecognizer())
    img = np.zeros((100, 400, 3), np.uint8)
    text = pipe.get_text(pipe.predict(img))
    assert "word1" in text and "word2" in text and "word3" in text
    pages = pipe.process_batch([img, img])
    assert len(pages) == 2 and all(isinstance(p, mb.Page) for p in pages)
    assert all(isinstance(p, mb.Page) for p in pipe.process_batch([img], vis=True))


def test_pipeline_pil_input_and_defaults(mb, tmp_path, monkeypatch):
    from PIL import Image

    rng = np.random.default_rng(3)
    arr = rng.integers(0, 256, (100, 400, 3), dtype=np.uint8)
    rec = DummyRecognizer()
    page = mb.Pipeline(detector=DummyDetector(mb), recognizer=rec).predict(Image.fromarray(arr))
    np.testing.assert_array_equal(rec.seen[1], arr[10:50, 110:200])
    assert [w.text for w in page.blocks[0].words] == ["word1", "word2", "word3"]
    f = tmp_path / "page.png"
    Image.fromarray(arr).save(f)
    np.testing.assert_array_equal(mb.read_image(str(f)), arr)
    np.testing.assert_array_equal(mb.read_image(f), arr)
    # Pipeline() builds EAST() / TRBA() from the released weights like the reference (_pipeline.py:52-54); without them
    # (no network here) that is a FileNotFoundError, as the reference's torch.load raises
    monkeypatch.setenv("HOME", str(tmp_path))
    import manuscript_b200.east as east_mod
    import manuscript_b200.trba as trba_mod

    monkeypatch.setattr(east_mod, "DEFAULT_WEIGHTS", tmp_path / "east.pth")
    monkeypatch.setattr(trba_mod, "DEFAULT_DIR", tmp_path / "trba")
    with pytest.raises(FileNotFoundError):
        mb.Pipeline()
    with pytest.raises(FileNotFoundError):
        mb.Pipeline(detector=DummyDetector(mb))


def test_detector_input_matches_cv2_and_torchvision_formula(mb):
    """ms_detector_input = cv2.resize(img, (T, T)) [INTER_LINEAR] -> x / 255 -> (x - 0.5) / 0.5 (infer.py:301-305),
    bit for bit, shrinking, enlarging, by exactly 2, and unchanged."""
    import ctypes as C

    import cv2
    import torch

    rng = np.random.default_rng(11)
    ctx = mb.Context(0)
    for (h, w), t in [((333, 517), 256), ((700, 900), 512), ((100, 180), 256), ((512, 512), 256), ((256, 256), 256),
                      ((1031, 777), 640), ((64, 2000), 128)]:
        img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        d_img = torch.from_numpy(img).cuda()
        out = torch.empty((3, t, t), dtype=torch.float32, device="cuda")
        u8 = torch.empty((t, t, 3), dtype=torch.uint8, device="cuda")
        rc = ctx.lib.ms_detector_input(ctx.handle, d_img.data_ptr(), h, w, t, t, out.data_ptr(), u8.data_ptr(),
                                       C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0, mb._cabi.last_error()
        torch.cuda.synchronize()
        want_u8 = cv2.resize(img, (t, t))
        np.testing.assert_array_equal(u8.cpu().numpy(), want_u8, err_msg=f"{(h, w)} -> {t}")
        tt = torch.from_numpy(want_u8).permute(2, 0, 1).float().div(255.0)
        want = ((tt - 0.5) / 0.5).numpy()
        np.testing.assert_array_equal(out.cpu().numpy(), want)
        np.testing.assert_array_equal(want_u8, cpu.cv_resize(img, (t, t), "linear"))  # and the oracle agrees with cv2


def test_pipeline_fused_route_is_device_resident_and_exact(mb):
    """mb.EAST + mb.TRBA: one upload of the page, maps / boxes / crops never leave the device, the recogniser network
    reads views of the batch the crop kernel wrote.  Results against the oracle chain: boxes in the reference's
    reading order, every crop bit-exact, text written back to the right words."""
    import torch

    target, words = 512, 60
    score, geo, _ = synthdata.make_maps(5, target, words)
    img = synthdata.make_page_image(5, 700)[:600, :700].copy()
    net_in = {}

    class Net:
        def __call__(self, x):
            net_in["x"] = x
            return {"score": torch.from_numpy(score)[None, None].cuda(), "geometry": torch.from_numpy(geo)[None].cuda()}

    batches = []

    def rec_model(batch):
        assert batch.is_cuda
        batches.append(batch)
        return [(f"w{sum(len(b) for b in batches) - len(batch) + i}", 0.75) for i in range(len(batch))]

    det = mb.EAST(model=Net(), target_size=target)
    rec = mb.TRBA(model=rec_model, img_h=32, img_w=128, batch_size=32)
    uploads = []
    orig_upload = det.upload
    det.upload = lambda a: (uploads.append(a.nbytes), orig_upload(a))[1]
    pipe = mb.Pipeline(detector=det, recognizer=rec)
    page = pipe.predict(img)
    assert pipe.last_route == "fused" and uploads == [img.nbytes]  # the page crossed PCIe once
    # the network input was made on the device from that upload: cv2.resize + ToTensor + Normalize
    import cv2

    tt = torch.from_numpy(cv2.resize(img, (target, target))).permute(2, 0, 1).float().div(255.0)
    np.testing.assert_array_equal(net_in["x"][0].cpu().numpy(), ((tt - 0.5) / 0.5).numpy())
    # oracle chain + the reference's reading order (host restatement, pinned to the reference goldens)
    q = cpu.decode_quads_from_maps(score, geo, 0.6, 4.0, 2)
    boxes = cpu.east_postprocess(cpu.locality_aware_nms(q, 0.2), (600, 700), target_size=target)
    ib = []
    for b in boxes[:, :8]:
        xs, ys = np.trunc(b[0::2]).astype(np.int64), np.trunc(b[1::2]).astype(np.int64)
        ib.append((int(xs.min()), int(ys.min()), int(xs.max()), int(ys.max())))
    want = boxes[_host_order(mb, ib)]
    got_words = page.blocks[0].words
    assert len(got_words) == len(want)
    got = np.array([[v for pt in w.polygon for v in pt] + [w.detection_confidence] for w in got_words], np.float32)
    np.testing.assert_array_equal(got, want)
    rects, valid = cpu.word_rects(want, 600, 700, 5)
    all_crops = torch.cat(batches).cpu().numpy()
    assert len(all_crops) == int(valid.sum()) and all(len(b) <= 32 for b in batches)
    for j, r in enumerate(rects[valid]):
        np.testing.assert_array_equal(all_crops[j], cpu.crop_resize_pad(img, r, 32, 128)[1])
    texts = [w.text for w, ok in zip(got_words, valid) if ok]
    assert texts == [f"w{i}" for i in range(len(texts))]
    assert all(w.text is None for w, ok in zip(got_words, valid) if not ok)
    assert got_words[0].recognition_confidence == 0.75
    # same answer as the generic route (any detector + this TRBA: the page is uploaded once, crops stay on the device)
    batches.clear()
    dummy = DummyDetector(mb, "dict", [mb.Word(polygon=[tuple(p) for p in b[:8].reshape(4, 2).tolist()],
                                               detection_confidence=float(b[8])) for b in boxes])
    pipe2 = mb.Pipeline(detector=dummy, recognizer=rec)
    page2 = pipe2.predict(img)
    assert pipe2.last_route == "device_crops"
    np.testing.assert_array_equal(torch.cat(batches).cpu().numpy(), all_crops)
    assert [w.polygon for w in page2.blocks[0].words] == [w.polygon for w in got_words]
    # vis=True on the fused route
    from PIL import Image

    batches.clear()
    pg, vis_img = pipe.predict(img, vis=True)
    assert isinstance(vis_img, Image.Image) and len(pg.blocks[0].words) == len(want)
    # a repeated call on the same buffers replays the library's CUDA graph and gives the same page
    batches.clear()
    again = pipe.predict(img)
    assert [w.polygon for w in again.blocks[0].words] == [w.polygon for w in got_words]


# ---- reading order of pages beyond the shared-memory kernel: the global-memory kernel, then the flag + host restatement ---
def test_reading_order_large_pages(mb, golden_dir):
    """BASELINE configs[3] (10 000 boxes > 4096) and a page of 3000 boxes with > 28 672 intersecting pairs run in the
    global-memory kernel (reading_order_large_kernel): no flag, device order == the REAL reference's (committed by
    tests/golden/make_golden_large.py).  A page with more intersecting pairs than that kernel holds keeps its
    detection order and is flagged (MS_FLAG_ORDER_OVERFLOW); word_reading_order / reorder_words / Pipeline.predict
    then use the exact host restatement."""
    import ctypes as C

    import torch

    from manuscript_b200._cabi import MS_FLAG_ORDER_OVERFLOW
    from manuscript_b200.reading_order import host_word_order

    g = np.load(os.path.join(golden_dir, "large_pages.npz"))
    page, words = 4096, 10000
    score, geo, _ = synthdata.make_maps(3, page, words)
    img = synthdata.make_page_image(3, page)
    plain = mb.PageBatch(device=0, params=mb.EastParams.default(target_size=page), cap_boxes=16384, want_batch=False)
    final = plain.run(torch.from_numpy(score[None]).cuda(), torch.from_numpy(geo[None]).cuda(), None,
                      sync=True).page_boxes(0).cpu().numpy()
    assert len(final) == int(g["cfg3_n_final"])
    order = mb.word_reading_order(final[:, :8])            # 10 000 boxes: the global-memory kernel
    np.testing.assert_array_equal(order, g["cfg3_order"])  # == the reference's order
    np.testing.assert_array_equal(host_word_order(final[:, :8]), g["cfg3_order"])  # the last-resort host restatement too
    ro = mb.PageBatch(device=0, params=mb.EastParams.default(target_size=page, sort_reading_order=1), cap_boxes=16384,
                      crops_cap=12000)
    res = ro.run(torch.from_numpy(score[None]).cuda(), torch.from_numpy(geo[None]).cuda(),
                 torch.from_numpy(img[None]).cuda(), sync=False)
    torch.cuda.synchronize()
    assert int(res.flags.cpu()[0]) == 0 and list(res.order_overflow_pages()) == []
    np.testing.assert_array_equal(res.page_boxes(0).cpu().numpy(), final[g["cfg3_order"]])
    res.raise_for_flags()
    rects, valid = cpu.word_rects(final[g["cfg3_order"]], page, page, 5)
    nc = int(res.n_crops.cpu()[0])
    np.testing.assert_array_equal(res.crops[:nc].cpu().numpy()[:, 1:], rects[valid])  # the crops follow the reading order

    # the whole thing through Pipeline.predict: fused route, everything on the device
    class Net:
        def __call__(self, x):
            return {"score": torch.from_numpy(score)[None, None].cuda(), "geometry": torch.from_numpy(geo)[None].cuda()}

    seen = []
    rec = mb.TRBA(model=lambda b: (seen.append(len(b)), [("t", 0.5)] * len(b))[1], img_h=32, img_w=128, batch_size=512)
    pipe = mb.Pipeline(detector=mb.EAST(model=Net(), target_size=page, cap_boxes=16384), recognizer=rec)
    pg = pipe.predict(img)
    assert pipe.last_route == "fused"
    got = np.array([[v for pt in w.polygon for v in pt] for w in pg.blocks[0].words], np.float32)
    np.testing.assert_array_equal(got, final[g["cfg3_order"], :8])
    assert sum(seen) == sum(1 for w in pg.blocks[0].words if w.text == "t") == 10000

    # <= 4096 boxes but more intersecting pairs than the shared-memory kernel holds: the global-memory kernel again
    rng = np.random.default_rng(7)
    n = 3000
    x0, y0 = rng.integers(0, 800, n), rng.integers(0, 800, n)
    bx = np.stack([x0, y0, x0 + rng.integers(20, 80, n), y0 + rng.integers(10, 40, n)], axis=1)
    b64 = bx.astype(np.int64)
    inter = ~((b64[:, None, 2] <= b64[None, :, 0]) | (b64[None, :, 2] <= b64[:, None, 0]) |
              (b64[:, None, 3] <= b64[None, :, 1]) | (b64[None, :, 3] <= b64[:, None, 1]))
    n_pairs = (int(inter.sum()) - n) // 2
    assert 28672 < n_pairs < 65536, n_pairs
    assert list(mb.word_reading_order(_boxes_to_polys(bx))) == _host_order(mb, bx)

    # far too many intersecting pairs for either kernel: flagged on the device, ordered by the host restatement
    x0, y0 = rng.integers(0, 300, n), rng.integers(0, 300, n)
    bx = np.stack([x0, y0, x0 + rng.integers(20, 80, n), y0 + rng.integers(10, 40, n)], axis=1)
    polys = _boxes_to_polys(bx)
    assert list(mb.word_reading_order(polys)) == _host_order(mb, bx)
    ctx = mb.ops.default_context()
    rows = np.zeros((n, 9), np.float32)
    rows[:, :8] = np.asarray(polys, np.float32).reshape(n, 8)
    rows[:, 8] = np.arange(n)
    d_rows = torch.from_numpy(rows).cuda()
    d_cnt = torch.tensor([n], dtype=torch.int32, device="cuda")
    d_ord = torch.full((n,), -1, dtype=torch.int32, device="cuda")
    d_out = torch.zeros_like(d_rows)
    d_flags = torch.zeros((1,), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    mb._cabi.check(ctx.lib.ms_reading_order(ctx.handle, d_rows.data_ptr(), d_cnt.data_ptr(), 1, n, d_ord.data_ptr(),
                                            d_out.data_ptr(), d_flags.data_ptr(), C.c_void_p(0)))
    torch.cuda.synchronize()
    assert int(d_flags.cpu()[0]) == MS_FLAG_ORDER_OVERFLOW
    np.testing.assert_array_equal(d_ord.cpu().numpy(), np.arange(n))   # detection order, every row intact
    np.testing.assert_array_equal(d_out.cpu().numpy(), rows)
    with pytest.raises(mb.CABIError):
        mb.batch._raise_for_flags(d_flags.cpu().numpy())
    mb.batch._raise_for_flags(d_flags.cpu().numpy(), allow_order_overflow=True)


def test_reading_order_large_kernel_on_every_golden(golden_dir):
    """MS_B200_RO_FORCE_LARGE=1 (read when a context is created) sends every page through the global-memory kernel:
    the reference's 30 golden cases, detector output with fractional coordinates, duplicated boxes (the dict / first-match
    quirks), boxes of zero height (avg_h <= 0: every box its own line) and a batch of pages of different sizes."""
    import ctypes as C

    import torch

    import manuscript_b200 as mb

    os.environ["MS_B200_RO_FORCE_LARGE"] = "1"
    try:
        ctx = mb._cabi.Context(0)
    finally:
        del os.environ["MS_B200_RO_FORCE_LARGE"]
    g = np.load(os.path.join(golden_dir, "reading_order.npz"))
    for i in range(int(g["n_cases"])):
        boxes = g[f"boxes_{i}"]
        got = mb.word_reading_order(_boxes_to_polys(boxes), ctx=ctx)
        np.testing.assert_array_equal(boxes[got].reshape(-1, 4), g[f"sorted_res_{i}"], err_msg=f"case {i}")
        assert list(got) == _host_order(mb, boxes), f"case {i}"
    rng = np.random.default_rng(11)
    cases = []
    for n, side in ((1, 50), (2, 50), (700, 900), (2500, 2000), (5000, 3000)):
        x0, y0 = rng.integers(0, side, n), rng.integers(0, side, n)
        cases.append(np.stack([x0, y0, x0 + rng.integers(1, 90, n), y0 + rng.integers(1, 40, n)], axis=1))
    dup = cases[2].copy()
    dup[100:200] = dup[300:400]          # exact duplicates
    dup[400:450, 2:] = dup[500:550, 2:]  # boxes that share a corner with another one
    dup[:, 2] = np.maximum(dup[:, 2], dup[:, 0] + 1)  # (the Pipeline's integer boxes are min / max hulls: x0 <= x1)
    dup[:, 3] = np.maximum(dup[:, 3], dup[:, 1] + 1)
    cases.append(dup)
    flat = cases[2].copy()
    flat[:, 3] = flat[:, 1]              # zero height: avg_h == 0
    cases.append(flat)
    page_wide = cases[2].copy()
    page_wide[5] = (0, 0, 900, 900)      # one box over more than 64 grid cells: all-pairs search
    cases.append(page_wide)
    for ci, bx in enumerate(cases):
        assert list(mb.word_reading_order(_boxes_to_polys(bx), ctx=ctx)) == _host_order(mb, bx), f"random case {ci}"
    # a batch of pages (more pages than scratch slots) through the device entry point
    P, cap = 11, 3000
    rows = np.zeros((P, cap, 9), np.float32)
    cnts = np.zeros(P, np.int32)
    per_page = []
    for pg in range(P):
        n = int(rng.integers(0, 2500)) if pg != 4 else 0
        x0, y0 = rng.integers(0, 1500, n), rng.integers(0, 1500, n)
        bx = np.stack([x0, y0, x0 + rng.integers(1, 90, n), y0 + rng.integers(1, 40, n)], axis=1).reshape(n, 4)
        per_page.append(bx)
        cnts[pg] = n
        if n:
            rows[pg, :n, :8] = np.asarray(_boxes_to_polys(bx), np.float32).reshape(n, 8)
            rows[pg, :n, 8] = np.arange(n)
    d_rows, d_cnt = torch.from_numpy(rows).cuda(), torch.from_numpy(cnts).cuda()
    d_ord = torch.full((P, cap), -1, dtype=torch.int32, device="cuda")
    d_out = torch.zeros_like(d_rows)
    d_flags = torch.zeros((P,), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    mb._cabi.check(ctx.lib.ms_reading_order(ctx.handle, d_rows.data_ptr(), d_cnt.data_ptr(), P, cap, d_ord.data_ptr(),
                                            d_out.data_ptr(), d_flags.data_ptr(), C.c_void_p(0)))
    torch.cuda.synchronize()
    assert not d_flags.cpu().numpy().any()
    for pg in range(P):
        want = _host_order(mb, per_page[pg])
        assert d_ord[pg, : cnts[pg]].cpu().tolist() == want, f"page {pg}"
        np.testing.assert_array_equal(d_out[pg, : cnts[pg]].cpu().numpy(), rows[pg, want] if len(want) else rows[pg, :0])
    ctx.close()


# ---- BASELINE configs[0]: the plumbing run on the reference's example image, random-init reference network -----------------
def test_configs0_example_image_random_init_network(mb, golden_dir):
    """tests/golden/make_golden_cfg0.py ran the reference's OWN network module (detectors/_east/east.py, random init,
    seed 0, CPU) on example/ocr_example_image.jpg prepared as EAST.predict prepares it, and the reference's
    post-processing on the maps it produced (score_thresh = the map's median: random init never reaches 0.6).  Here
    the maps are replayed (the geometry map at the pixels the decode reads) through mb.EAST and mb.Pipeline: the network
    input made on the device is bit-identical to the reference's, and candidates / kept rows / final boxes equal the
    reference's outputs."""
    import hashlib

    import torch

    g = np.load(os.path.join(golden_dir, "cfg0_example.npz"))
    target, thr = int(g["target"]), float(g["score_thresh"])
    score, resized = g["score"], g["resized"]
    # the fixture keeps the geometry only at the pixels a quantisation-2 decode reads (the centre of every 2x2 cell);
    # every other pixel is zero, so a decode that reads a wrong pixel gets a wrong quad
    geo = np.zeros((8, *score.shape), np.float32)
    geo[:, 1::2, 1::2] = g["geo_centres"]
    seen = {}

    class Net:  # stands in for the reference's network: checks its input, replays the maps the real one produced
        def __call__(self, x):
            seen["sha"] = hashlib.sha256(x[0].cpu().numpy().tobytes()).hexdigest()
            return {"score": torch.from_numpy(score)[None, None].cuda(), "geometry": torch.from_numpy(geo)[None].cuda()}

    det = mb.EAST(model=Net(), target_size=target, score_thresh=thr, cap_boxes=8192)
    quads = mb.decode_quads_from_maps(score, geo, thr, 4.0, 2)
    assert len(quads) == int(g["n_candidates"])
    assert hashlib.sha256(quads.tobytes()).hexdigest() == str(g["quads_sha"])
    np.testing.assert_array_equal(mb.locality_aware_nms(quads, 0.2), g["lanms"])
    orig_hw = tuple(int(v) for v in g["orig_hw"])
    np.testing.assert_array_equal(det.boxes_from_maps(score, geo, orig_hw), g["final"])
    # EAST.predict / Pipeline.predict on the (already resized) example image: same network input as the reference made
    out = det.predict(resized, return_maps=True)
    assert seen["sha"] == str(g["input_sha"])
    np.testing.assert_array_equal(out["score_map"], score)
    want = cpu.east_postprocess(g["lanms"], (target, target), target_size=target)
    got = np.array([[v for pt in w.polygon for v in pt] + [w.detection_confidence] for w in out["page"].blocks[0].words],
                   np.float32)
    np.testing.assert_array_equal(got, want)
    rec = mb.TRBA(model=lambda b: [("", 0.0)] * len(b), img_h=64, img_w=256)  # the reference's default canvas
    pipe = mb.Pipeline(detector=det, recognizer=rec)
    page = pipe.predict(resized)
    assert pipe.last_route in ("fused", "fused+host_order")
    assert len(page.blocks[0].words) == len(want)
