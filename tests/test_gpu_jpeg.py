"""Baseline-JPEG decode on the device (ms_jpeg_decode_batch through EAST.upload / upload_batch and the fused Pipeline
routes): every page equal in every byte to cv2.cvtColor(cv2.imread(path), cv2.COLOR_BGR2RGB), and every file the
device takes decoded there (EAST.device_decoded).  Every file is encoded in the test from seeded arrays."""
import ctypes as C
import io

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

from test_gpu_batch_pipeline import T, StubEAST, StubTRBA, page_fields  # noqa: E402
from test_jpeg_inspect import SAMPLING, encode, with_orientation  # noqa: E402

pytestmark = pytest.mark.gpu

SIZES = [(1, 1), (7, 9), (8, 8), (16, 16), (17, 1), (1, 2049), (2047, 1531)]


@pytest.fixture(scope="module")
def mb():
    import manuscript_b200 as m

    return m


@pytest.fixture(scope="module")
def det(mb):
    return mb.EAST(model=None)


def content(kind, h, w, seed):
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == "blank":
        return np.full((h, w, 3), 255, np.uint8)
    a = np.full((h, w, 3), 244, np.uint8) + rng.integers(0, 8, (h, w, 3), dtype=np.uint8)  # paper and ink
    for _ in range(max(1, h * w // 3000)):
        y, x = int(rng.integers(0, h)), int(rng.integers(0, w))
        a[y:y + 9, x:x + 40] = int(rng.integers(0, 70))
    return a


def write(tmp_path, name, data):
    p = tmp_path / name
    p.write_bytes(data)
    return p


def cv2_rgb(p):
    return cv2.cvtColor(cv2.imread(str(p)), cv2.COLOR_BGR2RGB)


def check_batch(det, paths, on_device=True):
    pages = det.upload_batch(paths)
    got = [pg.cpu().numpy() for pg in pages]
    for p, g in zip(paths, got):
        np.testing.assert_array_equal(g, cv2_rgb(p), err_msg=str(p))
    if on_device is not None:
        assert det.device_decoded == [on_device] * len(paths)
    return pages


def encode_gray_or(img, sampling, **kw):
    if sampling == "gray":
        return encode(cv2.cvtColor(img, cv2.COLOR_RGB2GRAY), **kw)
    return encode(img, sampling, **kw)


@pytest.mark.parametrize("quality", [30, 75, 90, 100])
@pytest.mark.parametrize("sampling", list(SAMPLING) + ["gray"])
def test_sampling_quality_sizes_contents(det, tmp_path, sampling, quality):
    paths = []
    for i, (h, w) in enumerate(SIZES):
        for kind in ("noise", "blank", "doc"):
            if (h, w) == (2047, 1531) and kind != "doc" and quality not in (30, 100):
                continue  # the large noise / blank pages at the two extreme qualities only
            data = encode_gray_or(content(kind, h, w, i * 31 + quality), sampling, quality=quality)
            paths.append(write(tmp_path, f"{sampling}_{quality}_{h}x{w}_{kind}.jpg", data))
    check_batch(det, paths)


@pytest.mark.parametrize("rst", [0, 1, 3, 64])
@pytest.mark.parametrize("optimize", [False, True])
def test_restart_intervals_and_optimised_tables(det, tmp_path, rst, optimize):
    paths = []
    for sampling in ("420", "444", "411", "gray"):
        for kind, (h, w) in (("doc", (301, 517)), ("noise", (97, 131)), ("blank", (64, 200))):
            data = encode_gray_or(content(kind, h, w, rst + 7), sampling, quality=85, rst=rst, optimize=optimize)
            paths.append(write(tmp_path, f"{sampling}_{kind}_r{rst}_o{int(optimize)}.jpg", data))
    check_batch(det, paths)


def test_pil_encoded_files(det, tmp_path):
    from PIL import Image

    paths = []
    for i, (q, ss, opt) in enumerate([(75, 2, False), (95, 0, False), (50, 1, False), (80, 2, True), (90, 0, True)]):
        buf = io.BytesIO()
        kind = "doc" if i % 2 or opt else "noise"  # PIL's one-pass optimised encoder has no room for noise
        Image.fromarray(content(kind, 211, 333, i)).save(buf, "JPEG", quality=q, subsampling=ss, optimize=opt)
        paths.append(write(tmp_path, f"pil_{i}.jpg", buf.getvalue()))
    buf = io.BytesIO()
    Image.fromarray(content("doc", 99, 77, 3)[:, :, 0]).save(buf, "JPEG", quality=70)  # grayscale
    paths.append(write(tmp_path, "pil_gray.jpg", buf.getvalue()))
    check_batch(det, paths)


def test_configs0_shape_page(det, tmp_path):
    data = encode(content("doc", 4250, 5390, 0), "420", quality=90)
    pages = check_batch(det, [write(tmp_path, "cfg0.jpg", data)])
    assert tuple(pages[0].shape) == (4250, 5390, 3)


def mixed_corpus(tmp_path):
    paths = []
    for i, (sampling, (h, w), kind, q, rst) in enumerate([
            ("420", (2047, 1531), "doc", 90, 0), ("444", (17, 1), "noise", 100, 1), ("gray", (1, 2049), "doc", 30, 0),
            ("422", (16, 16), "blank", 75, 3), ("440", (7, 9), "noise", 90, 64), ("411", (301, 517), "doc", 75, 0),
            ("420", (1, 1), "noise", 90, 0), ("444", (8, 8), "doc", 100, 0), ("420", (640, 480), "blank", 90, 1)]):
        data = encode_gray_or(content(kind, h, w, 100 + i), sampling, quality=q, rst=rst)
        paths.append(write(tmp_path, f"mix_{i}.jpg", data))
    return paths


def test_one_batch_mixes_everything(det, tmp_path):
    paths = mixed_corpus(tmp_path)
    pages = check_batch(det, paths)
    ptrs = [pg.data_ptr() for pg in pages]
    assert len(set(ptrs)) == len(ptrs) and all(p % 16 == 0 for p in ptrs)
    base = det._batch_buf[tuple(tuple(pg.shape[:2]) for pg in pages)][0].data_ptr()
    assert all(base <= p < base + det._batch_buf[tuple(tuple(pg.shape[:2]) for pg in pages)][0].numel() for p in ptrs)
    # one page alone, through upload
    one = det.upload(paths[0])
    assert det.device_decoded == [True]
    np.testing.assert_array_equal(one.cpu().numpy(), cv2_rgb(paths[0]))


def bad_files(tmp_path):
    img = content("doc", 300, 400, 9)
    data = encode(img, "420", quality=90)
    sos = data.index(b"\xff\xda")
    truncated = data[:sos + (len(data) - sos) // 2]
    corrupt = bytearray(data)
    k = sos + 200 + (len(data) - sos - 200) // 3
    corrupt[k:k + 2] = b"\xff\xc8"  # a marker in the middle of the entropy-coded data
    rdata = encode(img, "420", quality=90, rst=4)
    rs = bytearray(rdata)
    j = rdata.index(b"\xff\xd2")  # the third restart marker renumbered: a wrong RST sequence
    rs[j + 1] = 0xD5
    return [write(tmp_path, "trunc.jpg", truncated), write(tmp_path, "corrupt.jpg", bytes(corrupt)),
            write(tmp_path, "rst.jpg", bytes(rs))]


def test_bad_entropy_data_takes_the_host_result(mb, det, tmp_path):
    import torch

    paths = bad_files(tmp_path)
    check_batch(det, paths, on_device=False)
    # the C ABI reports them with a status
    datas = [p.read_bytes() for p in paths]
    outs = [torch.empty((300, 400, 3), dtype=torch.uint8, device="cuda") for _ in datas]
    keep = [C.c_char_p(d) for d in datas]
    files = (C.c_void_p * 3)(*[C.cast(k, C.c_void_p).value for k in keep])
    sizes = (C.c_int64 * 3)(*[len(d) for d in datas])
    ptrs = (C.c_void_p * 3)(*[o.data_ptr() for o in outs])
    status = (C.c_int32 * 3)()
    ctx = det._runner.ctx
    mb._cabi.check(ctx.lib.ms_jpeg_decode_batch(ctx.handle, files, sizes, 3, ptrs, status, None))
    torch.cuda.synchronize()
    assert list(status) == [mb.MS_JPEG_BAD_ENTROPY] * 3


def test_progressive_and_rotated_files_take_the_host_path(mb, det, tmp_path):
    img = content("doc", 120, 90, 4)
    good = write(tmp_path, "good.jpg", encode(img, "420"))
    prog = write(tmp_path, "prog.jpg", encode(img, "420", progressive=True))
    rot = write(tmp_path, "rot.jpg", with_orientation(encode(img, "444"), 6))
    png = tmp_path / "page.png"
    cv2.imwrite(str(png), img)
    paths = [prog, good, rot, png]
    pages = det.upload_batch(paths)
    assert det.device_decoded == [False, True, False, False]
    for p, pg in zip(paths, pages):
        np.testing.assert_array_equal(pg.cpu().numpy(), mb.read_image(p))
    assert tuple(pages[2].shape) == (90, 120, 3)


def make_pipe(mb, torch, rotated):
    net = StubEAST(torch, torch.float32)
    det = mb.EAST(model=net, target_size=T)
    rec = mb.TRBA(model=StubTRBA(), img_h=32, img_w=128, batch_size=24)
    return mb.Pipeline(detector=det, recognizer=rec, rotated_crops=rotated)


@pytest.mark.parametrize("rotated", [False, True])
def test_pipeline_paths_equal_arrays(mb, tmp_path, rotated):
    import synthdata
    import torch

    imgs = [synthdata.make_page_image(40 + i, 1100)[:h, :w].copy()
            for i, (h, w) in enumerate([(600, 700), (900, 640), (512, 512), (1000, 1100)])]
    imgs.insert(2, np.full((480, 360, 3), 255, np.uint8))
    paths = []
    for i, im in enumerate(imgs):
        paths.append(write(tmp_path, f"page{i}.jpg", encode(im, "420" if i % 2 else "444", quality=90)))
    arrays = [cv2_rgb(p) for p in paths]
    pipe = make_pipe(mb, torch, rotated)
    want = [pipe.predict(a) for a in arrays]
    route = "fused_rotated" if rotated else "fused"
    assert pipe.last_route == route
    got = [pipe.predict(p) for p in paths]
    assert pipe.last_route == route and pipe.detector.device_decoded == [True]
    assert [page_fields(p) for p in got] == [page_fields(p) for p in want]
    page, vis = pipe.predict(str(paths[0]), vis=True)
    _, vis_want = pipe.predict(arrays[0], vis=True)
    assert page_fields(page) == page_fields(want[0])
    np.testing.assert_array_equal(np.asarray(vis), np.asarray(vis_want))
    batch = pipe.process_batch(paths, max_pages=3)
    assert pipe.last_route == ("fused_batch_rotated" if rotated else "fused_batch")
    assert [page_fields(p) for p in batch] == [page_fields(p) for p in want]
    assert pipe.detector.device_decoded == [True, True]  # the last chunk
    # a second identical call: same page buffer (the page batch replays its graph), same pages
    views = [v.data_ptr() for v in pipe.detector.upload_batch(paths[:3])]
    again = pipe.process_batch(paths, max_pages=3)
    assert [v.data_ptr() for v in pipe.detector.upload_batch(paths[:3])] == views
    assert [page_fields(p) for p in again] == [page_fields(p) for p in want]
    # EAST.predict on a path decodes on the device too
    d = pipe.detector.predict(paths[1])
    assert pipe.detector.device_decoded == [True]
    assert [page_fields(p) for p in [d["page"]]] == [page_fields(pipe.detector.predict(arrays[1])["page"])]
