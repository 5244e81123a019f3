"""ms_jpeg_inspect_host (host only): the size cv2.imread decodes to and the device / host decision, for files encoded in
the test from seeded arrays."""
import struct

import numpy as np
import pytest

cv2 = pytest.importorskip("cv2")

SAMPLING = {"444": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_444, "422": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_422,
            "440": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_440, "420": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420,
            "411": cv2.IMWRITE_JPEG_SAMPLING_FACTOR_411}
SIZES = [(1, 1), (7, 9), (8, 8), (16, 16), (17, 1), (1, 2049), (2047, 1531)]


def encode(img, sampling=None, quality=90, rst=0, optimize=False, progressive=False):
    p = [cv2.IMWRITE_JPEG_QUALITY, quality, cv2.IMWRITE_JPEG_OPTIMIZE, int(optimize),
         cv2.IMWRITE_JPEG_PROGRESSIVE, int(progressive)]
    if sampling:
        p += [cv2.IMWRITE_JPEG_SAMPLING_FACTOR, SAMPLING[sampling]]
    if rst:
        p += [cv2.IMWRITE_JPEG_RST_INTERVAL, rst]
    ok, buf = cv2.imencode(".jpg", img, p)
    assert ok
    return buf.tobytes()


def with_orientation(data, orientation):
    """the file with an APP1 Exif segment (little-endian TIFF, IFD0 holding only the orientation) after SOI"""
    tiff = b"II*\x00" + struct.pack("<I", 8) + struct.pack("<H", 1) + struct.pack("<HHIHH", 0x0112, 3, 1, orientation, 0)
    tiff += struct.pack("<I", 0)
    payload = b"Exif\x00\x00" + tiff
    return data[:2] + b"\xff\xe1" + struct.pack(">H", len(payload) + 2) + payload + data[2:]


def inspect(data):
    from manuscript_b200 import jpeg_inspect

    return jpeg_inspect(data)


def decoded_shape(data):
    return cv2.imdecode(np.frombuffer(data, np.uint8), cv2.IMREAD_COLOR).shape[:2]


@pytest.mark.parametrize("h,w", SIZES)
@pytest.mark.parametrize("sampling", list(SAMPLING) + ["gray"])
def test_size_and_decision_of_the_corpus(h, w, sampling):
    rng = np.random.default_rng(h * 7919 + w)
    img = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if sampling == "gray":
        data = encode(cv2.cvtColor(img, cv2.COLOR_BGR2GRAY), rst=3)
    else:
        data = encode(img, sampling, rst=3)
    info = inspect(data)
    assert (info.height, info.width) == decoded_shape(data)
    assert info.device == 1 and info.reason == 0
    assert info.components == (1 if sampling == "gray" else 3)
    assert info.restart_interval == 3


def test_decisions():
    import manuscript_b200 as mb

    rng = np.random.default_rng(5)
    img = rng.integers(0, 256, (37, 53, 3), dtype=np.uint8)
    base = encode(img, "420")
    assert inspect(base).device == 1
    prog = inspect(encode(img, "420", progressive=True))
    assert (prog.device, prog.reason) == (0, mb.MS_JPEG_PROGRESSIVE)
    assert (prog.height, prog.width) == (37, 53)
    rot = with_orientation(base, 6)
    r = inspect(rot)
    assert (r.device, r.reason) == (0, mb.MS_JPEG_ORIENTATION)
    assert (r.height, r.width) == decoded_shape(rot) == (53, 37)  # cv2.imread turns the page
    one = inspect(with_orientation(base, 1))
    assert one.device == 1 and (one.height, one.width) == decoded_shape(with_orientation(base, 1))
    sos = base.index(b"\xff\xda")
    t = inspect(base[:sos - 40])  # the header cut inside the tables
    assert (t.device, t.reason) == (0, mb.MS_JPEG_NOT_JPEG)
    ok, png = cv2.imencode(".png", img)
    n = inspect(png.tobytes())
    assert (n.device, n.reason) == (0, mb.MS_JPEG_NOT_JPEG)
    assert inspect(b"").device == 0
