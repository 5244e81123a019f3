"""The resize oracle (oracle/oracle.c) against cv2.resize itself, swept over every axis size the crop and detector-input
kernels are held to.  Every GPU crop test compares with cpu.cv_resize / cpu.crop_resize_pad, so this pins that reference
to the specification: cv2 (4.x, the version in this image) plus the ResizeAndPadA paste of transforms.py:85-120.

An axis pair (ssize -> dsize) is checked on a 1-pixel-wide strip in each direction, which keeps the other axis at scale
1; the two-row detector-input strips do the same for the page-sized linear shrinks."""
import numpy as np
import pytest

from oracle import cpu

cv2 = pytest.importorskip("cv2")

RNG_BYTES = np.random.default_rng(1234).integers(0, 256, 4096 * 2 * 3, dtype=np.uint8)


def resize_and_pad(crop, ih, iw):
    """ResizeAndPadA.apply (transforms.py:85-120) written out: scale to fit, Python round (half to even), INTER_AREA
    when a side shrinks else INTER_LINEAR, pasted left-aligned and vertically centred on a 255 canvas"""
    h, w = crop.shape[:2]
    sc = min(ih / h, iw / w)
    nw, nh = max(1, int(round(w * sc))), max(1, int(round(h * sc)))
    interp = cv2.INTER_AREA if (nh < h or nw < w) else cv2.INTER_LINEAR
    canvas = np.full((ih, iw, 3), 255, np.uint8)
    y0 = (ih - nh) // 2
    canvas[y0:y0 + nh, :nw] = cv2.resize(crop, (nw, nh), interpolation=interp)
    return canvas


def sweep_axis_pairs(pairs, interp, rows=1):
    """cpu.cv_resize == cv2.resize on an ssize x `rows` strip along x and along y, for every (ssize, dsize)"""
    flag = cv2.INTER_AREA if interp == "area" else cv2.INTER_LINEAR
    bad = []
    for s, d in pairs:
        strip = RNG_BYTES[: s * rows * 3]
        for img, dsize in ((strip.reshape(rows, s, 3), (d, rows)), (strip.reshape(s, rows, 3), (rows, d))):
            if not np.array_equal(cpu.cv_resize(img, dsize, interp), cv2.resize(img, dsize, interpolation=flag)):
                bad.append((s, d, img.shape[:2]))
                if len(bad) >= 20:
                    return bad
    return bad


def test_area_axis_pairs_match_cv2():
    """every INTER_AREA shrink with dsize 1..256 and ssize up to 3.2 dsize (the persistent kernel's range and past it):
    integer ratios (cv2's fast path) and the float decimation tables, clipped last entries included"""
    pairs = [(s, d) for d in range(1, 257) for s in range(d + 1, int(3.2 * d) + 1)]
    assert len(pairs) > 70000
    assert sweep_axis_pairs(pairs, "area") == []


def test_linear_axis_pairs_match_cv2():
    """every INTER_LINEAR enlargement with dsize 1..256 (ResizeAndPadA's upscale path)"""
    pairs = [(s, d) for d in range(2, 257) for s in range(1, d)]
    assert sweep_axis_pairs(pairs, "linear") == []


@pytest.mark.parametrize("target", [640, 1024, 1280])
def test_detector_input_linear_axes_match_cv2(target):
    """the detector input (infer.py:304): a whole page to target x target with INTER_LINEAR, from every side length up
    to 4096 -- shrinking and enlarging -- on two-row strips"""
    pairs = [(s, target) for s in range(1, 4097) if s != target]
    assert sweep_axis_pairs(pairs, "linear", rows=2) == []


@pytest.mark.parametrize("ih,iw", [(32, 128), (64, 256)])
def test_word_crops_match_cv2(ih, iw):
    """cpu.crop_resize_pad (canvas and normalised batch) == cv2.resize + the ResizeAndPadA paste for word boxes of
    every shape class: copy, INTER_LINEAR, 3- and 4-tap INTER_AREA, exact 2 x 2 and 3 x 3, shrink factors past 3"""
    rng = np.random.default_rng(ih)
    H, W = 600, 1500
    page = rng.integers(0, 256, (H, W, 3), dtype=np.uint8)
    sizes = [(w, h) for h in (1, 2, ih - 1, ih, ih + 1, 2 * ih, 3 * ih, int(2.5 * ih) + 1)
             for w in (1, 2, 3, iw - 1, iw, iw + 1, 2 * iw, 3 * iw, 4 * iw + 3)]
    sizes += [(int(rng.integers(1, 1200)), int(rng.integers(1, 4 * ih))) for _ in range(3000)]
    for w, h in sizes:
        x, y = int(rng.integers(0, W - w + 1)), int(rng.integers(0, H - h + 1))
        want = resize_and_pad(page[y:y + h, x:x + w], ih, iw)
        canvas, chw = cpu.crop_resize_pad(page, (x, y, x + w, y + h), ih, iw)
        assert np.array_equal(canvas, want), (w, h)
        norm = (want.astype(np.float32) - np.float32(127.5)) * (np.float32(1) / np.float32(127.5))
        assert np.array_equal(chw, norm.transpose(2, 0, 1)), (w, h)
