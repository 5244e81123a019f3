"""The axis-aligned crop path (crop.cu, crop_common.cuh) held to cv2.resize without sampling.

Two layers:
  * the device functions that size a crop and build its coefficient tables (plan_resize, area_entry, build_tables,
    linear_entry_x / _y), evaluated on the device by ms_test_resize_tables_host and compared bit for bit -- every index
    and every float32 weight -- with a float64 numpy restatement of OpenCV's computeResizeAreaTab and of its
    INTER_LINEAR coefficient code;
  * whole canvases from ms_crop_resize_pad_ex (float32 batch and u8 canvas), every pixel of every crop compared with
    cv2.resize plus the ResizeAndPadA paste (transforms.py:85-120), at all four shared-memory tiers of the persistent
    kernel (4, 3, 2 and 1 CTAs per SM) and an odd canvas, with the kernel each crop went to checked through
    ms_crop_last_counts against a restatement of make_plan's staging decision.
"""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

cv2 = pytest.importorskip("cv2")

CANVASES = [(32, 128), (64, 256), (128, 512), (256, 1024), (31, 127)]  # 4, 3, 2, 1 CTAs per SM; scalar padding
K_SRC_BUF = 40 * 1024  # crop.cu kSrcBuf: the largest staged crop
INV = float(np.float32(1) / np.float32(127.5))


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


@pytest.fixture(scope="module")
def tally():
    """what the module compared (printed at the end: run with -s to see it)"""
    t = {"crops": 0, "fast": 0, "entries": 0, "plans": 0}
    yield t
    print(f"\ncrop sweep: {t['crops']} crops compared in full ({t['fast']} by the persistent kernel), "
          f"{t['entries']} table entries and {t['plans']} plans compared bit for bit")


# ---- references ---------------------------------------------------------------------------------------------------
def plan_ref(w, h, ih, iw):
    """transforms.py:80-98 for arrays of (w, h): nw, nh, y0, interp (0 copy, 1 linear, 2 area integer ratio, 3 area
    general), isx, isy and whether the plan alone admits the persistent kernel"""
    w, h = np.asarray(w, np.int64), np.asarray(h, np.int64)
    sc = np.minimum(ih / np.maximum(h, 1), iw / np.maximum(w, 1))
    nw = np.minimum(np.maximum(1, np.rint(w * sc)), iw).astype(np.int64)  # Python round(): half to even
    nh = np.minimum(np.maximum(1, np.rint(h * sc)), ih).astype(np.int64)
    y0 = np.clip((ih - nh) // 2, 0, ih - nh)
    sx, sy = 1.0 / (nw / w), 1.0 / (nh / h)
    isx, isy = np.rint(sx).astype(np.int64), np.rint(sy).astype(np.int64)
    eps = np.finfo(np.float64).eps
    exact = (np.abs(sx - isx) < eps) & (np.abs(sy - isy) < eps)
    interp = np.where((nw == w) & (nh == h), 0, np.where((nh < h) | (nw < w), np.where(exact, 2, 3), 1))
    fast = ((interp == 3) & (sx < 2.999) & (sy < 2.999)) | ((interp == 2) & (isx == 2) & (isy == 2))
    return dict(nw=nw, nh=nh, y0=y0, interp=interp, isx=isx, isy=isy, fast=fast)


def area_ref(ss, ds, d):
    """OpenCV computeResizeAreaTab, entry d of an ssize -> dsize axis (float64, vectorised)"""
    scale = 1.0 / (ds / ss)
    f1 = d * scale
    f2 = f1 + scale
    cell = np.minimum(scale, ss - f1)
    s2 = np.minimum(np.floor(f2).astype(np.int64), ss - 1)
    s1 = np.minimum(np.ceil(f1).astype(np.int64), s2)
    first = (s1 - f1) > 1e-3
    last = (f2 - s2) > 1e-3
    nmid = np.maximum(s2 - s1, 0)
    return dict(s0=np.where(first, s1 - 1, s1), n=first + nmid + last, first=first, nmid=nmid, last=last,
                af=((s1 - f1) / cell).astype(np.float32), am=(1.0 / cell).astype(np.float32),
                al=(np.minimum(np.minimum(f2 - s2, 1.0), cell) / cell).astype(np.float32))


def linear_ref(ss, ds, d, axis):
    """OpenCV's INTER_LINEAR table entry (resize.cpp: float32 position, 11-bit coefficients): x -- source column, edge
    flag, c0, c1; y -- top and bottom source rows, c0, c1"""
    scale = 1.0 / (ds / ss)
    f = ((d + 0.5) * scale - 0.5).astype(np.float32)
    s = np.floor(f).astype(np.int64)
    f = f - s.astype(np.float32)
    if axis == "x":
        f = np.where(s < 0, np.float32(0), f)
        s = np.maximum(s, 0)
        edge = s + 1 >= ss
        f = np.where(edge, np.float32(0), f)
        s0, s1 = np.where(edge, ss - 1, s), edge.astype(np.int64)
    else:
        s0, s1 = np.clip(s, 0, ss - 1), np.clip(s + 1, 0, ss - 1)
    c0 = np.rint((np.float32(1) - f) * np.float32(2048)).astype(np.int64)
    c1 = np.rint(f * np.float32(2048)).astype(np.int64)
    return s0, s1, c0, c1


def resize_and_pad_patch(crop, ih, iw):
    """cv2.resize of ResizeAndPadA.apply: the pasted patch and its row y0 (left-aligned, vertically centred)"""
    h, w = crop.shape[:2]
    sc = min(ih / h, iw / w)
    nw, nh = max(1, int(round(w * sc))), max(1, int(round(h * sc)))
    interp = cv2.INTER_AREA if (nh < h or nw < w) else cv2.INTER_LINEAR
    return cv2.resize(crop, (nw, nh), interpolation=interp), (ih - nh) // 2


def expect_fast(crops, base, n_pages, H, W, ih, iw):
    """make_plan's decision for every crop row: valid, staged (TMA rows fit the 40 KB stage and do not run past the
    page tensor) and a plan the persistent kernel takes"""
    page, x1, y1, x2, y2 = (crops[:, i].astype(np.int64) for i in range(5))
    w, h = x2 - x1, y2 - y1
    ok = (page >= 0) & (page < n_pages) & (w > 0) & (h > 0) & (x1 >= 0) & (y1 >= 0) & (x2 <= W) & (y2 <= H)
    w1, h1 = np.maximum(w, 1), np.maximum(h, 1)
    stride = 3 * W
    first = base + ((page * H + y1) * W + x1) * 3
    last_end = first + (h1 - 1) * stride + 3 * w1
    hi = base + n_pages * H * W * 3
    mis = first & 15 if stride % 16 == 0 else np.full_like(first, 15)
    pitch = (mis + 3 * w1 + 15) & ~15
    staged = (pitch * h1 + 16 <= K_SRC_BUF) & (((last_end + 15) & ~15) <= hi) & (base % 16 == 0)
    return ok & staged & plan_ref(w1, h1, ih, iw)["fast"]


# ---- device evaluation ----------------------------------------------------------------------------------------------
def device_plans(mb, ctx, w, h, ih, iw):
    wh = np.ascontiguousarray(np.stack([w, h], 1), np.int32)
    out = np.zeros((len(wh), 8), np.int32)
    mb._cabi.check(ctx.lib.ms_test_resize_tables_host(ctx.handle, ih, iw, wh.ctypes.data, len(wh), out.ctypes.data,
                                                     None, 0, None, 0))
    return out


def device_tables(mb, ctx, axes):
    """entries (sum of dsize, 8) int32 of the (ssize, dsize, mode) axes"""
    axes = np.ascontiguousarray(axes, np.int32)
    total = int(axes[:, 1].sum())
    out = np.zeros((total, 8), np.int32)
    mb._cabi.check(ctx.lib.ms_test_resize_tables_host(ctx.handle, 1, 1, None, 0, None, axes.ctypes.data, len(axes),
                                                     out.ctypes.data, total))
    return out


def axis_chunks(pairs, limit=1 << 22):
    """(ssize, dsize) pairs in runs of at most `limit` table entries"""
    run, n = [], 0
    for s, d in pairs:
        if run and n + d > limit:
            yield np.array(run, np.int64)
            run, n = [], 0
        run.append((s, d))
        n += d
    if run:
        yield np.array(run, np.int64)


def entry_index(pairs):
    """per entry: its axis' ssize, dsize, first entry and destination index d"""
    ss, ds = pairs[:, 0], pairs[:, 1]
    first = np.concatenate([[0], np.cumsum(ds)[:-1]])
    rep = lambda v: np.repeat(v, ds)  # noqa: E731
    d = np.arange(int(ds.sum())) - rep(first)
    return rep(ss), rep(ds), rep(first), d


def f32_bits(v):
    return np.asarray(v, np.float32).view(np.int32)


def check_area_tables(mb, ctx, pairs, modes, tally):
    for chunk in axis_chunks(pairs):
        ss, ds, first, d = entry_index(chunk)
        ref = area_ref(ss, ds, d)
        taps = [np.where(k < ref["first"], ref["af"], np.where(k < ref["first"] + ref["nmid"], ref["am"], ref["al"]))
                for k in range(4)]
        for mode in modes:
            axes = np.concatenate([chunk, np.full((len(chunk), 1), mode)], 1)
            got = device_tables(mb, ctx, axes)
            tally["entries"] += len(got)
            what = f"mode {mode}"
            if mode == 2:  # the generic kernel's entry: every field the resampling reads
                np.testing.assert_array_equal(got[:, 0], ref["s0"], what)
                np.testing.assert_array_equal(got[:, 1], ref["n"], what)
                np.testing.assert_array_equal(got[:, 2], ref["first"], what)
                np.testing.assert_array_equal(got[:, 3], ref["nmid"], what)
                for col, key, used in ((4, "af", ref["first"]), (5, "am", ref["nmid"] > 0), (6, "al", ref["last"])):
                    bad = used & (got[:, col] != f32_bits(ref[key]))
                    assert not bad.any(), (what, key, list(zip(ss[bad][:5], ds[bad][:5], d[bad][:5])))
                continue
            # build_tables: packed s0 | n << 16 (0xffff << 16 beyond 4 taps), four weights, 0 beyond n
            fits = ref["n"] <= 4
            packed = np.where(fits, ref["s0"] | (ref["n"] << 16), 0xFFFF0000).astype(np.uint32).view(np.int32)
            flat = got.reshape(-1)
            if mode == 0:  # x tables: structure of arrays over the axis' dsize columns
                at = [8 * first + k * ds + d for k in range(5)]
            else:  # y records
                at = [8 * (first + d)] + [8 * (first + d) + 4 + k for k in range(4)]
            np.testing.assert_array_equal(flat[at[0]], packed, what)
            for k in range(4):
                want = np.where(k < ref["n"], f32_bits(taps[k]), 0)
                bad = flat[at[1 + k]] != want
                assert not bad.any(), (what, k, list(zip(ss[bad][:5], ds[bad][:5], d[bad][:5])))


def check_linear_tables(mb, ctx, pairs, tally):
    for chunk in axis_chunks(pairs):
        ss, ds, first, d = entry_index(chunk)
        for mode, axis in ((3, "x"), (4, "y")):
            got = device_tables(mb, ctx, np.concatenate([chunk, np.full((len(chunk), 1), mode)], 1))
            tally["entries"] += len(got)
            for col, want in enumerate(linear_ref(ss, ds, d, axis)):
                bad = got[:, col] != want
                assert not bad.any(), (axis, col, list(zip(ss[bad][:5], ds[bad][:5], d[bad][:5])))


# ---- tables and plans -------------------------------------------------------------------------------------------------
def test_area_tables_fast_range_bit_exact(mb, ctx, tally):
    """dsize 1..256, ssize dsize+1 .. 3.2 dsize: the persistent kernel's x tables and y records (build_tables) and the
    generic kernel's entries (area_entry as fill_axis_table calls it); and dsize 1000 and 1024 (canvases up to 1024
    wide), the only axes here whose windows can end between 1e-4 and 1e-3 past a pixel edge, around OpenCV's 1e-3
    tap threshold"""
    pairs = [(s, d) for d in [*range(1, 257), 1000, 1024] for s in range(d + 1, int(3.2 * d) + 1)]
    check_area_tables(mb, ctx, pairs, (0, 1, 2), tally)


def test_area_tables_generic_range_bit_exact(mb, ctx, tally):
    """dsize 1..64, ssize up to 4096: long decimation windows (the generic kernel) and the y axes of tall crops"""
    pairs = [(s, d) for d in range(1, 65) for s in range(d + 1, 4097)]
    check_area_tables(mb, ctx, pairs, (2,), tally)


def test_linear_tables_bit_exact(mb, ctx, tally):
    """INTER_LINEAR: every enlargement with dsize 1..256 (ResizeAndPadA) and the detector input's 640 / 1024 / 1280
    targets from every side length up to 4096 (linear_entry_x / _y also build detector_input_plan_kernel's tables)"""
    pairs = [(s, d) for d in range(2, 257) for s in range(1, d)]
    pairs += [(s, t) for t in (640, 1024, 1280) for s in range(1, 4097) if s != t]
    check_linear_tables(mb, ctx, pairs, tally)


@pytest.mark.parametrize("ih,iw", CANVASES + [(300, 128)])
def test_plan_sweep(mb, ctx, tally, ih, iw):
    """plan_resize for every (w, h) in 1..2048 x 1..512 against rint of the transforms.py formula"""
    w, h = (a.reshape(-1) for a in np.meshgrid(np.arange(1, 2049), np.arange(1, 513)))
    got = device_plans(mb, ctx, w, h, ih, iw)
    ref = plan_ref(w, h, ih, iw)
    tally["plans"] += len(w)
    for col, key in enumerate(("nw", "nh", "y0", "interp", "isx", "isy", "fast")):
        bad = got[:, col] != ref[key]
        assert not bad.any(), (key, list(zip(w[bad][:5], h[bad][:5], got[bad, col][:5], ref[key][bad][:5])))


# ---- canvases ---------------------------------------------------------------------------------------------------------
def crop_call(mb, torch, ctx, pages, crops, ih, iw, batch=True, canvas=True):
    n = len(crops)
    d_crops = torch.from_numpy(np.ascontiguousarray(crops, np.int32)).cuda()
    n_dev = torch.tensor([n], dtype=torch.int32, device="cuda")
    out = torch.empty((n, 3, ih, iw), dtype=torch.float32, device="cuda") if batch else None
    can = torch.empty((n, ih, iw, 3), dtype=torch.uint8, device="cuda") if canvas else None
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    rc = ctx.lib.ms_crop_resize_pad_ex(ctx.handle, pages.data_ptr(), int(pages.shape[0]), int(pages.shape[1]),
                                       int(pages.shape[2]), d_crops.data_ptr(), n_dev.data_ptr(), n, ih, iw,
                                       out.data_ptr() if batch else None, mb._cabi.MS_DTYPE_F32,
                                       can.data_ptr() if canvas else None, st)
    assert rc == 0, mb._cabi.last_error()
    counts = (C.c_int32 * 2)()
    mb._cabi.check(ctx.lib.ms_crop_last_counts(ctx.handle, counts))
    return out, can, (counts[0], counts[1])


def expected_canvas(torch, pages_np, crops, ih, iw):
    """the u8 canvases cv2.resize + the ResizeAndPadA paste give, built on the device from the pasted patches"""
    n = len(crops)
    patches, nw, nh, y0 = [], np.zeros(n, np.int64), np.zeros(n, np.int64), np.zeros(n, np.int64)
    H, W = pages_np.shape[1:3]
    for i, (p, x1, y1, x2, y2) in enumerate(crops.tolist()):
        if not (0 <= p < len(pages_np) and x2 > x1 and y2 > y1 and x1 >= 0 and y1 >= 0 and x2 <= W and y2 <= H):
            continue  # an invalid row: all padding
        patch, y0[i] = resize_and_pad_patch(pages_np[p, y1:y2, x1:x2], ih, iw)
        nh[i], nw[i] = patch.shape[:2]
        patches.append(patch.reshape(-1))
    want = torch.full((n, ih, iw, 3), 255, dtype=torch.uint8, device="cuda")
    if patches:
        r = torch.from_numpy(np.concatenate(patches)).cuda().view(-1, 3)
        cnt = torch.from_numpy(nw * nh).cuda()
        ci = torch.repeat_interleave(torch.arange(n, device="cuda"), cnt)
        local = torch.arange(len(ci), device="cuda") - (torch.cumsum(cnt, 0) - cnt)[ci]
        nw_d, y0_d = torch.from_numpy(nw).cuda()[ci], torch.from_numpy(y0).cuda()[ci]
        dy = torch.div(local, nw_d, rounding_mode="floor")
        want.view(-1, 3)[(ci * ih + y0_d + dy) * iw + (local - dy * nw_d)] = r
    return want


def check_crops(mb, torch, ctx, tally, pages_np, pages, crops, ih, iw, what, route=True):
    """every pixel of every crop (float32 batch and u8 canvas) against cv2, the kernel counts against make_plan's
    decision; returns the number of crops the persistent kernel took"""
    crops = np.ascontiguousarray(crops, np.int32)
    fast = expect_fast(crops, pages.data_ptr(), *pages_np.shape[:3], ih, iw)
    per = max(1, (1 << 27) // (ih * iw))  # canvas pixels per call
    for lo in range(0, len(crops), per):
        part, fpart = crops[lo:lo + per], fast[lo:lo + per]
        out, can, counts = crop_call(mb, torch, ctx, pages, part, ih, iw)
        want = expected_canvas(torch, pages_np, part, ih, iw)
        bad = (can != want).flatten(1).any(1)
        bad |= (out != (want.float() - 127.5).mul_(INV).permute(0, 3, 1, 2)).flatten(1).any(1)
        idx = bad.nonzero().flatten().tolist()
        assert not idx, (f"{what} at {ih}x{iw}: {len(idx)} of {len(part)} crops differ from cv2, e.g. "
                         f"{[(part[i].tolist(), 'fast' if fpart[i] else 'generic') for i in idx[:6]]}")
        want_counts = (int(fpart.sum()), len(part) - int(fpart.sum()))
        if route:
            assert counts == want_counts, f"{what} at {ih}x{iw}: kernel counts {counts}, make_plan gives {want_counts}"
        tally["crops"] += len(part)
        tally["fast"] += counts[0]
    return int(fast.sum())


def place(rng, sizes, n_pages, H, W):
    """crop rows for (w, h) sizes at random places on random pages"""
    rows = []
    for w, h in sizes:
        p, x, y = int(rng.integers(0, n_pages)), int(rng.integers(0, W - w + 1)), int(rng.integers(0, H - h + 1))
        rows.append((p, x, y, x + w, y + h))
    return np.array(rows, np.int32)


def fast_sizes(ih, iw):
    """(w, h) that the persistent kernel takes at this canvas in the worst 16-byte misalignment: shrink factors from
    1.3 (3 taps) to 2.9 (4 taps) and the exact 2 x 2 ratio, as wide as the 40 KB stage allows"""
    out = []
    for f in (1.3, 1.7, 2.0, 2.5, 2.9):
        h = int(f * ih) + (0 if f == 2.0 else 1)
        wmax = ((K_SRC_BUF - 16) // h // 16 * 16 - 30) // 3
        w = min(int(f * iw) - 1, wmax, 300)
        step = 2 if f == 2.0 else 1
        w -= w % step
        while w > step and not plan_ref(w, h, ih, iw)["fast"]:
            w -= step
        out.append((w, h))
    return out


@pytest.fixture(scope="module")
def word_pages(torch):
    rng = np.random.default_rng(5)
    pages_np = rng.integers(0, 256, (2, 800, 1400, 3), dtype=np.uint8)
    return pages_np, torch.from_numpy(pages_np).cuda()


@pytest.mark.parametrize("ih,iw", CANVASES)
def test_word_crop_families_vs_cv2(mb, torch, ctx, tally, word_pages, ih, iw):
    """every w in 1..1200 at 11 heights around 32 / 64 / 96 (copy, INTER_LINEAR, 3- and 4-tap INTER_AREA, exact 2 x 2
    and 3 x 3, shrink >= 3), every h in 1..200 at 5 widths (tall crops, y-only shrink, nw clamped to 1), tall narrow
    crops that shrink by 1..3 at this canvas (the persistent kernel at this canvas' shared-memory tier), and invalid
    rows mixed in"""
    pages_np, pages = word_pages
    rng = np.random.default_rng(ih * 1000 + iw)
    n_pages, H, W = pages_np.shape[:3]
    wide = place(rng, [(w, h) for h in (33, 40, 47, 48, 63, 64, 65, 80, 95, 96, 97) for w in range(1, 1201)],
                 n_pages, H, W)
    tall = place(rng, [(w, h) for w in (7, 64, 129, 300, 500) for h in range(1, 201)], n_pages, H, W)
    tier = []
    for h in range(ih + 1, min(3 * ih, H)):
        wmax = ((K_SRC_BUF - 16) // h // 16 * 16 - 30) // 3
        tier += [(w, h) for w in {1, 2, max(1, wmax // 2), max(1, wmax)} if w <= W]
    tier = place(rng, tier, n_pages, H, W)
    invalid = np.array([[0, 50, 50, 50, 90], [1, 10, 20, 30, 20], [0, W - 10, 5, W + 20, 40], [0, 5, H - 3, 60, H + 1],
                        [2, 0, 0, 10, 10], [-1, 0, 0, 10, 10], [0, -1, 0, 10, 10]], np.int32)
    mixed = np.concatenate([tall, invalid])
    mixed = mixed[rng.permutation(len(mixed))]
    check_crops(mb, torch, ctx, tally, pages_np, pages, wide, ih, iw, "w sweep")
    check_crops(mb, torch, ctx, tally, pages_np, pages, mixed, ih, iw, "h sweep + invalid rows")
    assert check_crops(mb, torch, ctx, tally, pages_np, pages, tier, ih, iw, "tier crops") >= 50

    # the u8-only and float32-only instantiations write the bytes of the float32 + u8 one
    sub = np.concatenate([tier[::4], mixed[::8]])
    out, can, _ = crop_call(mb, torch, ctx, pages, sub, ih, iw)
    out_only, _, _ = crop_call(mb, torch, ctx, pages, sub, ih, iw, canvas=False)
    _, can_only, _ = crop_call(mb, torch, ctx, pages, sub, ih, iw, batch=False)
    assert torch.equal(out_only.view(torch.int32), out.view(torch.int32))
    assert torch.equal(can_only, can)


@pytest.mark.parametrize("ih,iw", CANVASES)
def test_source_misalignment_vs_cv2(mb, torch, ctx, tally, ih, iw):
    """x1 = 0..15 for sizes the persistent kernel takes, on pages whose rows are a multiple of 16 bytes (512, 2048: one
    misalignment for all rows, area4_strips' kAligned form) and are not (501, 333: it changes from row to row)"""
    rng = np.random.default_rng(7)
    sizes = fast_sizes(ih, iw)
    for W in (512, 2048, 501, 333):
        pages_np = rng.integers(0, 256, (1, 800, W, 3), dtype=np.uint8)
        pages = torch.from_numpy(pages_np).cuda()
        rows = [(0, x1, y1, x1 + w, y1 + h) for w, h in sizes for x1 in range(16) for y1 in (0, 3)
                if x1 + w <= W and y1 + h <= 800]
        crops = np.array(rows, np.int32)
        assert expect_fast(crops, pages.data_ptr(), 1, 800, W, ih, iw).all(), f"page width {W}: not all staged"
        check_crops(mb, torch, ctx, tally, pages_np, pages, crops, ih, iw, f"misalignment, page width {W}")


@pytest.mark.parametrize("ih,iw", CANVASES)
def test_crops_ending_on_the_last_page_byte(mb, torch, ctx, tally, ih, iw):
    """crops whose bottom-right pixel is the last pixel of the page tensor (one page, and the last of three): the
    staged copy rounds the last row up to 16 bytes, which must stay inside the tensor (tail_ok) -- staged when the
    tensor ends on a 16-byte boundary (width 512), generic when it does not (width 333, 801 rows: an odd byte count),
    while the same crops one row higher are staged; exact either way"""
    rng = np.random.default_rng(9)
    H = 801
    for n_pages, W in ((1, 512), (3, 512), (1, 333), (3, 333)):
        pages_np = rng.integers(0, 256, (n_pages, H, W, 3), dtype=np.uint8)
        pages = torch.from_numpy(pages_np).cuda()
        sizes = fast_sizes(ih, iw)
        crops = np.array([(n_pages - 1, W - w, H - h, W, H) for w, h in sizes], np.int32)
        fast = check_crops(mb, torch, ctx, tally, pages_np, pages, crops, ih, iw, f"tail, {n_pages} x {H} x {W}")
        assert fast == (len(crops) if W == 512 else 0)
        higher = np.array([(n_pages - 1, W - w, H - h - 1, W, H - 1) for w, h in sizes], np.int32)
        fast = check_crops(mb, torch, ctx, tally, pages_np, pages, higher, ih, iw, f"one row up, {n_pages} x {H} x {W}")
        assert fast == len(higher)


def test_stage_limit_boundary(mb, torch, ctx, tally):
    """h = 64 at 32 x 128 with w stepped across the 40 KB stage (pitch * h + 16 <= kSrcBuf) at 16-byte misalignments 0
    and 15: the crops on each side go where make_plan says; and 853 x 11 at a 300 x 128 canvas, whose 48-byte pitch
    fills the stage exactly (853 * 48 + 16 == 40960), goes to the persistent kernel"""
    rng = np.random.default_rng(3)
    pages_np = rng.integers(0, 256, (1, 900, 512, 3), dtype=np.uint8)
    pages = torch.from_numpy(pages_np).cuda()
    assert pages.data_ptr() % 16 == 0
    rows = [(0, x1, y1, x1 + w, y1 + 64) for w in range(190, 216) for x1 in (16, 5) for y1 in (0, 7)]  # 3 * 5 % 16 = 15
    crops = np.array(rows, np.int32)
    fast = check_crops(mb, torch, ctx, tally, pages_np, pages, crops, 32, 128, "stage limit")
    assert 0 < fast < len(crops)
    exact = np.array([(0, x1, 10, x1 + 11, 863) for x1 in (0, 5, 16, 21)], np.int32)
    assert check_crops(mb, torch, ctx, tally, pages_np, pages, exact, 300, 128, "stage filled exactly") == len(exact)
