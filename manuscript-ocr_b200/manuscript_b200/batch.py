"""Batched device path: score/geometry maps + page images of many pages -> boxes + TRBA crop batch.

One call of ms_page_batch (include/manuscript_b200.h) runs, for every page of the batch and without a
host round trip, what the reference runs page by page on the CPU:
decode_quads_from_maps (utils.py:328) -> locality_aware_nms (lanms.py:156) -> expand_boxes (utils.py:384)
-> EAST box filters (infer.py:134-233) -> Pipeline crop rectangles (_pipeline.py:125-137,204-221)
-> ResizeAndPadA + normalise + stack (transforms.py:85-120,185-193; recognizers/_trba/__init__.py:382-390).

torch is used for device memory and streams only.
"""
import ctypes as C
from dataclasses import dataclass

import numpy as np

from ._cabi import (MS_FLAG_CAND_OVERFLOW, MS_FLAG_EDGE_OVERFLOW, MS_FLAG_INDEX_ERROR, MS_FLAG_ORDER_OVERFLOW, CABIError,
                    Context, EastParams, batch_dtype_code, check)


def shard_pages(n_pages, world_size, rank):
    """Contiguous page range of `rank` (SURVEY 8e): page i belongs to rank i*world_size//n_pages.
    Pages are independent through the whole path, so there is no collective -- results are gathered
    on the host."""
    if world_size < 1 or not (0 <= rank < world_size):
        raise ValueError("bad world_size / rank")
    lo = -(-rank * n_pages // world_size)  # ceil(rank*n/world)
    hi = -(-(rank + 1) * n_pages // world_size)
    return range(lo, hi)


@dataclass
class PageBatchResult:
    """Results of one batch.  They are VALID ONLY WHEN `flags` is all zero (see raise_for_flags): a page flagged
    MS_FLAG_EDGE_OVERFLOW was resolved with suppression edges missing (boxes that should be gone are returned),
    MS_FLAG_CAND_OVERFLOW means rows were truncated at cap_boxes, MS_FLAG_INDEX_ERROR is where the reference raises
    IndexError (utils.py:370), MS_FLAG_ORDER_OVERFLOW (only with sort_reading_order) means the page is correct but still
    in detection order.  The tensors are owned by the PageBatch runner and are overwritten by its next call of
    the same kind and page count: clone() what has to outlive it."""
    boxes: object        # (P, cap_boxes, 9) f32: rows [0, box_counts[p]) are page p's final boxes
    box_counts: object   # (P,) int32
    crops: object        # (crops_cap, 5) int32 rows [page, x1, y1, x2, y2), first n_crops valid
    n_crops: object      # () / (1,) int32
    batch: object        # (crops_cap | n_crops, 3, h, w) CUDA tensor of the runner's batch_dtype (None if not requested)
    flags: object        # (P,) int32 MS_FLAG_* bits

    def page_boxes(self, p):
        return self.boxes[p, : int(self.box_counts[p])]

    def flags_host(self):
        """The per-page flags as a numpy array (device results: one small D2H copy, synchronises the stream)."""
        f = self.flags
        return f.cpu().numpy() if hasattr(f, "cpu") else np.asarray(f)

    def raise_for_flags(self, allow_order_overflow=False):
        """IndexError / CABIError exactly as the *_host entry points raise them; returns self when all pages are clean.
        allow_order_overflow: pages flagged MS_FLAG_ORDER_OVERFLOW (valid, but in detection order) do not raise."""
        _raise_for_flags(self.flags_host(), allow_order_overflow)
        return self

    def order_overflow_pages(self):
        """Indices of the pages whose reading order was left to the host (MS_FLAG_ORDER_OVERFLOW)."""
        return np.flatnonzero(self.flags_host().reshape(-1) & MS_FLAG_ORDER_OVERFLOW)


class ReadingOrderCapacity(CABIError):
    """MS_FLAG_ORDER_OVERFLOW: the results are valid but in detection order; order them with the host restatement
    (manuscript_b200.reading_order) -- Pipeline.predict and reorder_words do that by themselves."""


def _raise_for_flags(flags, allow_order_overflow=False):
    f = int(np.bitwise_or.reduce(np.asarray(flags).reshape(-1))) if len(flags) else 0
    if allow_order_overflow:
        f &= ~MS_FLAG_ORDER_OVERFLOW
    if f & MS_FLAG_INDEX_ERROR:
        raise IndexError("quantised pixel index outside the map (the reference raises IndexError at utils.py:370)")
    if f & MS_FLAG_CAND_OVERFLOW:
        raise CABIError(-3, "more boxes than cap_boxes on at least one page")
    if f & MS_FLAG_EDGE_OVERFLOW:
        raise CABIError(-3, "NMS suppression-edge buffer exceeded")
    if f & MS_FLAG_ORDER_OVERFLOW:
        raise ReadingOrderCapacity(-3, "a page exceeds the device reading-order capacity (max(65536, 16 cap_boxes) intersecting "
                                       "pairs): its boxes and crops are in detection order")


class PageBatch:
    """Reusable runner for one GPU.  Output buffers are allocated once per shape and reused.

    batch_dtype: element type of the crop batch, torch.float32 (default), torch.float16 or torch.bfloat16.  A 16-bit
    batch is written by the crop kernels directly and equals the float32 batch cast with .to(batch_dtype).

    crops_cap: crop rows of the buffers (default n_pages * cap_boxes); it may be changed between calls, and the next
    call reallocates.  max_buffer_sets: keep the device buffers of at most this many page counts, dropping the least
    recently used (default: one set per page count seen)."""

    def __init__(self, device=0, params=None, min_text_size=5, out_hw=(32, 128), cap_boxes=4096, crops_cap=None,
                 want_batch=True, batch_dtype=None, max_buffer_sets=None):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("manuscript_b200.PageBatch needs a CUDA device: there is no CPU fallback")
        self.torch = torch
        self.device = torch.device("cuda", int(device))
        self.ctx = Context(int(device))
        self.params = params if params is not None else EastParams.default()
        self.min_text_size = int(min_text_size)
        self.out_h, self.out_w = int(out_hw[0]), int(out_hw[1])
        self.cap_boxes = int(cap_boxes)
        self.crops_cap = crops_cap
        self.want_batch = bool(want_batch)
        self.batch_dtype = torch.float32 if batch_dtype is None else batch_dtype
        self._dtype_code = batch_dtype_code(self.batch_dtype)
        self.max_buffer_sets = max_buffer_sets
        self._bufs = {}
        self._host = {}
        self._ragged_tables = {}

    # ---- device tensors in, device tensors out; stream-ordered, no synchronisation --------------------------------
    def _device_bufs(self, n_pages):
        torch = self.torch
        key = n_pages
        cap = self.crops_cap if self.crops_cap is not None else n_pages * self.cap_boxes
        b = self._bufs.pop(key, None)  # re-inserted below: the dict is kept in least-recently-used order
        if b is not None and b["cap"] != cap:
            b = None
        if b is None:
            if self.max_buffer_sets is not None:
                while len(self._bufs) >= self.max_buffer_sets:
                    del self._bufs[next(iter(self._bufs))]
            dev = self.device
            b = dict(
                boxes=torch.empty((n_pages, self.cap_boxes, 9), dtype=torch.float32, device=dev),
                counts=torch.zeros((n_pages,), dtype=torch.int32, device=dev),
                crops=torch.zeros((cap, 5), dtype=torch.int32, device=dev),
                n_crops=torch.zeros((1,), dtype=torch.int32, device=dev),
                flags=torch.zeros((n_pages,), dtype=torch.int32, device=dev),
                batch=(torch.empty((cap, 3, self.out_h, self.out_w), dtype=self.batch_dtype, device=dev)
                       if self.want_batch else None),
                cap=cap,
            )
        self._bufs[key] = b
        return b

    def run(self, score, geo, pages=None, sync=False):
        """score (P,H,W) or (P,1,H,W) f32, geo (P,8,H,W) f32, pages (P,IH,IW,3) u8 -- CUDA tensors on this
        runner's device.  Enqueues the whole path on the current stream and returns device tensors.

        sync=False (default): nothing is read back; the results are valid only if `result.flags` is all zero --
        call result.raise_for_flags() (one small D2H copy) before trusting them.
        sync=True: reads the flags, grows the NMS neighbour-pair capacity and runs again on MS_FLAG_EDGE_OVERFLOW
        (the policy of the *_host entry points) and raises IndexError / CABIError for the other flags."""
        if sync:
            while True:
                res = self.run(score, geo, pages, sync=False)
                f = int(np.bitwise_or.reduce(res.flags_host().reshape(-1))) if len(res.flags) else 0
                if (f & MS_FLAG_EDGE_OVERFLOW) and not (f & (MS_FLAG_INDEX_ERROR | MS_FLAG_CAND_OVERFLOW)) \
                        and self.ctx.grow_edge_factor():
                    continue
                return res.raise_for_flags()
        torch = self.torch
        if score.dim() == 4:
            score = score[:, 0]
        P, H, W = score.shape
        assert geo.shape == (P, 8, H, W), geo.shape
        assert score.is_cuda and geo.is_cuda and score.dtype == torch.float32 and geo.dtype == torch.float32
        score = score.contiguous()
        geo = geo.contiguous()
        img_h = img_w = 0
        if pages is not None:
            assert pages.is_cuda and pages.dtype == torch.uint8 and pages.shape[0] == P and pages.shape[3] == 3
            pages = pages.contiguous()
            img_h, img_w = int(pages.shape[1]), int(pages.shape[2])
        b = self._device_bufs(P)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        lib = self.ctx.lib
        with torch.cuda.device(self.device):
            check(lib.ms_page_batch_ex(
                self.ctx.handle, score.data_ptr(), geo.data_ptr(), pages.data_ptr() if pages is not None else None,
                P, H, W, img_h, img_w, C.byref(self.params), self.min_text_size, self.out_h, self.out_w,
                self.cap_boxes, b["boxes"].data_ptr(), b["counts"].data_ptr(), b["crops"].data_ptr(), b["cap"],
                b["n_crops"].data_ptr(), b["batch"].data_ptr() if b["batch"] is not None else None, self._dtype_code,
                None, b["flags"].data_ptr(), C.c_void_p(stream)))
        return PageBatchResult(b["boxes"], b["counts"], b["crops"], b["n_crops"], b["batch"], b["flags"])

    def run_ragged(self, score, geo, pages, sync=False, allow_order_overflow=False):
        """As run(), for page images of their own sizes: `pages` is a list of P CUDA uint8 tensors (H_i, W_i, 3) -- the
        original images, while the maps come from the detector's fixed target_size.  Boxes are scaled to each page's
        size and crops are cut from its pixels (EAST.predict + Pipeline.predict semantics).  `sync` as in run()."""
        if sync:
            while True:
                res = self.run_ragged(score, geo, pages, sync=False)
                f = int(np.bitwise_or.reduce(res.flags_host().reshape(-1))) if len(res.flags) else 0
                if (f & MS_FLAG_EDGE_OVERFLOW) and not (f & (MS_FLAG_INDEX_ERROR | MS_FLAG_CAND_OVERFLOW)) \
                        and self.ctx.grow_edge_factor():
                    continue
                return res.raise_for_flags(allow_order_overflow)
        torch = self.torch
        if score.dim() == 4:
            score = score[:, 0]
        P, H, W = score.shape
        assert geo.shape == (P, 8, H, W) and len(pages) == P
        assert score.is_cuda and geo.is_cuda and score.dtype == torch.float32 and geo.dtype == torch.float32
        score, geo = score.contiguous(), geo.contiguous()
        keep = []
        for pg in pages:
            assert pg.is_cuda and pg.dtype == torch.uint8 and pg.dim() == 3 and pg.shape[2] == 3
            keep.append(pg.contiguous())
        # the pointer / size tables live on the device; the same pages (a serving loop over persistent buffers) reuse
        # the same tables, so that the call's arguments repeat and the library replays its CUDA graph
        sig = tuple((pg.data_ptr(), int(pg.shape[0]), int(pg.shape[1])) for pg in keep)
        cached = self._ragged_tables.get(sig)
        if cached is None:
            if len(self._ragged_tables) >= 8:
                self._ragged_tables.clear()
            cached = self._ragged_tables[sig] = (
                torch.tensor([v[0] for v in sig], dtype=torch.int64).to(self.device),
                torch.tensor([[v[1], v[2]] for v in sig], dtype=torch.int32).to(self.device))
        ptrs, hw = cached
        b = self._device_bufs(P)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            check(self.ctx.lib.ms_page_batch_ragged_ex(
                self.ctx.handle, score.data_ptr(), geo.data_ptr(), ptrs.data_ptr(), hw.data_ptr(), P, H, W,
                C.byref(self.params), self.min_text_size, self.out_h, self.out_w, self.cap_boxes, b["boxes"].data_ptr(),
                b["counts"].data_ptr(), b["crops"].data_ptr(), b["cap"], b["n_crops"].data_ptr(),
                b["batch"].data_ptr() if b["batch"] is not None else None, self._dtype_code, None, b["flags"].data_ptr(),
                C.c_void_p(stream)))
        res = PageBatchResult(b["boxes"], b["counts"], b["crops"], b["n_crops"], b["batch"], b["flags"])
        res._keepalive = (keep, ptrs, hw)  # the kernels read them after this call returns
        return res

    def run_host_ragged(self, score, geo, pages, check_flags=True):
        """As run_host(), `pages` a list of P numpy uint8 arrays (H_i, W_i, 3) of their own sizes."""
        torch = self.torch
        s = np.ascontiguousarray(score, dtype=np.float32)
        if s.ndim == 4:
            s = np.ascontiguousarray(s[:, 0])
        g = np.ascontiguousarray(geo, dtype=np.float32)
        P, H, W = s.shape
        assert g.shape == (P, 8, H, W) and len(pages) == P
        imgs = [np.ascontiguousarray(pg, dtype=np.uint8) for pg in pages]
        for im in imgs:
            assert im.ndim == 3 and im.shape[2] == 3
        ptrs = (C.c_void_p * P)(*[im.ctypes.data for im in imgs])
        hw = np.array([[im.shape[0], im.shape[1]] for im in imgs], np.int32)
        h = self._host_bufs(P)
        dev_batch = C.c_void_p(h["batch"].data_ptr() if self.want_batch else None)
        rc = self.ctx.lib.ms_page_batch_ragged_host_ex(
            self.ctx.handle, s.ctypes.data, g.ctypes.data, ptrs, hw.ctypes.data, P, H, W, C.byref(self.params),
            self.min_text_size, self.out_h, self.out_w, self.cap_boxes, h["boxes"].data_ptr(), h["counts"].data_ptr(),
            h["crops"].data_ptr(), h["cap"], h["n_crops"].data_ptr(), None, self._dtype_code,
            C.byref(dev_batch) if self.want_batch else None, h["flags"].data_ptr())
        if check_flags or rc not in (0, -3, -4):
            check(rc)
        n_crops = int(h["n_crops"][0])
        batch = h["batch"][:n_crops] if self.want_batch and n_crops > 0 else None
        return PageBatchResult(h["boxes"].numpy(), h["counts"].numpy(), h["crops"].numpy(), h["n_crops"].numpy(),
                               batch, h["flags"].numpy())

    # ---- host buffers in, host results out (the crop batch stays on the device, as the reference leaves ------------
    # ---- it on `self.device`, recognizers/_trba/__init__.py:288) ---------------------------------------------------
    def _host_bufs(self, n_pages):
        torch = self.torch
        h = self._host.get(n_pages)
        if h is None:
            cap = self.crops_cap if self.crops_cap is not None else n_pages * self.cap_boxes
            pin = dict(pin_memory=True)
            h = dict(
                boxes=torch.empty((n_pages, self.cap_boxes, 9), dtype=torch.float32, **pin),
                counts=torch.zeros((n_pages,), dtype=torch.int32, **pin),
                crops=torch.zeros((cap, 5), dtype=torch.int32, **pin),
                n_crops=torch.zeros((1,), dtype=torch.int32, **pin),
                flags=torch.zeros((n_pages,), dtype=torch.int32, **pin),
                # the crop batch stays on the device; the runner owns it (never freed under a live view)
                batch=(torch.empty((cap, 3, self.out_h, self.out_w), dtype=self.batch_dtype, device=self.device)
                       if self.want_batch else None),
                cap=cap,
            )
            self._host[n_pages] = h
        return h

    def run_host(self, score, geo, pages=None, check_flags=True):
        """numpy arrays or (pinned) CPU torch tensors of the shapes of run(); score / geo may also be CUDA tensors of
        this GPU (maps the detector left on the device: used in place, only the page images are uploaded).  Copies in, runs, copies the
        boxes / counts / crop list back and synchronises (ms_page_batch_host).  On MS_FLAG_EDGE_OVERFLOW the library
        grows the NMS pair capacity and runs again; other flags raise (check_flags=False returns them instead).

        Lifetime: `result.batch` is a view of a device tensor this runner owns and reuses -- it stays valid memory for
        the runner's life, but the next run_host call with the same page count overwrites it (clone() to keep it);
        the numpy results are views of the runner's pinned host buffers with the same rule."""
        torch = self.torch

        class _Dev:  # a CUDA tensor passed where a host array is expected: the library uses it in place
            def __init__(self, t):
                assert t.dtype == torch.float32 and t.device == self_device, "device maps must be float32 on this GPU"
                self.t = t.contiguous()
                self.shape, self.ndim = tuple(self.t.shape), self.t.dim()
                self.ctypes = type("P", (), {"data": self.t.data_ptr()})

        self_device = self.device

        def as_np(a, dtype):
            if isinstance(a, torch.Tensor):
                if a.is_cuda:
                    return _Dev(a)
                a = a.numpy()
            a = np.asarray(a)
            if a.dtype != dtype or not a.flags.c_contiguous:
                a = np.ascontiguousarray(a, dtype=dtype)
            return a

        s = as_np(score, np.float32)
        if s.ndim == 4:
            s = as_np(score[:, 0], np.float32) if isinstance(s, _Dev) else np.ascontiguousarray(s[:, 0])
        g = as_np(geo, np.float32)
        P, H, W = s.shape
        assert g.shape == (P, 8, H, W), g.shape
        img_h = img_w = 0
        pg = None
        if pages is not None:
            pg = as_np(pages, np.uint8)
            assert pg.shape[0] == P and pg.shape[3] == 3
            img_h, img_w = pg.shape[1], pg.shape[2]
        h = self._host_bufs(P)
        dev_batch = C.c_void_p(h["batch"].data_ptr() if self.want_batch else None)
        lib = self.ctx.lib
        rc = lib.ms_page_batch_host_ex(
            self.ctx.handle, s.ctypes.data, g.ctypes.data, pg.ctypes.data if pg is not None else None, P, H, W,
            img_h, img_w, C.byref(self.params), self.min_text_size, self.out_h, self.out_w, self.cap_boxes,
            h["boxes"].data_ptr(), h["counts"].data_ptr(), h["crops"].data_ptr(), h["cap"], h["n_crops"].data_ptr(),
            None, self._dtype_code, C.byref(dev_batch) if self.want_batch else None, h["flags"].data_ptr())
        if check_flags:
            check(rc)
        elif rc not in (0, -3, -4):
            check(rc)
        n_crops = int(h["n_crops"][0])
        batch = h["batch"][:n_crops] if self.want_batch and n_crops > 0 else None
        return PageBatchResult(h["boxes"].numpy(), h["counts"].numpy(), h["crops"].numpy(), h["n_crops"].numpy(),
                               batch, h["flags"].numpy())
