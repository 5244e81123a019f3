"""EAST detector wrapper with the reference's predict() contract, post-processing on the B200.

Mirrors `EAST` (reference detectors/_east/infer.py:28-132 constructor kwargs, 235-402 predict): image ->
resize -> network -> score / geometry maps -> decode -> LANMS -> expand -> scale -> box filters -> Page.
The network (a ResNet-FPN, reference detectors/_east/east.py) is outside the hot path and is supplied by the
caller as any callable / nn.Module returning {"score": (1,1,H,W), "geometry": (1,8,H,W)}.  Everything around it runs
in the CUDA kernels of this package: the ORIGINAL image is uploaded once, the resized + normalised network input is made
on the device (ms_detector_input = cv2.resize INTER_LINEAR + ToTensor + Normalize, infer.py:301-305), and the maps never
leave the device (the reference's `.cpu().numpy()` at infer.py:312-313 is gone).

Many pages at once: upload_batch puts a list of images into one device buffer, and network_inputs makes all their
network inputs with one ms_detector_input_batch launch.  input_dtype=torch.float16 / torch.bfloat16 (an extension) makes
the network input 16-bit: exactly the float32 input cast with `.to(input_dtype)`.  The caller owns the network's dtype
and memory format: maps in float32, float16 or bfloat16, at any strides (a channels_last geometry), are read by the
post-processing kernels as the network left them, with the results of their float32 dense copies.
"""
import ctypes as C
import time
from pathlib import Path

import numpy as np

from ._cabi import MS_FLAG_EDGE_OVERFLOW, EastParams, batch_dtype_code, check, load_library, maps_descriptor
from .batch import PageBatch, _raise_for_flags
from .imaging import read_image, visualize_page
from .reading_order import reorder_words
from .types import Block, Page, Word

DEFAULT_WEIGHTS = Path.home() / ".manuscript" / "east" / "east_quad_23_05.pth"  # infer.py:101-103


_WORD_FIELDS = frozenset(("polygon", "detection_confidence"))
_FLOAT32 = "float32"  # the default `dtype` of maps_from_device_page(s): torch.float32 (torch is imported lazily)


class JpegInfo(C.Structure):
    """ms_jpeg_info: what ms_jpeg_inspect_host reads from a file's markers."""

    _fields_ = [("height", C.c_int32), ("width", C.c_int32), ("components", C.c_int32), ("device", C.c_int32),
                ("reason", C.c_int32), ("luma_h", C.c_int32), ("luma_v", C.c_int32),
                ("restart_interval", C.c_int32)]


def jpeg_inspect(data):
    """bytes of a file -> JpegInfo (host only, no device needed): the size cv2.imread returns and whether
    ms_jpeg_decode_batch decodes it on the device (reason: MS_JPEG_* code when not)."""
    info = JpegInfo()
    check(load_library().ms_jpeg_inspect_host(data, len(data), C.byref(info)))
    return info


def kernel_maps(score, geo):
    """The maps as the post-processing kernels read them: the tensors themselves when both are float32, float16 or
    bfloat16 of one dtype (at any strides), float32 copies otherwise."""
    import torch

    if score.dtype == geo.dtype and score.dtype in (torch.float32, torch.float16, torch.bfloat16):
        return score, geo
    return score.float(), geo.float()


def _is_path(source):
    return isinstance(source, (str, Path))


def words_from_boxes(boxes):
    """(K, 9) float32 rows -> list of Word (infer.py:359-363).  Scores that pydantic would reject (outside 0..1, NaN)
    go through the validating constructor so that the reference's ValidationError is raised; valid rows are built the
    way BaseModel.model_construct builds them (same attributes, fields_set = the two the reference passes) but without
    its per-field bookkeeping, which at ~2000 words per page would cost more than every kernel of the path together."""
    b = np.asarray(boxes, dtype=np.float32).reshape(-1, 9)
    if len(b) == 0:
        return []
    xy = b[:, :8].astype(np.float64)
    pts = list(zip(xy[:, 0::2].ravel().tolist(), xy[:, 1::2].ravel().tolist()))  # all (x, y) tuples, made in C
    scores = b[:, 8].astype(np.float64).tolist()
    if not bool(np.all((b[:, 8] >= 0.0) & (b[:, 8] <= 1.0))):
        return [Word(polygon=pts[4 * i:4 * i + 4], detection_confidence=s) for i, s in enumerate(scores)]
    out = []
    new, setattr_ = object.__new__, object.__setattr__
    for i, s in enumerate(scores):
        w = new(Word)
        setattr_(w, "__dict__", {"polygon": pts[4 * i:4 * i + 4], "detection_confidence": s, "text": None,
                                 "recognition_confidence": None})
        setattr_(w, "__pydantic_fields_set__", set(_WORD_FIELDS))
        setattr_(w, "__pydantic_extra__", None)
        setattr_(w, "__pydantic_private__", None)
        out.append(w)
    return out


class EAST:
    def __init__(self, model=None, target_size=1280, expand_ratio_w=0.9, expand_ratio_h=0.9, score_thresh=0.6,
                 iou_threshold=0.2, score_geo_scale=0.25, quantization=2, axis_aligned_output=True,
                 remove_area_anomalies=True, anomaly_sigma_threshold=5.0, anomaly_min_box_count=30, device=0,
                 cap_boxes=8192, input_dtype=None):
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("manuscript_b200.EAST needs a CUDA device: there is no CPU fallback")
        self.torch = torch
        self.device = torch.device("cuda", int(device)) if not isinstance(device, torch.device) else device
        self.model = model
        self.target_size = int(target_size)
        self.score_thresh = score_thresh
        self.score_geo_scale = score_geo_scale
        self.iou_threshold = iou_threshold
        self.expand_ratio_w = expand_ratio_w
        self.expand_ratio_h = expand_ratio_h
        self.quantization = quantization
        self.axis_aligned_output = axis_aligned_output
        self.remove_area_anomalies = remove_area_anomalies
        self.anomaly_sigma_threshold = anomaly_sigma_threshold
        self.anomaly_min_box_count = anomaly_min_box_count
        self.cap_boxes = int(cap_boxes)
        self.input_dtype = torch.float32 if input_dtype is None else input_dtype
        self._input_code = batch_dtype_code(self.input_dtype)
        self._runner = PageBatch(device=self.device.index or 0, params=self._params(), cap_boxes=cap_boxes,
                                 want_batch=False)
        self._page_buf = {}   # (h, w) -> persistent device image: stable addresses let repeated calls replay a CUDA graph
        self._input_buf = None
        self._batch_buf = {}  # tuple of image shapes -> (device buffer, page views): see upload_batch
        self._tables = {}     # page views -> their device pointer / size tables
        self._inputs_buf = None
        self.device_decoded = []  # per page of the last upload / upload_batch: decoded from its JPEG on the device

    @classmethod
    def from_pretrained(cls, weights_path=None, **kwargs):
        """What the reference's `EAST()` does (infer.py:94-112): the released weights from
        ~/.manuscript/east/east_quad_23_05.pth (downloaded there by the reference; this package has no network code)
        inside the reference's own network module.  FileNotFoundError when the weights are missing -- what the
        reference's torch.load raises offline -- and ImportError when the reference package that defines the network
        (manuscript.detectors._east.east.EAST) is not installed next to this one."""
        path = Path(weights_path) if weights_path is not None else DEFAULT_WEIGHTS
        if not path.exists():
            raise FileNotFoundError(f"EAST weights not found: {path} (the reference downloads them on first use; "
                                    "pass EAST(model=...) or weights_path=...)")
        from manuscript.detectors._east.east import EAST as EASTModel  # the network is outside this package (infer.py:15)

        det = cls(model=None, **kwargs)
        det.model = EASTModel(pretrained_backbone=False, pretrained_model_path=str(path)).to(det.device).eval()
        return det

    def _params(self, **over):
        return EastParams.default(
            score_thresh=float(np.float32(self.score_thresh)), scale=1.0 / self.score_geo_scale,
            quantization=int(self.quantization), iou_threshold=float(self.iou_threshold),
            expand_ratio_w=float(self.expand_ratio_w), expand_ratio_h=float(self.expand_ratio_h),
            target_size=int(self.target_size), axis_aligned_output=int(bool(self.axis_aligned_output)),
            remove_area_anomalies=int(bool(self.remove_area_anomalies)),
            anomaly_sigma_threshold=float(self.anomaly_sigma_threshold),
            anomaly_min_box_count=int(self.anomaly_min_box_count), **over)

    # ---- the hot path: maps (device or host) -> final boxes (K,9) float32 on the host -----------------------------
    def boxes_from_maps(self, score_map, geo_map, orig_hw):
        """score (H,W) / (1,H,W), geo (8,H,W) torch CUDA tensors or numpy arrays; orig_hw = (h, w) of the image
        the boxes are scaled back to (infer.py:346-348).  Runs infer.py:319-356 on the device.  CUDA tensors of this
        device in float32, float16 or bfloat16 (both the same) are read in place at their strides; anything else is
        converted to float32 first."""
        torch = self.torch
        if all(isinstance(t, torch.Tensor) and t.device == self.device for t in (score_map, geo_map)):
            s, g = kernel_maps(score_map, geo_map)
        else:
            s = torch.as_tensor(score_map, dtype=torch.float32, device=self.device)
            g = torch.as_tensor(geo_map, dtype=torch.float32, device=self.device)
        if s.dim() == 3:
            s = s[0]
        H, W = s.shape
        if g.shape != (8, H, W):
            raise ValueError(f"geo_map must be (8,{H},{W}), got {tuple(g.shape)}")
        maps = maps_descriptor(s[None], g[None])
        r = self._runner
        r.params = self._params()
        ctx, lib = r.ctx, r.ctx.lib
        cap = ((H + max(self.quantization, 1) - 1) // max(self.quantization, 1)) * \
              ((W + max(self.quantization, 1) - 1) // max(self.quantization, 1))
        cap = max(cap, 1)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        cand = torch.empty((cap, 9), dtype=torch.float32, device=self.device)
        kept = torch.empty((cap, 9), dtype=torch.float32, device=self.device)
        out = torch.empty((cap, 9), dtype=torch.float32, device=self.device)
        meta = torch.zeros((8,), dtype=torch.int32, device=self.device)  # n_cand, n_kept, n_out, flags, orig h, w
        meta[4] = int(orig_hw[0])
        meta[5] = int(orig_hw[1])
        p = r.params
        while True:
            meta[:4] = 0
            with torch.cuda.device(self.device):
                check(lib.ms_decode_quads_maps(ctx.handle, C.byref(maps), 1, H, W, p.score_thresh, p.scale,
                                               p.quantization, cand.data_ptr(), cap, meta[0:].data_ptr(),
                                               meta[3:].data_ptr(), C.c_void_p(stream)))
                check(lib.ms_lanms(ctx.handle, cand.data_ptr(), meta[0:].data_ptr(), 1, cap, p.iou_threshold,
                                   kept.data_ptr(), meta[1:].data_ptr(), meta[3:].data_ptr(), C.c_void_p(stream)))
                check(lib.ms_east_boxes(ctx.handle, kept.data_ptr(), meta[1:].data_ptr(), 1, cap, C.byref(p),
                                        meta[4:].data_ptr(), out.data_ptr(), meta[2:].data_ptr(), C.c_void_p(stream)))
            m = meta.cpu().numpy()
            # very dense candidates: grow the NMS neighbour-pair capacity and run again
            if (int(m[3]) & MS_FLAG_EDGE_OVERFLOW) and not (int(m[3]) & 3) and ctx.grow_edge_factor():
                continue
            break
        _raise_for_flags(m[3:4])
        return out[: int(m[2])].cpu().numpy()

    # ---- image -> device, device image -> network input -> maps (nothing returns to the host) --------------------
    def _sources(self, images):
        """Host side of an upload: per source either ("jpeg", file bytes, (h, w, 3)) for a JPEG file the device decodes
        (ms_jpeg_inspect_host) or ("array", contiguous (H, W, 3) uint8 RGB array, shape); other paths go through
        read_image, as they always have."""
        out = []
        for src in images:
            if _is_path(src):
                data = Path(src).read_bytes() if Path(src).is_file() else b""
                info = jpeg_inspect(data) if data else None
                if info is not None and info.device:
                    out.append(("jpeg", data, (int(info.height), int(info.width), 3)))
                    continue
                src = read_image(src)
            a = np.asarray(src)
            if a.ndim != 3 or a.shape[2] != 3 or a.dtype != np.uint8:
                raise ValueError(f"EAST expects (H, W, 3) uint8 RGB images, got shape {a.shape} dtype {a.dtype}")
            a = np.ascontiguousarray(a)
            out.append(("array", a, a.shape))
        return out

    def _decode_jpegs(self, jobs):
        """jobs: (file bytes, device view, path) -> every file decoded into its view (ms_jpeg_decode_batch, one call);
        a file the device does not finish is read with read_image and copied.  Returns the per-job device mask."""
        torch = self.torch
        if not jobs:
            return []
        n = len(jobs)
        keep = [C.c_char_p(d) for d, _, _ in jobs]
        files = (C.c_void_p * n)(*[C.cast(k, C.c_void_p).value for k in keep])
        sizes = (C.c_int64 * n)(*[len(d) for d, _, _ in jobs])
        outs = (C.c_void_p * n)(*[v.data_ptr() for _, v, _ in jobs])
        status = torch.empty((n,), dtype=torch.int32, pin_memory=True)
        stream = torch.cuda.current_stream(self.device)
        with torch.cuda.device(self.device):
            check(self._runner.ctx.lib.ms_jpeg_decode_batch(self._runner.ctx.handle, files, sizes, n, outs,
                                                            status.data_ptr(), C.c_void_p(stream.cuda_stream)))
        stream.synchronize()  # the statuses
        ok = (status.numpy() == 0).tolist()
        for good, (_, v, path) in zip(ok, jobs):
            if not good:  # the host decode: libjpeg's own result for data the device does not take
                a = np.ascontiguousarray(read_image(path))
                if a.shape != tuple(v.shape):
                    raise ValueError(f"{path}: the decoded image is {a.shape}, its header says {tuple(v.shape)}")
                v.copy_(torch.from_numpy(a), non_blocking=True)
        return ok

    def upload(self, img):
        """(H, W, 3) uint8 RGB host array, or a path -> the same image on the device, in a buffer this detector keeps per
        image size.  This is the ONE host-to-device copy of pixels per page: the detector input and the word crops are both
        made from it.  A JPEG file the device takes (ms_jpeg_inspect_host) crosses PCIe compressed and is decoded there,
        bit for bit what read_image gives; self.device_decoded is [True] then, [False] for any other source."""
        torch = self.torch
        (kind, a, shape), = self._sources([img])
        buf = self._page_buf.get(shape[:2])
        if buf is None:
            if len(self._page_buf) >= 4:
                self._page_buf.clear()
            buf = self._page_buf[shape[:2]] = torch.empty(shape, dtype=torch.uint8, device=self.device)
        if kind == "jpeg":
            self.device_decoded = self._decode_jpegs([(a, buf, img)])
        else:
            buf.copy_(torch.from_numpy(a), non_blocking=True)
            self.device_decoded = [False]
        return buf

    def upload_batch(self, images):
        """List of (H_i, W_i, 3) uint8 RGB host arrays or paths -> list of device views of the same images, one
        host-to-device copy of pixels per page.  All pages live in one device buffer, each at a 16-byte-aligned offset (the
        crop kernels stage such pages' rows by TMA); the buffer is kept per list of shapes, so a serving loop over batches
        of the same shapes reuses the same addresses and the page batch replays its CUDA graph.  JPEG files the device
        takes are decoded into their views by one ms_jpeg_decode_batch call (self.device_decoded: per page, True for
        those); every other source is read with read_image and copied."""
        torch = self.torch
        srcs = self._sources(images)
        key = tuple(shape[:2] for _, _, shape in srcs)
        entry = self._batch_buf.get(key)
        if entry is None:
            offs, total = [], 0
            for _, _, shape in srcs:
                offs.append(total)
                total += (int(np.prod(shape)) + 15) & ~15
            if len(self._batch_buf) >= 4:
                self._batch_buf.clear()
                self._tables.clear()
            buf = torch.empty((max(total, 16),), dtype=torch.uint8, device=self.device)
            views = [buf[o:o + int(np.prod(shape))].view(shape) for o, (_, _, shape) in zip(offs, srcs)]
            entry = self._batch_buf[key] = (buf, views)
        jobs, decoded = [], [False] * len(srcs)
        for i, (v, (kind, a, _)) in enumerate(zip(entry[1], srcs)):
            if kind == "jpeg":
                jobs.append((a, v, images[i]))
            else:
                v.copy_(torch.from_numpy(a), non_blocking=True)
        ok = iter(self._decode_jpegs(jobs))
        self.device_decoded = [next(ok) if kind == "jpeg" else False for kind, _, _ in srcs]
        return list(entry[1])

    def _page_tables(self, pages_dev):
        """(pointer table, (P, 2) int32 size table) on the device for a list of device images, kept per list"""
        torch = self.torch
        for pg in pages_dev:
            if not (pg.is_cuda and pg.dtype == torch.uint8 and pg.dim() == 3 and pg.shape[2] == 3 and pg.is_contiguous()):
                raise ValueError("pages must be contiguous (H, W, 3) uint8 CUDA tensors")
        sig = tuple((pg.data_ptr(), int(pg.shape[0]), int(pg.shape[1])) for pg in pages_dev)
        t = self._tables.get(sig)
        if t is None:
            if len(self._tables) >= 8:
                self._tables.clear()
            t = self._tables[sig] = (torch.tensor([v[0] for v in sig], dtype=torch.int64).to(self.device),
                                     torch.tensor([[v[1], v[2]] for v in sig], dtype=torch.int32).to(self.device))
        return t

    def network_inputs(self, pages_dev):
        """infer.py:301-305 for a list of P device images of their own sizes in one launch (ms_detector_input_batch):
        -> (P, 3, T, T) CUDA tensor of input_dtype, page i bit-identical to network_input(pages_dev[i]) (cast with
        .to(input_dtype)).  The tensor is owned by this detector and overwritten by its next call."""
        torch = self.torch
        T, P = self.target_size, len(pages_dev)
        if P == 0:
            raise ValueError("network_inputs needs at least one page")
        ptrs, hw = self._page_tables(pages_dev)
        shape = (P, 3, T, T)
        if self._inputs_buf is None or tuple(self._inputs_buf.shape) != shape or self._inputs_buf.dtype != self.input_dtype:
            self._inputs_buf = torch.empty(shape, dtype=self.input_dtype, device=self.device)
        r = self._runner
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            check(r.ctx.lib.ms_detector_input_batch(r.ctx.handle, ptrs.data_ptr(), hw.data_ptr(), P, T, T,
                                                    self._inputs_buf.data_ptr(), self._input_code, C.c_void_p(stream)))
        return self._inputs_buf

    def network_input(self, page_dev):
        """infer.py:301-305 on the device: (H, W, 3) u8 CUDA tensor -> (1, 3, T, T) of input_dtype, bit-identical to
        cv2.resize(img, (T, T)) -> ToTensor -> Normalize(0.5, 0.5) (cast with .to(input_dtype))."""
        torch = self.torch
        T = self.target_size
        if self.input_dtype != torch.float32:
            return self.network_inputs([page_dev])
        if self._input_buf is None or self._input_buf.shape[-1] != T:
            self._input_buf = torch.empty((1, 3, T, T), dtype=torch.float32, device=self.device)
        r = self._runner
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            check(r.ctx.lib.ms_detector_input(r.ctx.handle, page_dev.data_ptr(), int(page_dev.shape[0]),
                                              int(page_dev.shape[1]), T, T, self._input_buf.data_ptr(), None,
                                              C.c_void_p(stream)))
        return self._input_buf

    def _maps_as(self, score, geo, dtype):
        if dtype is None:
            return score, geo
        dtype = self.torch.float32 if dtype is _FLOAT32 else dtype
        return score.to(dtype), geo.to(dtype)

    def maps_from_device_page(self, page_dev, dtype=_FLOAT32):
        """Device image -> (score (1,H',W'), geometry (8,H',W')) CUDA tensors (infer.py:301-313 without the host), in
        float32 by default; dtype=None returns the network's own tensors as they are (their dtype and strides)."""
        if self.model is None:
            raise RuntimeError("EAST(model=...) is required for predict(): the detector network is outside this "
                               "package (use boxes_from_maps / predict_from_maps when the maps already exist)")
        with self.torch.no_grad():
            out = self.model(self.network_input(page_dev))
        return self._maps_as(out["score"][0], out["geometry"][0], dtype)

    def maps_from_device_pages(self, pages_dev, dtype=_FLOAT32):
        """List of P device images -> (score (P,1,H',W'), geometry (P,8,H',W')) CUDA tensors, float32 by default
        (dtype=None: the network's own tensors as they are): one network_inputs launch and one call of the network on
        the (P, 3, T, T) input."""
        if self.model is None:
            raise RuntimeError("EAST(model=...) is required for predict()")
        with self.torch.no_grad():
            out = self.model(self.network_inputs(pages_dev))
        return self._maps_as(out["score"], out["geometry"], dtype)

    def predict_from_maps(self, score_map, geo_map, orig_hw, sort_reading_order=False):
        words = words_from_boxes(self.boxes_from_maps(score_map, geo_map, orig_hw))
        if sort_reading_order and len(words) > 0:
            words = reorder_words(words)  # infer.py:366-385
        return Page(blocks=[Block(words=words)])

    def predict(self, img_or_path, vis=False, profile=False, return_maps=False, sort_reading_order=False):
        """Same contract as the reference's EAST.predict: dict with "page", "vis_image", "score_map", "geo_map".  A path
        is decoded by upload (on the device for the JPEG files it takes); vis=True downloads that page to draw on."""
        t0 = time.time()
        if _is_path(img_or_path):
            page_dev = self.upload(img_or_path)
            img = page_dev.cpu().numpy() if vis else page_dev
        else:
            img = read_image(img_or_path)
            page_dev = self.upload(img)
        score, geo = self.maps_from_device_page(page_dev, dtype=None)  # read in place by the post-processing
        if profile:
            self.torch.cuda.synchronize()
            print(f"  Model inference: {time.time() - t0:.3f}s")
        t0 = time.time()
        page = self.predict_from_maps(score, geo, tuple(img.shape[:2]), sort_reading_order=sort_reading_order)
        if profile:
            print(f"  Decode + NMS + box filters (device): {time.time() - t0:.3f}s")
            print(f"    Boxes after NMS: {sum(len(b.words) for b in page.blocks)}")
        return {
            "page": page,
            "vis_image": visualize_page(img, page, show_order=False) if vis else None,  # infer.py:390
            "score_map": score[0].float().cpu().numpy() if return_maps else None,
            "geo_map": geo.float().cpu().numpy() if return_maps else None,
        }
