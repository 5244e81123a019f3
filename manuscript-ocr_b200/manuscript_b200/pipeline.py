"""Pipeline with the reference's duck-typed detector / recogniser contract (reference _pipeline.py:18-202).

    detector.predict(image, vis=False, profile=...)  ->  {"page": Page, ...} | (Page, ...) | Page
    recognizer.predict(List[np.ndarray RGB u8])      ->  List[{"text", "confidence"}]  (or (text, conf) tuples)

Three routes through predict(), all with the reference's results:

* FUSED -- detector is this package's EAST and recogniser its TRBA: the page image is uploaded ONCE; the network
  input is made from it on the device, the maps stay on the device as the network returned them (float32, float16 or
  bfloat16, any strides), and one ms_page_batch_ragged_maps call (decode, LANMS, box filters, reading order, crop
  rectangles, resize-and-pad) writes the recogniser's batch, which the recogniser network reads in place.  Device -> host: the final boxes and the crop list (a few tens of kB), never pixels.
* DEVICE CROPS -- any detector, this package's TRBA: the page is uploaded once, reading order + crop rectangles + the
  crop batch are computed on the device from the detector's polygons.
* HOST CROPS -- a foreign recogniser gets the list of uint8 crops it expects (plain slices of the page image), in the
  reading order computed on the device.

process_batch on the fused route works on chunks of pages: one upload buffer, one detector-input launch, one network
call and one ms_page_batch_ragged call per chunk, and recogniser batches that span pages ("fused_batch").

rotated_crops=True (an extension) takes the same fused routes ("fused_rotated", "fused_batch_rotated") with
ms_page_batch_ragged_quads: the crop stage is the rectified patch of every final quad, and the crop list rows
[page, box, w, h, 0] name the words by their position in the page's reading order.

With this package's TRBA, the device routes (and rotated_crops) write the recogniser batch in the TRBA's batch_dtype
(float32 by default); a foreign recogniser still gets uint8 slices.
"""
import ctypes as C
import time
from pathlib import Path

import numpy as np

from . import ops
from ._cabi import batch_dtype_code, check
from .batch import PageBatch
from .east import EAST, kernel_maps, words_from_boxes
from .imaging import read_image, visualize_page
from .reading_order import reorder_words
from .trba import TRBA
from .types import Block, Page


def _page_of(det_out):
    """_pipeline.py:69-77: the three shapes a detector may answer in."""
    if isinstance(det_out, dict):
        page = det_out.get("page")
    elif isinstance(det_out, tuple):
        page = det_out[0]
    else:
        page = det_out
    if page is None:
        raise RuntimeError("Detector did not return a Page result.")
    return page


def _text_and_confidence(result):
    """_pipeline.py:152-159: dict, (text, confidence) tuple or anything printable."""
    if isinstance(result, dict):
        return result.get("text", ""), result.get("confidence", None)
    if isinstance(result, tuple) and len(result) == 2:
        return result
    return (str(result) if result is not None else ""), None


def host_crop_rects(boxes, img_h, img_w, min_text_size):
    """_pipeline.py:125-137 + 204-221 for (K, >=8) float boxes, vectorised: int32 truncation, size filter, clamped
    slice bounds with Python's slice semantics.  Returns (rects (K,4) int32 [x1,y1,x2,y2), valid (K,) bool).  Used to
    map the device's crop list back to words; the two are compared on every call."""
    b = np.asarray(boxes, dtype=np.float32)
    b = b.reshape(len(b), -1)[:, :8] if len(b) else np.zeros((0, 8), np.float32)
    poly = b.astype(np.int32)  # np.array(polygon, dtype=np.int32): truncation towards zero
    xs, ys = poly[:, 0::2], poly[:, 1::2]
    x_min, x_max, y_min, y_max = xs.min(1), xs.max(1), ys.min(1), ys.max(1)
    big = ((x_max - x_min) >= min_text_size) & ((y_max - y_min) >= min_text_size)
    x1, y1 = np.maximum(0, x_min), np.maximum(0, y_min)
    x2, y2 = np.minimum(img_w, x_max), np.minimum(img_h, y_max)

    def py_slice(a, b_, n):  # image[a:b] for a >= 0: a negative stop counts from the end
        b_ = np.where(b_ < 0, np.maximum(b_ + n, 0), b_)
        a = np.minimum(a, n)
        return a, np.maximum(b_, a)

    x1, x2 = py_slice(x1, x2, img_w)
    y1, y2 = py_slice(y1, y2, img_h)
    valid = big & (x2 > x1) & (y2 > y1)
    return np.stack([x1, y1, x2, y2], axis=1).astype(np.int32), valid


def host_patch_sizes(boxes):
    """The patch size of the rotated crop (quadcrop.cu quad_patch_size) for (K, >=8) float boxes: the longer of each
    pair of opposite edges in float64 from the float32 vertices, rounded half to even.  Returns (w, h, ok): ok is
    False where a coordinate is not finite, a side is above 32767 or below 2.  Used to check the device's quad crop
    list against the word boxes."""
    b = np.asarray(boxes, dtype=np.float32)
    q = (b.reshape(len(b), -1)[:, :8] if len(b) else np.zeros((0, 8), np.float32)).astype(np.float64)
    x, y = q[:, 0::2], q[:, 1::2]

    def edge(a, c):
        dx, dy = x[:, c] - x[:, a], y[:, c] - y[:, a]
        return np.sqrt(dx * dx + dy * dy)

    e01, e32, e03, e12 = edge(0, 1), edge(3, 2), edge(0, 3), edge(1, 2)
    ew, eh = np.where(e32 > e01, e32, e01), np.where(e12 > e03, e12, e03)
    ok = np.isfinite(e01) & np.isfinite(e32) & np.isfinite(e03) & np.isfinite(e12) & (ew <= 32767) & (eh <= 32767)
    w = np.rint(np.where(ok, ew, 0)).astype(np.int64)
    h = np.rint(np.where(ok, eh, 0)).astype(np.int64)
    return w, h, ok & (w >= 2) & (h >= 2)


_BATCH_CROPS_CAP0 = 8192  # first crop capacity of process_batch's page batch (grown to what a chunk needs)


class Pipeline:
    def __init__(self, detector=None, recognizer=None, min_text_size=5, rotated_crops=False):
        # _pipeline.py:52-54: missing parts are built from the released weights (EAST() / TRBA() in the reference);
        # offline that raises FileNotFoundError, as the reference's torch.load does
        self.detector = detector if detector is not None else EAST.from_pretrained()
        self.recognizer = recognizer if recognizer is not None else TRBA.from_pretrained()
        self.min_text_size = min_text_size
        # EXTENSION (SURVEY 8f-4, reference todo.md:1): rectify every word quad with a perspective warp instead of
        # cutting its bounding rectangle.  Off by default = the reference's behaviour.
        self.rotated_crops = bool(rotated_crops)
        self._runners = {}  # False: the one-page route's PageBatch, True: the batched route's, each with its key
        # "fused" | "fused_batch" | "fused_rotated" | "fused_batch_rotated" | "device_crops" | "host_crops" |
        # "rotated_crops" | "detect_only" (introspection for tests / bench)
        self.last_route = None

    # ---- route 1: everything between the image upload and the recogniser network on the device ---------------------
    def _fused_runner(self, batch=False):
        """The PageBatch of the one-page route, or (batch=True) of process_batch's: its crop buffer holds the chunk's
        crops (_BATCH_CROPS_CAP0 rows at first, grown to a power of two when a chunk needs more) instead of cap_boxes
        per page, and it keeps the buffers of at most two chunk sizes (the full chunk and the last one).  With
        rotated_crops its crop stage is the rectified quad crop, border constant 0 (the border of the per-image route)."""
        det, rec = self.detector, self.recognizer
        crops = "quads" if self.rotated_crops else "rects"
        key = (det.device, det.cap_boxes, rec.img_h, rec.img_w, int(self.min_text_size), rec.batch_dtype, crops)
        entry = self._runners.get(batch)
        if entry is None or entry[0] != key:
            kw = dict(crops_cap=_BATCH_CROPS_CAP0, max_buffer_sets=2) if batch else {}
            entry = self._runners[batch] = (key, PageBatch(
                device=det.device.index or 0, params=det._params(sort_reading_order=1),
                min_text_size=int(self.min_text_size), out_hw=(rec.img_h, rec.img_w), cap_boxes=det.cap_boxes,
                batch_dtype=rec.batch_dtype, crops=crops, border_mode=0, border_value=0, **kw))
        entry[1].params = det._params(sort_reading_order=1)
        return entry[1]

    @staticmethod
    def _host_boxes(res, n_pages):
        """Each page's final boxes as numpy (K_p, 9), from one device-to-host copy"""
        counts = res.box_counts.cpu().numpy()
        kmax = int(counts.max()) if n_pages else 0
        boxes = res.boxes[:n_pages, :kmax].cpu().numpy()         # D2H: P x K_max x 36 bytes
        return [boxes[p, :int(counts[p])] for p in range(n_pages)]

    def _predict_fused(self, img, profile, page_dev=None):
        """img: the page array, or (a path's route) its device copy, of which only the shape is read"""
        t0 = time.time()
        if page_dev is None:
            page_dev = self.detector.upload(img)                # the one H2D copy of pixels
        # network input + maps stay on the device, in the network's own dtype and layout
        score, geo = kernel_maps(*self.detector.maps_from_device_page(page_dev, dtype=None))
        res = self._fused_runner().run_ragged(score[None] if score.dim() == 2 else score, geo[None], [page_dev],
                                              sync=True, allow_order_overflow=True)
        return self._fused_pages(res, self._host_boxes(res, 1), [img], [page_dev], t0, profile)[0]

    def _predict_fused_batch(self, imgs, profile, pages_dev=None):
        """The fused route for a chunk of pages: one upload buffer, one detector-input launch, one network call, one
        page batch, and recogniser batches cut from the one crop batch.  imgs: page arrays, or where a page came from a
        file, its device copy (pages_dev given: the chunk is uploaded already), of which only the shape is read."""
        t0 = time.time()
        if pages_dev is None:
            pages_dev = self.detector.upload_batch(imgs)        # one H2D copy of pixels per page
        score, geo = kernel_maps(*self.detector.maps_from_device_pages(pages_dev, dtype=None))
        runner = self._fused_runner(batch=True)
        while True:
            res = runner.run_ragged(score, geo, pages_dev, sync=True, allow_order_overflow=True)
            boxes = self._host_boxes(res, len(imgs))
            if self.rotated_crops:  # a quad makes at most one crop (whether its system is singular is the device's call)
                need = sum(len(b) for b in boxes)
            else:
                need = sum(int(host_crop_rects(b, im.shape[0], im.shape[1], self.min_text_size)[1].sum())
                           for b, im in zip(boxes, imgs))
            if need <= runner.crops_cap:
                break
            # the crop list stopped at crops_cap: run the chunk again with room for all of its crops
            runner.crops_cap = 1 << (need - 1).bit_length()
        return self._fused_pages(res, boxes, imgs, pages_dev, t0, profile)

    def _fused_page(self, img, boxes, crops, overflow, page_dev, profile):
        """One page of a fused page batch: its final boxes (K, 9) and its rows of the crop list.  Returns the Page and
        its words that take the crops' texts, in crop order (None when the page was finished on the host)."""
        if overflow:
            # more boxes (or intersecting pairs) than the device reading-order kernel holds: the boxes came back in
            # detection order; order them with the host restatement and cut the crops from the uploaded page
            page = Page(blocks=[Block(words=words_from_boxes(boxes))])
            self.last_route = "fused+host_order"
            return self._finish_from_page(page, img, profile, page_dev=page_dev), None
        words = words_from_boxes(boxes)                         # already in reading order (_pipeline.py:105-123)
        page = Page(blocks=[Block(words=words)])
        rects, valid = host_crop_rects(boxes, img.shape[0], img.shape[1], self.min_text_size)
        if self.rotated_crops:
            # rows [page, box, w, h, 0]: boxes in increasing order, each with the patch size the host computes for it
            w, h, ok = host_patch_sizes(boxes)
            ok &= (w >= self.min_text_size) & (h >= self.min_text_size)
            b = crops[:, 1].astype(np.int64)
            if len(b) and (b[0] < 0 or b[-1] >= len(boxes) or np.any(np.diff(b) <= 0) or not ok[b].all()
                           or not np.array_equal(crops[:, 2], w[b]) or not np.array_equal(crops[:, 3], h[b])):
                raise RuntimeError("quad crop list of the device and the word boxes disagree")
            if not valid.any():  # the per-image route recognises nothing on a page without a crop rectangle
                return page, None
            return page, [words[j] for j in b.tolist()]
        if int(valid.sum()) != len(crops) or not np.array_equal(rects[valid], crops[:, 1:]):
            raise RuntimeError("crop list of the device and the word boxes disagree")
        return page, [words[j] for j in np.flatnonzero(valid).tolist()]

    def _fused_pages(self, res, boxes, imgs, pages_dev, t0, profile):
        """Pages of a fused page batch (res; boxes: each page's final boxes on the host), with the texts of the
        recogniser run over the crop batch in chunks of rec.batch_size, which may span pages."""
        rec = self.recognizer
        torch = rec.torch
        n = int(res.n_crops[0])
        crops = res.crops[:n].cpu().numpy()                     # D2H: n x 20 bytes
        overflow = set(res.order_overflow_pages().tolist())
        pages, targets, rows = [], [], []
        for p, img in enumerate(imgs):
            mine = np.flatnonzero(crops[:, 0] == p)              # the page's rows: the list is in (page, box) order
            page, words = self._fused_page(img, boxes[p], crops[mine], p in overflow, pages_dev[p], profile)
            pages.append(page)
            if words is not None:
                targets.extend(words)
                rows.append(mine)
        if profile:
            print(f"Detection + crops (device): {time.time() - t0:.3f}s")
        rows = np.concatenate(rows) if rows else np.zeros(0, np.int64)
        if len(rows):
            t0 = time.time()
            batch = res.batch[:n]                               # a view of the batch the crop kernel wrote
            if len(rows) != n:                                  # a page finished on the host left rows out
                batch = batch.index_select(0, torch.from_numpy(rows).to(batch.device))
            results = []
            for i in range(0, len(rows), rec.batch_size):       # recognizers/_trba/__init__.py:382: chunks of 32
                results.extend(rec.model(batch[i:i + rec.batch_size]))
            if profile:
                torch.cuda.synchronize()
                print(f"Recognition: {time.time() - t0:.3f}s")
            for word, result in zip(targets, results):
                text, conf = _text_and_confidence(result)
                d = word.__dict__  # Word has no validate_assignment (nor has the reference's): plain attribute writes
                d["text"], d["recognition_confidence"] = text, conf
                word.__pydantic_fields_set__.update(("text", "recognition_confidence"))
        return pages

    # ---- routes 2 and 3: a Page from any detector ---------------------------------------------------------------------
    def _ordered_crop_rects(self, page, img_h, img_w):
        """Reading order per block (_pipeline.py:105-123, mutates block.words like the reference), then the crop
        rectangle of every word that passes the size filter (_pipeline.py:125-137, 204-221)."""
        words, rects = [], []
        for block in page.blocks:
            block.words = reorder_words(block.words)
            if not block.words:
                continue
            polys = np.array([w.polygon for w in block.words], dtype=np.float32).reshape(len(block.words), -1)
            block_rects, valid = ops.word_rects(polys, img_h, img_w, self.min_text_size)
            for word, rect, ok in zip(block.words, block_rects, valid):
                if ok:
                    words.append(word)
                    rects.append(rect)
        return words, (np.stack(rects).astype(np.int32) if rects else np.zeros((0, 4), np.int32))

    def _recognise_rotated(self, image_array, words, page_dev=None):
        """rotated_crops=True: one rectified patch per word quad; words without a patch (smaller than min_text_size on
        a side, degenerate) are skipped like the reference skips small boxes.  Returns (kept words, results).
        page_dev: the page already on the device (RGB uint8), used instead of a second upload."""
        rec = self.recognizer
        # a page that came from a file exists only on the device (image_array is that copy): its shape is all that is read
        rgb = image_array if (page_dev is not None and image_array is page_dev) else TRBA._as_rgb(image_array)
        quads = np.array([w.polygon for w in words], dtype=np.float32).reshape(len(words), -1)[:, :8]
        if not isinstance(rec, TRBA):
            patches = [ops.warp_quad(rgb, q) for q in quads]
            keep = [i for i, p in enumerate(patches)
                    if p is not None and min(p.shape[:2]) >= self.min_text_size]
            return [words[i] for i in keep], rec.predict([patches[i] for i in keep])
        torch = rec.torch
        if page_dev is None:
            page_dev = torch.from_numpy(np.ascontiguousarray(rgb)).to(rec.device)
        quads_dev = torch.from_numpy(np.ascontiguousarray(quads)).to(rec.device)
        n = len(words)
        batch = torch.empty((n, 3, rec.img_h, rec.img_w), dtype=rec.batch_dtype, device=rec.device)
        sizes = torch.zeros((n, 2), dtype=torch.int32, device=rec.device)
        stream = torch.cuda.current_stream(rec.device).cuda_stream
        with torch.cuda.device(rec.device):
            check(rec.ctx.lib.ms_quad_crop_resize_pad_ex(
                rec.ctx.handle, page_dev.data_ptr(), 1, int(rgb.shape[0]), int(rgb.shape[1]), quads_dev.data_ptr(), 8,
                None, n, int(self.min_text_size), 0, 0, rec.img_h, rec.img_w, batch.data_ptr(),
                batch_dtype_code(rec.batch_dtype), None, sizes.data_ptr(), C.c_void_p(stream)))
        valid = (sizes[:, 0] > 0).cpu().numpy()
        keep = torch.from_numpy(np.flatnonzero(valid)).to(rec.device)
        kept_batch = batch.index_select(0, keep)
        results = []
        for i in range(0, len(kept_batch), rec.batch_size):
            results.extend(rec.predict_batch(kept_batch[i:i + rec.batch_size]))
        return [w for w, ok in zip(words, valid) if ok], results

    def _finish_from_page(self, page, image_array, profile, page_dev=None):
        """Routes 2 / 3 from a detector's Page: reading order, crop rectangles, recognition, text written back."""
        words, rects = self._ordered_crop_rects(page, *image_array.shape[:2])
        if words and self.rotated_crops:  # predict's rotated branch, cut from the uploaded page
            words, results = self._recognise_rotated(image_array, [w for b in page.blocks for w in b.words],
                                                     page_dev=page_dev)
            for word, result in zip(words, results):
                word.text, word.recognition_confidence = _text_and_confidence(result)
        elif words:
            results = self._recognise(image_array, rects, page_dev=page_dev)
            for word, result in zip(words, results):
                word.text, word.recognition_confidence = _text_and_confidence(result)
        return page

    def _recognise(self, image_array, rects, page_dev=None):
        rec = self.recognizer
        if not isinstance(rec, TRBA):
            self.last_route = "host_crops"
            return rec.predict([image_array[y1:y2, x1:x2] for x1, y1, x2, y2 in rects])
        # the page goes to the device once; every recogniser batch is cut from that copy and never visits the host
        if self.last_route != "fused+host_order":
            self.last_route = "device_crops"
        torch = rec.torch
        if page_dev is None:
            rgb = np.ascontiguousarray(TRBA._as_rgb(image_array))
            page_dev = torch.from_numpy(rgb).to(rec.device)
        crops = np.zeros((len(rects), 5), np.int32)
        crops[:, 1:] = rects
        batch = rec.crops_to_batch(page_dev, torch.from_numpy(crops).to(rec.device), len(rects))
        results = []
        for i in range(0, len(rects), rec.batch_size):
            results.extend(rec.predict_batch(batch[i:i + rec.batch_size]))
        return results

    # ---- the reference's public surface ---------------------------------------------------------------------------
    def _fused_ok(self, recognize_text):
        return (recognize_text and isinstance(self.detector, EAST)
                and isinstance(self.recognizer, TRBA) and self.detector.model is not None
                and self.recognizer.model is not None and self.detector.device == self.recognizer.device)

    @staticmethod
    def _is_rgb_u8(img):
        return isinstance(img, np.ndarray) and img.ndim == 3 and img.shape[2] == 3 and img.dtype == np.uint8

    def _fused_image_ok(self, img):
        """an image the fused route takes: uint8 RGB and, for rotated crops, at most 32767 pixels on a side (larger
        pages keep the per-image route, which raises)"""
        return self._is_rgb_u8(img) and (not self.rotated_crops or max(img.shape[:2]) <= 32767)

    def _fused_size_ok(self, page_dev):
        return not self.rotated_crops or max(page_dev.shape[:2]) <= 32767

    @staticmethod
    def _is_path(image):
        return isinstance(image, (str, Path))

    def predict(self, image, recognize_text=True, vis=False, profile=False):
        t_start = time.time()
        if self._fused_ok(recognize_text) and self._is_path(image):
            # a file: decoded into the detector's page buffer (on the device for the JPEG files it takes); no host array
            page_dev = self.detector.upload(image)
            if self._fused_size_ok(page_dev):
                self.last_route = "fused_rotated" if self.rotated_crops else "fused"
                page = self._predict_fused(page_dev, profile, page_dev=page_dev)
                if profile:
                    print(f"Pipeline total: {time.time() - t_start:.3f}s")
                if vis:  # _pipeline.py:166-174, drawn on the downloaded page
                    return page, visualize_page(page_dev.cpu().numpy(), page, show_order=True)
                return page
        elif self._fused_ok(recognize_text):
            img = read_image(image)
            if self._fused_image_ok(img):
                self.last_route = "fused_rotated" if self.rotated_crops else "fused"
                page = self._predict_fused(img, profile)
                if profile:
                    print(f"Pipeline total: {time.time() - t_start:.3f}s")
                if vis:  # _pipeline.py:166-174
                    return page, visualize_page(img, page, show_order=True)
                return page

        t0 = time.time()
        page = _page_of(self.detector.predict(image, vis=False, profile=profile))
        if profile:
            print(f"Detection: {time.time() - t0:.3f}s")
        if not recognize_text:
            self.last_route = "detect_only"
            if vis:  # _pipeline.py:81-87
                return page, visualize_page(read_image(image), page, show_order=False)
            return page

        image_array = read_image(image)
        t0 = time.time()
        words, rects = self._ordered_crop_rects(page, *image_array.shape[:2])
        if profile:
            print(f"Extract {len(words)} crops: {time.time() - t0:.3f}s")
        if words:
            t0 = time.time()
            if self.rotated_crops:
                self.last_route = "rotated_crops"
                words, results = self._recognise_rotated(image_array, [w for b in page.blocks for w in b.words])
            else:
                results = self._recognise(image_array, rects)
            if profile:
                print(f"Recognition: {time.time() - t0:.3f}s")
            for word, result in zip(words, results):
                word.text, word.recognition_confidence = _text_and_confidence(result)
        else:
            self.last_route = "no_crops"
        if profile:
            print(f"Pipeline total: {time.time() - t_start:.3f}s")
        if vis:  # _pipeline.py:166-174
            return page, visualize_page(image_array, page, show_order=True)
        return page

    def process_batch(self, images, recognize_text=True, vis=False, profile=False, max_pages=32):
        """_pipeline.py:178-191 (whose body calls a `self.process` that does not exist in the reference, so it can only
        raise AttributeError there): the evident intent, one predict per image, Pages only.

        On the fused route (this package's EAST and TRBA, recognize_text; "fused_batch_rotated" with rotated_crops,
        whose images must also be at most 32767 pixels on a side) with every image an
        (H, W, 3) uint8 RGB array, the images are processed in chunks of at most `max_pages` (which bounds the memory of
        the (P, 3, T, T) network input): one upload buffer, one detector-input launch, one detector network call and one
        page batch per chunk, and recogniser batches of rec.batch_size crops that may span pages (last_route
        "fused_batch").  The Pages are exactly [predict(img) for img in images] -- words, polygons, confidences and
        texts -- for a recogniser whose output for a row does not depend on the other rows of its batch (and a detector
        network that treats the rows of its input independently).  The images are read chunk by chunk; a chunk with an
        image that is not uint8 RGB, and every image off the fused route, runs predict per image.  The page batch of
        this route holds the crops the chunk needs (not cap_boxes per page) and the buffers of at most two chunk sizes."""
        max_pages = int(max_pages)
        if max_pages < 1:
            raise ValueError(f"max_pages must be at least 1, got {max_pages}")
        images = list(images)
        fused = self._fused_ok(recognize_text)
        results, routes = [], set()
        for i in range(0, len(images), max_pages):
            chunk = images[i:i + max_pages]
            if fused and any(self._is_path(im) for im in chunk):
                # files are decoded into the chunk's page buffer (JPEG on the device); only the arrays live on the host
                srcs = [im if self._is_path(im) else read_image(im) for im in chunk]
                if all(self._is_path(im) or self._fused_image_ok(im) for im in srcs):
                    pages_dev = self.detector.upload_batch(srcs)
                    if all(self._fused_size_ok(pg) for pg in pages_dev):
                        imgs = [pg if self._is_path(im) else im for im, pg in zip(srcs, pages_dev)]
                        results.extend(self._predict_fused_batch(imgs, profile, pages_dev=pages_dev))
                        routes.add("fused_batch")
                        continue
            imgs = [read_image(im) for im in chunk] if fused else None  # read chunk by chunk, not all at once
            if fused and all(self._fused_image_ok(im) for im in imgs):
                results.extend(self._predict_fused_batch(imgs, profile))
                routes.add("fused_batch")
                continue
            for img in chunk:
                res = self.predict(img, recognize_text=recognize_text, vis=vis, profile=profile)
                results.append(res[0] if vis else res)
                routes.add(self.last_route)
        if routes == {"fused_batch"}:
            self.last_route = "fused_batch_rotated" if self.rotated_crops else "fused_batch"
        return results

    def get_text(self, page):
        """_pipeline.py:193-202: one line per block, words left to right."""
        lines = []
        for block in page.blocks:
            texts = [w.text for w in sorted(block.words, key=lambda w: min(pt[0] for pt in w.polygon))
                     if getattr(w, "text", None)]
            if texts:
                lines.append(" ".join(texts))
        return "\n".join(lines)
