"""TRBA recogniser wrapper: batch assembly on the B200, the reference's predict() contract.

Mirrors `TRBA._preprocess_image` + the batching loop of `TRBA.predict` (reference
recognizers/_trba/__init__.py:264-288, 382-390) and `get_val_transform` / `ResizeAndPadA`
(recognizers/_trba/data/transforms.py:62-120, 185-193).  The recogniser network (SEResNet31 + BiLSTM +
attention) is outside the hot path and is supplied by the caller: `model(batch (n,3,h,w) f32 on the device)`
must return a list of {"text", "confidence"} dicts (or (text, confidence) tuples) of length n.

The batch is assembled on the device and stays there: a list of host crops is packed into one atlas, uploaded once,
and resampled by one launch of the crop kernels straight into the (n,3,h,w) float32 tensor the network reads -- where
the reference does one cv2.resize and one `.to(device)` per image (__init__.py:288).

batch_dtype=torch.float16 / torch.bfloat16 (an extension) makes the crop kernels write the batch in 16 bits: exactly
the float32 batch cast with `.to(batch_dtype)`, at half the bytes and without the cast.  It is for a network that runs
in that dtype; the caller owns the model's dtype (from_pretrained's reference network is float32 and stays so).
"""
import ctypes as C
import os
from pathlib import Path

import numpy as np

from ._cabi import Context, batch_dtype_code, check

DEFAULT_DIR = Path.home() / ".manuscript" / "trba" / "exp_1_baseline"  # recognizers/_trba/__init__.py:24-36


class TRBA:
    def __init__(self, model=None, img_h=64, img_w=256, device=0, batch_size=32, batch_dtype=None):
        # 64x256 is the reference class default (recognizers/_trba/__init__.py:150-151); configs/config.json
        # uses 32x128 -- both are supported
        import torch

        if not torch.cuda.is_available():
            raise RuntimeError("manuscript_b200.TRBA needs a CUDA device: there is no CPU fallback")
        self.torch = torch
        self.device = torch.device("cuda", int(device)) if not isinstance(device, torch.device) else device
        self.model = model
        self.img_h, self.img_w = int(img_h), int(img_w)
        self.batch_size = int(batch_size)
        self.batch_dtype = torch.float32 if batch_dtype is None else batch_dtype
        self._dtype_code = batch_dtype_code(self.batch_dtype)
        self._ctx = None

    @classmethod
    def from_pretrained(cls, model_path=None, config_path=None, **kwargs):
        """What the reference's `TRBA()` does (recognizers/_trba/__init__.py:120-168, 207-231): the released weights
        and config from ~/.manuscript/trba/exp_1_baseline/ (put there by the reference's downloader; this package has no
        network code) inside the reference's own TRBA, whose network then runs on the batches assembled here.
        FileNotFoundError when the checkpoint is missing, ImportError when the reference package is not installed.
        The reference network is float32: a batch_dtype other than torch.float32 needs a model converted by the
        caller."""
        weights = Path(model_path) if model_path is not None else DEFAULT_DIR / "weights.pth"
        if not weights.exists():
            raise FileNotFoundError(f"Model checkpoint not found: {weights} (the reference downloads it on first use; "
                                    "pass TRBA(model=...) or model_path=...)")
        from manuscript.recognizers import TRBA as ReferenceTRBA  # the network is outside this package

        ref = ReferenceTRBA(model_path=os.fspath(weights), config_path=config_path)
        rec = cls(model=None, img_h=ref.img_h, img_w=ref.img_w, **kwargs)

        # the reference's own loop (network call, token decode, confidence: __init__.py:391-432) runs on the rows of the
        # batch assembled here: its per-image preprocessing is replaced by "the row is already a network input"
        ref._preprocess_image = lambda row: row

        def run(batch, **kw):
            return ref.predict([batch[i:i + 1] for i in range(len(batch))], batch_size=max(1, len(batch)), **kw)

        rec.model = run
        return rec

    @property
    def ctx(self):
        if self._ctx is None:
            self._ctx = Context(self.device.index or 0)
        return self._ctx

    @staticmethod
    def _as_rgb(image):
        """recognizers/_trba/__init__.py:264-283: path / PIL / array -> (h, w, 3) uint8 RGB (grey -> RGB, RGBA -> RGB)."""
        if isinstance(image, str):
            import cv2

            if not os.path.exists(image):
                raise FileNotFoundError(f"Image file not found: {image}")
            bgr = cv2.imread(image)
            if bgr is None:
                raise ValueError(f"Cannot read image: {image}")
            return cv2.cvtColor(bgr, cv2.COLOR_BGR2RGB)
        if not isinstance(image, np.ndarray):
            if hasattr(image, "convert"):  # PIL
                return np.array(image.convert("RGB"))
            raise ValueError(f"Unsupported image type: {type(image)}")
        img = image
        if img.ndim == 2:
            img = np.repeat(img[:, :, None], 3, axis=2)
        elif img.shape[2] == 4:
            img = img[:, :, :3]
        if img.dtype != np.uint8:
            raise ValueError("TRBA expects uint8 images")
        return img

    def crops_to_batch(self, page_dev, crops_dev, n, out=None):
        """The device-resident step: page_dev (H, W, 3) or (P, H, W, 3) u8 CUDA tensor, crops_dev (>= n, 5) int32 CUDA
        rows [page, x1, y1, x2, y2) -> (n, 3, img_h, img_w) CUDA tensor of batch_dtype (ms_crop_resize_pad_ex;
        nothing touches the host)."""
        torch = self.torch
        if out is None:
            out = torch.empty((n, 3, self.img_h, self.img_w), dtype=self.batch_dtype, device=self.device)
        elif out.dtype != self.batch_dtype:
            raise ValueError(f"out is {out.dtype}, this TRBA writes {self.batch_dtype}")
        if n == 0:
            return out
        pages = page_dev if page_dev.dim() == 4 else page_dev[None]
        n_dev = torch.tensor([n], dtype=torch.int32, device=self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            check(self.ctx.lib.ms_crop_resize_pad_ex(self.ctx.handle, pages.data_ptr(), int(pages.shape[0]),
                                                     int(pages.shape[1]), int(pages.shape[2]), crops_dev.data_ptr(),
                                                     n_dev.data_ptr(), n, self.img_h, self.img_w, out.data_ptr(),
                                                     self._dtype_code, None, C.c_void_p(stream)))
        return out

    def preprocess(self, images):
        """List of (h,w,3) uint8 crops -> (n,3,img_h,img_w) CUDA tensor of batch_dtype: what the reference builds with
        one cv2.resize + .to(device) per image followed by torch.stack.  One upload (the packed atlas), one launch,
        no download."""
        torch = self.torch
        imgs = [self._as_rgb(im) for im in images]
        n = len(imgs)
        if n == 0:
            return torch.empty((0, 3, self.img_h, self.img_w), dtype=self.batch_dtype, device=self.device)
        # pack the crops into one atlas so that a single kernel launch resamples all of them
        wmax = max(im.shape[1] for im in imgs)
        htot = sum(im.shape[0] for im in imgs)
        atlas = np.zeros((htot, wmax, 3), np.uint8)
        crops = np.zeros((n, 5), np.int32)
        y = 0
        for i, im in enumerate(imgs):
            h, w = im.shape[:2]
            atlas[y:y + h, :w] = im
            crops[i] = (0, 0, y, w, y + h)
            y += h
        return self.crops_to_batch(torch.from_numpy(atlas).to(self.device), torch.from_numpy(crops).to(self.device), n)

    def predict(self, images, batch_size=None, **model_kwargs):
        if not isinstance(images, list):
            images = [images]
        if self.model is None:
            raise RuntimeError("TRBA(model=...) is required for predict(): the recogniser network is outside this package")
        bs = int(batch_size or self.batch_size)
        results = []
        for i in range(0, len(images), bs):  # recognizers/_trba/__init__.py:382
            batch = self.preprocess(images[i:i + bs])
            results.extend(self.predict_batch(batch, **model_kwargs))
        return results

    def predict_batch(self, batch, **model_kwargs):
        """batch (n,3,h,w) of batch_dtype on the device -> list of {"text", "confidence"}."""
        if self.model is None:
            raise RuntimeError("TRBA(model=...) is required")
        out = self.model(batch, **model_kwargs)
        res = []
        for r in out:
            if isinstance(r, dict):
                res.append({"text": r.get("text", ""), "confidence": r.get("confidence")})
            elif isinstance(r, tuple) and len(r) == 2:
                res.append({"text": r[0], "confidence": r[1]})
            else:
                res.append({"text": str(r) if r is not None else "", "confidence": None})
        return res
