"""The detector input of a stack of scans, one page per launch against one launch for all pages:
    python profiles/micro/detector_input_bench.py [out.json] [--parent-lib PATH]

Workload: 64 seeded ragged pages of scan sizes (sides drawn from 1700 to 3500 pixels, ~1.2 GB of source pixels, larger
than the 126 MB L2) resized to the default target_size T = 1280.  Kernel arms, alternated over three rounds, each timed
with CUDA events over STEPS steps of all 64 pages:
  single          64 one-page ms_detector_input calls (float32) with this library
  single_parent   the same with the library given by --parent-lib (the parent commit's build), selected with
                  MS_B200_LIB in a child process
  batch_f32       one ms_detector_input_batch call in float32
  batch_bf16      one ms_detector_input_batch call in bfloat16
Bytes are algorithmic, from shapes: per page the distinct source rows its y table names x 3 * w read, 3 * T * T * element
size written; the share is of the measured 6 557 GB/s copy peak (profiles/README.md).  Every arm's output is checked
equal to batch_f32 (bf16: equal to batch_f32.to(bfloat16)).
End to end: Pipeline.process_batch on the 64 pages against the loop [predict(img) for img], wall clock, with the stub
networks of bench.py's pipeline_predict_2048 (the detector replays one page's synthetic maps for every input row, the
recogniser returns constants), so the time is the path's, not a network's."""
import ctypes as C
import json
import os
import subprocess
import sys
import time
import zlib

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "manuscript-ocr_b200")]
import manuscript_b200 as mb  # noqa: E402
import synthdata  # noqa: E402

P, T, SIDE_LO, SIDE_HI, SEED = 64, 1280, 1700, 3500, 7
STEPS, ROUNDS = 20, 3
PEAK_GBS = 6557.0  # measured device-to-device copy peak of one B200 (profiles/README.md)


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def make_pages():
    rng = np.random.default_rng(SEED)
    shapes = [(int(rng.integers(SIDE_LO, SIDE_HI + 1)), int(rng.integers(SIDE_LO, SIDE_HI + 1))) for _ in range(P)]
    return [rng.integers(0, 256, (h, w, 3), dtype=np.uint8) for h, w in shapes]


def source_bytes(h, w):
    """distinct source rows the page's y table names (linear_entry_y, crop_common.cuh) x 3 * w"""
    scale = 1.0 / (T / h)
    fy = ((np.arange(T) + 0.5) * scale - 0.5).astype(np.float32)
    sy = np.floor(fy).astype(np.int64)
    rows = np.union1d(np.clip(sy, 0, h - 1), np.clip(sy + 1, 0, h - 1))
    return len(rows) * 3 * w


def timed(f, steps=STEPS):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        f()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


class Single:
    """64 one-page ms_detector_input calls into one (P, 3, T, T) float32 tensor.  The library is opened with plain ctypes
    and only the two entry points this arm calls are typed, so that a library without the batch entry point (the
    parent's) loads as well."""

    def __init__(self, imgs, lib_path):
        lib = C.CDLL(lib_path)
        lib.ms_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
        lib.ms_detector_input.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                          C.c_void_p, C.c_void_p]
        self.lib, self.handle = lib, C.c_void_p()
        assert lib.ms_create(0, C.byref(self.handle)) == 0
        self.pages = [torch.from_numpy(a).cuda() for a in imgs]
        self.out = torch.empty((P, 3, T, T), dtype=torch.float32, device="cuda")

    def __call__(self):
        s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        for i, pg in enumerate(self.pages):
            rc = self.lib.ms_detector_input(self.handle, pg.data_ptr(), int(pg.shape[0]), int(pg.shape[1]), T, T,
                                            self.out[i].data_ptr(), None, s)
            assert rc == 0, rc


def page_crcs(out):
    return [zlib.crc32(out[i].cpu().numpy().tobytes()) for i in range(out.shape[0])]


def child_single():
    """one round of the single-page arm with the library MS_B200_LIB names: prints {"ms", "crc"}"""
    lib_path = mb._cabi.library_path()
    arm = Single(make_pages(), lib_path)
    for _ in range(2):
        arm()
    ms = timed(arm)
    print(json.dumps({"ms": ms, "crc": page_crcs(arm.out), "lib": lib_path}))


def end_to_end(imgs):
    score, geo, _ = synthdata.make_maps(0, T, 500)
    d_score = torch.from_numpy(score).cuda()[None, None]
    d_geo = torch.from_numpy(geo).cuda()[None]

    class Net:
        def __call__(self, x):
            n = x.shape[0]
            return {"score": d_score.expand(n, -1, -1, -1), "geometry": d_geo.expand(n, -1, -1, -1)}

    det = mb.EAST(model=Net(), target_size=T)
    rec = mb.TRBA(model=lambda batch: [("w", 0.5)] * len(batch), img_h=32, img_w=128)
    pipe = mb.Pipeline(detector=det, recognizer=rec)
    arms = {"predict_loop": lambda: [pipe.predict(img) for img in imgs], "process_batch": lambda: pipe.process_batch(imgs)}
    out = {k: f() for k, f in arms.items()}  # warm-up (buffers, graph capture)
    same = all(len(a.blocks[0].words) == len(b.blocks[0].words) and
               [w.polygon for w in a.blocks[0].words] == [w.polygon for w in b.blocks[0].words]
               for a, b in zip(out["predict_loop"], out["process_batch"]))
    wall = {k: [] for k in arms}
    for _ in range(ROUNDS):
        for k, f in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            f()
            torch.cuda.synchronize()
            wall[k].append(1e3 * (time.perf_counter() - t0))
    words = sum(len(p.blocks[0].words) for p in out["process_batch"])
    return {"ms_rounds": wall, "ms_median": {k: float(np.median(v)) for k, v in wall.items()},
            "pages_per_s": {k: P / (float(np.median(v)) * 1e-3) for k, v in wall.items()}, "words": words,
            "same_pages": bool(same)}


def main():
    args = sys.argv[1:]
    if "--child-single" in args:
        return child_single()
    parent_lib = args[args.index("--parent-lib") + 1] if "--parent-lib" in args else None
    out_path = next((a for a in args if a.endswith(".json")), None)
    imgs = make_pages()
    src_bytes = sum(source_bytes(*a.shape[:2]) for a in imgs)
    single = Single(imgs, mb._cabi.library_path())
    det = mb.EAST(model=None, target_size=T)
    det_bf16 = mb.EAST(model=None, target_size=T, input_dtype=torch.bfloat16)
    views = det.upload_batch(imgs)
    arms = {"single": single, "batch_f32": lambda: det.network_inputs(views),
            "batch_bf16": lambda: det_bf16.network_inputs(views)}
    for f in arms.values():
        for _ in range(2):
            f()
    ref = det.network_inputs(views).clone()
    parity = {"single": torch.equal(single.out, ref),
              "batch_bf16": torch.equal(det_bf16.network_inputs(views).view(torch.int16),
                                        ref.to(torch.bfloat16).view(torch.int16))}
    ref_crc = page_crcs(ref)
    ms = {k: [] for k in list(arms) + (["single_parent"] if parent_lib else [])}
    for _ in range(ROUNDS):
        if parent_lib:
            env = dict(os.environ, MS_B200_LIB=os.path.abspath(parent_lib))
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child-single"], env=env,
                               capture_output=True, text=True)
            if r.returncode:
                sys.exit(r.stderr[-3000:])
            child = json.loads(r.stdout.strip().splitlines()[-1])
            ms["single_parent"].append(child["ms"])
            parity["single_parent"] = child["crc"] == ref_crc
        for k, f in arms.items():
            ms[k].append(timed(f))
    med = {k: float(np.median(v)) for k, v in ms.items()}
    written = {k: 3 * T * T * (2 if k == "batch_bf16" else 4) * P for k in ms}
    kern = {k: {"ms_rounds": ms[k], "ms_median": med[k], "alg_bytes": src_bytes + written[k],
                "alg_GBs": (src_bytes + written[k]) / med[k] / 1e6,
                "share_of_copy_peak": (src_bytes + written[k]) / med[k] / 1e6 / PEAK_GBS} for k in ms}
    del single, arms
    torch.cuda.empty_cache()
    res = {
        "gpu": gpu_identity(),
        "workload": f"{P} ragged pages, sides {SIDE_LO}..{SIDE_HI} (seed {SEED}), {sum(a.nbytes for a in imgs)} bytes of "
                    f"source pixels, target {T}x{T}",
        "steps_per_arm": STEPS, "rounds": ROUNDS,
        "parity_vs_batch_f32": {k: bool(v) for k, v in parity.items()},
        "source_bytes_read": src_bytes,
        "kernel": kern,
        "end_to_end": end_to_end(imgs),
        "copy_peak_GBs": PEAK_GBS,
    }
    text = json.dumps(res, indent=1)
    print(text)
    if out_path:
        with open(out_path, "w") as f:
            f.write(text + "\n")
    if not all(res["parity_vs_batch_f32"].values()) or not res["end_to_end"]["same_pages"]:
        sys.exit(1)


if __name__ == "__main__":
    main()
