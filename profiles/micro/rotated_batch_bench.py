"""Rotated-quad crops as the crop stage of the page batch:
    python profiles/micro/rotated_batch_bench.py [out.json]      (default profiles/rotated_batch_bench.json)

Arm A (wall clock, host included): Pipeline(EAST(axis_aligned_output=False), TRBA, rotated_crops=True).process_batch
over 64 seeded pages of 1700-3500 px on a side, on the fused route ("fused_batch_rotated") and on the per-image route
(forced by a detector wrapper that is not an EAST, so every page goes through EAST.predict + _recognise_rotated).  The
networks are bench.py's stubs: the detector replays one synthetic map pair from HBM, the recogniser returns constants.
Both routes must give the same Pages.

Arm B (device-resident, CUDA events, replayed graphs): one page batch over BASELINE configs[2] (64 x 2048^2, ~2000
words per page) with sort_reading_order=1 and axis_aligned_output=0, as ms_page_batch_quads (crops="quads") and as
ms_page_batch_ex (rectangles) on the same maps, plus the list and crop stages of each (ms_stage_timing: slot 3 is the
crop list -- word rectangles or quad list -- and slot 4 the crops, direct launches) and how the quads were served.

Arms alternate within each of ROUNDS rounds; medians and min / max are reported.  The GPU name and power limit are
read in the same run."""
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "manuscript-ocr_b200")]
import manuscript_b200 as mb  # noqa: E402
import synthdata  # noqa: E402

ROUNDS = 5
OUT_H, OUT_W = 32, 128


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def stats(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": xs}


class NotEAST:
    """a detector that is not this package's EAST: Pipeline takes the per-image route"""

    def __init__(self, det):
        self.det = det

    def predict(self, image, vis=False, profile=False):
        return self.det.predict(image, vis=vis, profile=profile)


def arm_a(dev):
    target = 1280
    score, geo, _ = synthdata.make_maps(7, target, 500)
    d_score = torch.from_numpy(score).to(dev)[None, None]
    d_geo = torch.from_numpy(geo).to(dev)[None]

    class Net:  # bench.py's stub detector: the same maps for every input row
        def __call__(self, x):
            n = x.shape[0]
            return {"score": d_score.expand(n, -1, -1, -1), "geometry": d_geo.expand(n, -1, -1, -1)}

    rng = np.random.default_rng(11)
    bases = [synthdata.make_page_image(900 + i, 3500) for i in range(4)]
    imgs = []
    for i in range(64):
        h, w = (int(v) for v in rng.integers(1700, 3501, 2))
        y, x = int(rng.integers(0, 3501 - h + 1)), int(rng.integers(0, 3501 - w + 1))
        imgs.append(np.ascontiguousarray(bases[i % 4][y:y + h, x:x + w]))

    def pipe(per_image):
        det = mb.EAST(model=Net(), target_size=target, axis_aligned_output=False)
        rec = mb.TRBA(model=lambda batch: [("w", 0.5)] * len(batch), img_h=OUT_H, img_w=OUT_W)
        return mb.Pipeline(detector=NotEAST(det) if per_image else det, recognizer=rec, rotated_crops=True)

    pipes = {"fused_batch_rotated": pipe(False), "per_image_rotated": pipe(True)}
    fields = {}
    for k, p in pipes.items():  # warm-up (buffers, graphs) and the check that both routes agree
        pages = p.process_batch(imgs)
        fields[k] = [[(w.polygon, w.detection_confidence, w.text) for w in b.words] for pg in pages for b in pg.blocks]
    assert pipes["fused_batch_rotated"].last_route == "fused_batch_rotated"
    same = fields["fused_batch_rotated"] == fields["per_image_rotated"]
    words = sum(len(b) for b in fields["fused_batch_rotated"])
    times = {k: [] for k in pipes}
    for _ in range(ROUNDS):
        for k, p in pipes.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            p.process_batch(imgs)
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
    out = {k: {"s_per_64_pages": stats(v), "pages_per_s": 64 / statistics.median(v)} for k, v in times.items()}
    out.update(pages_equal=bool(same), words=int(words), pages=64, target_size=target,
               page_sizes=[list(im.shape[:2]) for im in imgs][:8] + ["..."],
               speedup=statistics.median(times["per_image_rotated"]) / statistics.median(times["fused_batch_rotated"]))
    return out


def arm_b(dev):
    P, S, WORDS, steps = 64, 2048, 2000, 100
    score, geo, imgs = synthdata.make_batch(list(range(P)), S, WORDS)
    d_score, d_geo, d_pages = (torch.from_numpy(x).to(dev) for x in (score, geo, imgs))
    params = mb.EastParams.default(target_size=S, sort_reading_order=1, axis_aligned_output=0)
    kw = dict(device=0, params=params, cap_boxes=max(4096, 2 * WORDS), crops_cap=P * (WORDS + WORDS // 4 + 64),
              out_hw=(OUT_H, OUT_W))
    runners = {"quads": mb.PageBatch(crops="quads", **kw), "rects": mb.PageBatch(**kw)}
    res = {k: r.run(d_score, d_geo, d_pages, sync=True) for k, r in runners.items()}
    n = {k: int(r.n_crops.item()) for k, r in res.items()}
    qc = (C.c_int32 * 2)()
    mb._cabi.check(runners["quads"].ctx.lib.ms_quad_crop_last_counts(runners["quads"].ctx.handle, qc))
    same_boxes = torch.equal(res["quads"].box_counts, res["rects"].box_counts)
    stream = torch.cuda.current_stream()
    for r in runners.values():  # capture + replay
        for _ in range(3):
            r.run(d_score, d_geo, d_pages)
    torch.cuda.synchronize()

    def timed(r):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(steps):
            r.run(d_score, d_geo, d_pages)
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    step = {k: [] for k in runners}
    stage = {k: {"list": [], "crop": []} for k in runners}
    for _ in range(ROUNDS):
        for k, r in runners.items():
            step[k].append(timed(r))
        for k, r in runners.items():
            r.ctx.stage_timing(True)
            for _ in range(20):
                r.run(d_score, d_geo, d_pages)
            nb, st = r.ctx.stage_times()
            r.ctx.stage_timing(False)
            stage[k]["list"].append(st["word_rects"] / nb)
            stage[k]["crop"].append(st["crop"] / nb)
    out = {k: {"step_ms": stats(step[k]), "list_stage_ms": stats(stage[k]["list"]),
               "crop_stage_ms": stats(stage[k]["crop"]), "n_crops": n[k]} for k in runners}
    out["quads"]["staged"], out["quads"]["generic"] = int(qc[0]), int(qc[1])
    out["quads"]["crop_us_per_quad"] = 1e3 * statistics.median(stage["quads"]["crop"]) / max(1, n["quads"])
    out.update(boxes_equal=bool(same_boxes), pages=P, page=S, words_per_page=WORDS, steps_per_round=steps,
               note="BASELINE configs[2] with sort_reading_order=1, axis_aligned_output=0; the same device buffers every "
                    "step (working set in L2 between steps only in part: 64 pages are 805 MB)")
    return out


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "profiles", "rotated_batch_bench.json")
    if not torch.cuda.is_available():
        raise SystemExit("rotated_batch_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    result = {"gpu": gpu_identity(), "rounds": ROUNDS, "arm_b_page_batch": arm_b(dev),
              "arm_a_process_batch": arm_a(dev)}
    result["gpu_after"] = gpu_identity()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result)[:4000])


if __name__ == "__main__":
    main()
