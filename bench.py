#!/usr/bin/env python
"""bench.py -- pages/s of the EAST decode + LANMS + box filters + crop/resize/pad hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

A step = one pass of the hot path over one batch of synthetic pages PER GPU (pages are independent, so
ranks never exchange data: weak scaling, no collective on the data path; torch.distributed is used only
for the barrier and the max-over-ranks of the timings).  Exactly K steps are timed.  The inputs are generated from
fixed seeds, so runs with the same arguments compute on the same data; --dump-outputs DIR writes the results of the
last timed step there (dump_outputs) for comparing two builds output for output.

Workload (BASELINE.json configs[2]): 64 synthetic 2048x2048 pages per GPU, ~2000 word quads per page
(score map 512x512, geometry 8x512x512, page image 2048x2048x3 u8), TRBA 32x128 crop batch output.

One JSON line on rank 0:
  value    pages/s, inputs resident in HBM, device-timed (CUDA events on the launch stream), max over ranks
  e2e      pages/s through the C-ABI call with HOST buffers (pinned): H2D of maps+pages, the path, D2H of the
           boxes / counts / crop list, every step (the crop batch stays on the device for the recogniser, as
           the reference leaves it on `self.device`, recognizers/_trba/__init__.py:288)
  roofline the stage that dominates the step time, algorithmic bytes (SURVEY 8d) / its CUDA-event time
  stages   every stage: ms per step, algorithmic bytes, GB/s, fraction of the measured HBM peak
  cpu_baseline  the C oracle (a port of the reference's algorithm) on a bounded sample, 1 host thread
--impl reference: the CPU implementation (oracle port; the reference itself is numpy/numba/cv2 Python that
needs packages absent from this image) on all host threads, page-parallel, bounded sample per step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "manuscript-ocr_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

import synthdata  # noqa: E402

METRIC = "pages/sec (EAST decode+NMS+crop)"
OUT_H, OUT_W = 32, 128
FALLBACK_HBM_GBS = 6650.0


_REAL_STDOUT = None  # set when stdout's descriptor is redirected (multi-rank runs)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default: 250 for the b200 arm, a timed region of about 0.5 s at the default workload "
                         "(2.26 ms per step on one B200); 5 for the reference arm, whose steps take seconds on the host)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--pages", type=int, default=64, help="pages per GPU per step")
    ap.add_argument("--page-size", type=int, default=2048)
    ap.add_argument("--words", type=int, default=2000)
    ap.add_argument("--cpu-pages", type=int, default=8, help="pages in the bounded cpu_baseline sample")
    ap.add_argument("--corpus", type=int, default=1024, help="pages of the strong-scaling corpus run (BASELINE configs[4])")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-corpus", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle check of two pages of the step")
    ap.add_argument("--no-variants", action="store_true", help="skip the variant timings (reading order, rotated "
                                                               "crops, configs[1] / configs[3] shapes, Pipeline.predict)")
    ap.add_argument("--reading-order", action="store_true",
                    help="also run the reading-order sort between the box filters and the crops (what Pipeline.predict "
                         "does; not part of the BASELINE metric, reported under config.reading_order)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path returned in its last timed step (rank 0's pages) as DIR/<name>.npy, "
                         "so that two builds can be compared output for output: see dump_outputs()")
    a = ap.parse_args()
    if a.steps is None:
        a.steps = 250 if a.impl == "b200" else 5
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return a


BASELINE_SHAPES = {(1280, 500, 1): "configs[1]", (2048, 2000, 64): "configs[2]", (4096, 10000, None): "configs[3]"}


def workload_name(a):
    tag = BASELINE_SHAPES.get((a.page_size, a.words, a.pages)) or BASELINE_SHAPES.get((a.page_size, a.words, None))
    return (f"{a.pages}x{a.page_size}x{a.page_size} synthetic pages per GPU, ~{a.words} quads/page, "
            f"TRBA {OUT_H}x{OUT_W} crop batch ({'BASELINE ' + tag if tag else 'not a BASELINE shape'})")


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---- CPU side: the oracle chain for one page (test infrastructure used as the reported baseline) ------------------
def cpu_page(score, geo, img, page):
    from oracle import cpu

    quads = cpu.decode_quads_from_maps(score, geo, 0.6, 4.0, 2)
    nms = cpu.locality_aware_nms(quads, 0.2)
    boxes = cpu.east_postprocess(nms, (page, page), target_size=page)
    rects, valid = cpu.word_rects(boxes, page, page, 5)
    n = 0
    for r in rects[valid]:
        cpu.crop_resize_pad(img, r, OUT_H, OUT_W)
        n += 1
    return len(boxes), n


def cpu_baseline(a, n_pages, threads):
    """pages/s of the oracle on `n_pages` pages of the workload, `threads` host threads (page-parallel;
    the C oracle is called through ctypes, which releases the GIL)."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import cpu

    cpu.lib()
    data = [(synthdata.make_maps(10_000 + i, a.page_size, a.words)[:2], synthdata.make_page_image(10_000 + i, a.page_size))
            for i in range(n_pages)]

    def one(i):
        (s, g), img = data[i]
        return cpu_page(s, g, img, a.page_size)

    t0 = time.perf_counter()
    if threads <= 1:
        res = [one(i) for i in range(n_pages)]
    else:
        with ThreadPoolExecutor(threads) as ex:
            res = list(ex.map(one, range(n_pages)))
    dt = time.perf_counter() - t0
    return n_pages / dt, sum(r[0] for r in res), dt


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    threads = max(1, cores)
    per_step = max(2, min(a.pages, threads))
    for _ in range(max(0, min(a.warmup, 1))):
        cpu_baseline(a, min(2, per_step), threads)
    times, boxes = [], 0
    for _ in range(a.steps):
        pps, nb, dt = cpu_baseline(a, per_step, threads)
        times.append(dt)
        boxes += nb
    total = sum(times)
    value = per_step * a.steps / total
    sample = (f"{per_step} pages per step of the same synthetic workload, C oracle port page-parallel over "
              f"{threads} host threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "pages/s", "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * total / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64 (NMS) / f32 (boxes) / u8 (crops)", "data": "synthetic",
        "config": {"workload": workload_name(a), "sample": sample},
        "boxes_per_sec": boxes / total,
        "cpu_baseline": {"value": value, "unit": "pages/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "pages/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), file=_REAL_STDOUT or sys.stdout, flush=True)


# ---- clocks ----------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            if t < t0 or t > t1 + 0.2:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- the B200 arm ------------------------------------------------------------------------------------------------------
def parity_check(a, score_np, geo_np, imgs_np, res, pages=(0, 1), every=50):
    """Outside every timed region: pages `pages` of the step against the oracle chain -- final boxes and crop rectangles
    in full, one crop in `every` of the float32 batch -- bit for bit.  Returns a summary for the JSON line."""
    from oracle import cpu

    S = a.page_size
    counts = res.box_counts.cpu().numpy()
    n_crops = int(res.n_crops.cpu()[0])
    crops = res.crops[:n_crops].cpu().numpy()
    checked_boxes = checked_crops = 0
    for p in pages:
        if p >= len(counts):
            continue
        quads = cpu.decode_quads_from_maps(score_np[p], geo_np[p], 0.6, 4.0, 2)
        want = cpu.east_postprocess(cpu.locality_aware_nms(quads, 0.2), (S, S), target_size=S)
        if a.reading_order:
            import manuscript_b200 as mb

            want = want[mb.word_reading_order(want[:, :8])]
        got = res.boxes[p, : counts[p]].cpu().numpy()
        assert got.shape == want.shape and np.array_equal(got, want), f"page {p}: boxes differ from the oracle"
        rects, valid = cpu.word_rects(want, S, S, 5)
        rows = np.flatnonzero(crops[:, 0] == p)
        assert np.array_equal(crops[rows, 1:], rects[valid]), f"page {p}: crop rectangles differ from the oracle"
        for j in rows[::every]:
            chw = cpu.crop_resize_pad(imgs_np[p], crops[j, 1:], OUT_H, OUT_W)[1]
            assert np.array_equal(res.batch[int(j)].cpu().numpy(), chw), f"page {p}: crop {j} differs from the oracle"
            checked_crops += 1
        checked_boxes += len(want)
    return {"pages": list(pages), "boxes": int(checked_boxes), "crops": int(checked_crops),
            "against": "oracle/oracle.c chain (pinned to the reference's goldens), bit-exact"}


DUMP_BYTES = 64 << 20
DUMP_CROPS = 512


def dump_outputs(out_dir, res):
    """Write the results of one ms_page_batch step as <out_dir>/<name>.npy, float32 / float64 only, at most DUMP_BYTES in
    all: every page's final boxes (rows concatenated in page order), box counts, flags and the crop list in full, a float64
    sum of every crop of the float32 batch, and DUMP_CROPS crops of the batch chosen by a fixed seed (with their indices).
    The inputs are seeded, so two builds run with the same arguments can be compared file by file."""
    import torch

    counts = res.box_counts.cpu().numpy()
    boxes = res.boxes.cpu().numpy()
    n_crops = int(res.n_crops.cpu()[0])
    batch = res.batch[:n_crops]
    out = {
        "boxes": np.concatenate([boxes[p, : counts[p]] for p in range(len(counts))]),
        "box_counts": counts.astype(np.float64),
        "flags": res.flags.cpu().numpy().astype(np.float64),
        "crops": res.crops[:n_crops].cpu().numpy().astype(np.float64),
        "batch_crop_sums": torch.sum(batch, dim=(1, 2, 3), dtype=torch.float64).cpu().numpy(),
    }
    crop_bytes = batch[0].numel() * 4 if n_crops else 0
    room = DUMP_BYTES - sum(v.nbytes for v in out.values())
    if room < 0:
        raise SystemExit(f"bench.py: the outputs of this workload exceed {DUMP_BYTES >> 20} MB; use fewer --pages")
    k = min(n_crops, DUMP_CROPS, room // (crop_bytes + 8) if crop_bytes else 0)
    idx = np.sort(np.random.default_rng(0).choice(n_crops, k, replace=False))
    out["batch_sample_index"] = idx.astype(np.float64)
    out["batch_sample"] = batch[torch.from_numpy(idx).to(batch.device)].cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)
    return {"dir": out_dir, "files": sorted(out), "bytes": int(sum(v.nbytes for v in out.values()))}


def run_b200(a):
    import torch

    import manuscript_b200 as mb

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 arm has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # one process per GPU: stay on the cores (and NUMA node) next to this GPU before pinning host memory; when the
    # container's CPU set hides the GPU's socket, at least ask for the memory to be placed there
    from manuscript_b200.sharding import bind_to_gpu_cpus, gather_boxes_via_shm, prefer_numa_node_of_gpu, shard_pages

    cpus = bind_to_gpu_cpus(local)
    numa_node = prefer_numa_node_of_gpu(local)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        # stdout carries ONE JSON line: whatever libraries print to file descriptor 1 from here on (NCCL's version
        # banner at communicator creation) goes to stderr; rank 0 writes the line to the real stdout at the end
        global _REAL_STDOUT
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    # results are gathered on the HOST (BASELINE configs[4]): a gloo group carries the pickled per-page results, the
    # NCCL group only the barriers and the reductions of the timings
    host_group = dist.new_group(backend="gloo") if dist is not None else None

    def barrier():
        if dist is not None:
            dist.barrier()

    def reduce_ranks(x, op):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=op)
        return float(t[0])

    def max_over_ranks(x):
        return reduce_ranks(x, dist.ReduceOp.MAX) if dist is not None else x

    def sum_over_ranks(x):
        return reduce_ranks(x, dist.ReduceOp.SUM) if dist is not None else x

    P, S = a.pages, a.page_size
    seeds = [rank * P + i for i in range(P)]  # this rank's shard of the corpus: pages [rank*P, (rank+1)*P)
    score_np, geo_np, imgs_np = synthdata.make_batch(seeds, S, a.words)
    M = S // 4
    pin = dict(pin_memory=True)
    h_score = torch.empty((P, M, M), dtype=torch.float32, **pin)
    h_geo = torch.empty((P, 8, M, M), dtype=torch.float32, **pin)
    h_pages = torch.empty((P, S, S, 3), dtype=torch.uint8, **pin)
    h_score.copy_(torch.from_numpy(score_np))
    h_geo.copy_(torch.from_numpy(geo_np))
    h_pages.copy_(torch.from_numpy(imgs_np))
    d_score, d_geo, d_pages = h_score.to(dev), h_geo.to(dev), h_pages.to(dev)

    params = mb.EastParams.default(target_size=S, sort_reading_order=1 if a.reading_order else 0)
    cap_boxes = max(4096, 2 * a.words)
    crops_cap = P * (a.words + a.words // 4 + 64)
    runner = mb.PageBatch(device=local, params=params, cap_boxes=cap_boxes, crops_cap=crops_cap, out_hw=(OUT_H, OUT_W))
    ctx = runner.ctx
    stream = torch.cuda.current_stream()

    # warm-up (also sizes the scratch arenas)
    W = max(a.warmup, 3)
    for _ in range(W):
        res = runner.run(d_score, d_geo, d_pages)
    torch.cuda.synchronize()
    res.raise_for_flags()

    # parity of THIS step's results with the oracle, before anything is timed
    parity = None
    if rank == 0 and not a.no_parity:
        # the first and the last page: one from each of the two concurrent halves of the batch's front stages
        parity = parity_check(a, score_np, geo_np, imgs_np, res, pages=(0, P - 1) if P > 1 else (0,))

    # per-page work counts for the algorithmic-byte model (outside the timed region)
    counts = res.box_counts.cpu().numpy().astype(np.int64)
    n_crops = int(res.n_crops.item())
    crops = res.crops[:n_crops].cpu().numpy().astype(np.int64)
    src_px = int(((crops[:, 3] - crops[:, 1]) * (crops[:, 4] - crops[:, 2])).sum())
    cand = torch.empty((P, (M // 2) * (M // 2), 9), dtype=torch.float32, device=dev)
    ccnt = torch.zeros((P,), dtype=torch.int32, device=dev)
    cflg = torch.zeros((P,), dtype=torch.int32, device=dev)
    mb._cabi.check(ctx.lib.ms_decode_quads(ctx.handle, d_score.data_ptr(), d_geo.data_ptr(), P, M, M, 0.6, 4.0, 2,
                                           cand.data_ptr(), cand.shape[1], ccnt.data_ptr(), cflg.data_ptr(),
                                           torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    n_cand = int(ccnt.sum().item())
    # NMS output count == boxes before the filters; the filters only drop boxes, so use the NMS count from lanms
    nms_out = torch.empty_like(cand)
    ncnt = torch.zeros((P,), dtype=torch.int32, device=dev)
    mb._cabi.check(ctx.lib.ms_lanms(ctx.handle, cand.data_ptr(), ccnt.data_ptr(), P, cand.shape[1], 0.2,
                                    nms_out.data_ptr(), ncnt.data_ptr(), cflg.data_ptr(),
                                    torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    n_nms = int(ncnt.sum().item())
    del cand, nms_out
    n_boxes = int(counts.sum())

    alg = {  # bytes per step on this GPU (SURVEY 8d)
        "decode": 4 * M * M * P + 72 * n_cand,
        "lanms": 36 * n_cand + 36 * n_nms,
        "east_boxes": 36 * n_nms + 36 * n_boxes,
        "word_rects": 36 * n_boxes + 20 * n_crops,
        "crop": 3 * src_px + 3 * OUT_H * OUT_W * 4 * n_crops,
    }

    # ---- timed region 1: inputs resident in HBM, device-timed: K steps -----------------------------------------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    # The call a serving loop makes: ms_page_batch on persistent buffers, which the library replays as a CUDA graph from
    # its second occurrence on.  The counting calls above may have grown the scratch arena (a grown arena drops the
    # recorded graph), so the call is recorded and captured again here, outside the timed region.
    for _ in range(3):
        runner.run(d_score, d_geo, d_pages)
    torch.cuda.synchronize()
    launches0 = ctx.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_timed = a.steps
    barrier()
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    ev0.record(stream)
    for _ in range(n_timed):
        last = runner.run(d_score, d_geo, d_pages)
    ev1.record(stream)
    torch.cuda.synchronize()
    barrier()
    ms_total = max_over_ranks(ev0.elapsed_time(ev1))
    launches = ctx.launches - launches0  # per K steps
    # the runner's output buffers are overwritten by the next pass: write the last timed step's results now
    dumped = dump_outputs(a.dump_outputs, last.raise_for_flags()) if a.dump_outputs and rank == 0 else None
    # ---- the same steps once more with the library's stage events (CUDA events between the stages on the launch
    # stream): per-stage times and the dominant kernel's duration.  Events between the stages need direct launches
    # instead of the graph replay, so this pass is a few per cent slower than the one above and is reported beside it.
    n_staged = min(n_timed, 256)                    # the library keeps the events of at most 256 batches
    ctx.stage_timing(True)
    ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    torch.cuda.synchronize()
    ev2.record(stream)
    for _ in range(n_staged):
        runner.run(d_score, d_geo, d_pages)
    ev3.record(stream)
    torch.cuda.synchronize()
    barrier()
    ms_staged = max_over_ranks(ev2.elapsed_time(ev3)) / n_staged
    nb, stage_ms = ctx.stage_times()
    ctx.stage_timing(False)
    assert nb == n_staged, (nb, n_staged)

    # ---- timed region 2: end to end through the host-buffer C-ABI call -------------------------------------------
    e2e = None
    if not a.no_e2e:
        for _ in range(2):
            runner.run_host(h_score, h_geo, h_pages)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            rh = runner.run_host(h_score, h_geo, h_pages)
        torch.cuda.synchronize()
        t_e2e = max_over_ranks(time.perf_counter() - t0)
        barrier()
        nch = int(rh.n_crops[0])
        assert nch == n_crops and int(rh.box_counts.sum()) == n_boxes
        # Geometry: the pinned host tensor is not uploaded -- the decode kernel gathers the candidate cells straight from
        # it over PCIe (zero copy).  Counted as one 32-byte sector per candidate and plane, an upper bound (neighbouring
        # candidates share sectors).  MS_B200_NO_ZEROCOPY=1 uploads the rows a quantised decode can read instead.
        if os.environ.get("MS_B200_NO_ZEROCOPY"):
            geo_rows = M // 2 if (params.quantization == 2 and M % 2 == 0) else M
            geo_bytes, geo_how = P * 8 * geo_rows * M * 4, "geometry rows uploaded (strided DMA)"
        else:
            geo_bytes, geo_how = n_cand * 8 * 32, "geometry gathered from pinned host memory by the decode kernel (zero copy)"
        h2d = h_score.numel() * 4 + geo_bytes + h_pages.numel()
        d2h = P * int(counts.max()) * 36 + P * 8 + 4 + nch * 20
        e2e = {"value": world * P * a.steps / t_e2e, "unit": "pages/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": int(d2h), "ms_per_step": 1e3 * t_e2e / a.steps,
               "note": "ms_page_batch_host with pinned host buffers; " + geo_how +
                       "; crop batch left on the device for the recogniser"}
        # what the box can move: the same bytes as plain pinned cudaMemcpyAsync copies, all ranks at once
        h2d_dst = torch.empty_like(d_pages)
        sc_dst = torch.empty_like(d_score)
        for _ in range(2):
            h2d_dst.copy_(h_pages, non_blocking=True)
            sc_dst.copy_(h_score, non_blocking=True)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        reps_c = max(2, a.steps // 2)
        for _ in range(reps_c):
            h2d_dst.copy_(h_pages, non_blocking=True)
            sc_dst.copy_(h_score, non_blocking=True)
        torch.cuda.synchronize()
        t_c = max_over_ranks(time.perf_counter() - t0)
        barrier()
        # the same bytes in the entry point's own pattern (chunks of P / 8 pages, score + pages of a chunk in turn): on
        # boxes where several GPUs share a PCIe switch the ranks' transfers interleave differently; the faster of the
        # two patterns is the reference
        step_c = max(1, (P + 7) // 8)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps_c):
            for c0 in range(0, P, step_c):
                sc_dst[c0:c0 + step_c].copy_(h_score[c0:c0 + step_c], non_blocking=True)
                h2d_dst[c0:c0 + step_c].copy_(h_pages[c0:c0 + step_c], non_blocking=True)
        torch.cuda.synchronize()
        t_c2 = max_over_ranks(time.perf_counter() - t0)
        barrier()
        t_c = min(t_c, t_c2)
        copy_bytes = h_pages.numel() + h_score.numel() * 4
        ceil_pps = world * P * reps_c / t_c
        e2e["h2d_ceiling"] = {"pages_per_s": ceil_pps, "gbs_per_gpu": copy_bytes * reps_c / t_c / 1e9,
                              "frac_of_ceiling": e2e["value"] / ceil_pps,
                              "note": "page images + score maps of one step as plain pinned cudaMemcpyAsync copies (whole "
                                      "tensors, and in the entry point's chunks; the faster of the two), every rank at "
                                      "once, nothing else running: the host-to-device reference of this box at this N"}
        del h2d_dst, sc_dst
        # the deployment SURVEY 8f-3 describes: the detector ran on this GPU, its maps are already in HBM and only the
        # page images cross PCIe (same entry point: device pointers for the maps are used in place)
        for _ in range(2):
            runner.run_host(d_score, d_geo, h_pages)
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            rm = runner.run_host(d_score, d_geo, h_pages)
        torch.cuda.synchronize()
        t_m = max_over_ranks(time.perf_counter() - t0)
        barrier()
        assert int(rm.n_crops[0]) == n_crops
        e2e["maps_on_device"] = {"value": world * P * a.steps / t_m, "unit": "pages/s",
                                 "ms_per_step": 1e3 * t_m / a.steps,
                                 "h2d_bytes_per_step": int(h_pages.numel()), "d2h_bytes_per_step": int(d2h),
                                 "frac_of_ceiling": (world * P * a.steps / t_m) /
                                                    (world * P * reps_c / t_c * copy_bytes / h_pages.numel())}

    # ---- BASELINE configs[4]: a fixed corpus strong-scaled over the ranks, results gathered on rank 0's host ---------
    corpus = None
    if not a.no_e2e and not a.no_corpus and a.corpus >= world:
        mine = shard_pages(a.corpus, world, rank)  # contiguous page range of this rank
        n_mine = len(mine)

        def corpus_pass():
            cnts, rows = [], []
            for c0 in range(0, n_mine, P):
                n = min(P, n_mine - c0)
                r = runner.run_host(h_score[:n], h_geo[:n], h_pages[:n])
                cnt = r.box_counts[:n].copy()
                cnts.append(cnt)
                rows.extend(r.boxes[i, : cnt[i]].copy() for i in range(n))
            return np.concatenate(cnts), np.concatenate(rows)

        corpus_pass()
        gather_boxes_via_shm(np.zeros(1, np.int32), np.zeros((1, 9), np.float32), group=host_group)  # connections up
        barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        local_cnt, local_rows = corpus_pass()
        gathered = gather_boxes_via_shm(local_cnt, local_rows, group=host_group)
        t_corpus = max_over_ranks(time.perf_counter() - t0)
        barrier()
        if rank == 0:
            g_cnt, g_rows = gathered
            assert len(g_cnt) == a.corpus and len(g_rows) == int(g_cnt.sum()), "gathered corpus is incomplete"
            assert np.array_equal(g_rows[: int(g_cnt[0])], local_rows[: int(local_cnt[0])])
            corpus = {"pages": a.corpus, "pages_per_s": a.corpus / t_corpus, "seconds": t_corpus, "scaling": "strong",
                      "boxes_gathered": int(len(g_rows)),
                      "note": f"BASELINE configs[4]: {a.corpus} page instances (this rank's {P} synthetic pages, cycled) "
                              f"page-sharded over {world} GPU(s) by shard_pages, every chunk of {P} pages through "
                              "ms_page_batch_host from pinned host memory, every page's boxes gathered on rank 0's host "
                              "(POSIX shared memory between the ranks of the box, sizes and barriers over a gloo group) inside the timed region; crop batches stay on their GPU "
                              "for the recogniser"}
    t_wall2 = time.perf_counter()
    if rank == 0:
        sampler.stop()

    # ---- variants (not the BASELINE metric; N = 1 only, outside both timed regions' clocks) ------------------------
    variants = None
    if world == 1 and not a.no_variants:
        variants = run_variants(a, mb, torch, dev, local, ctx, res, counts, d_score, d_geo, d_pages, h_pages, imgs_np,
                                cap_boxes, crops_cap, stream)

    total_boxes = sum_over_ranks(float(n_boxes))
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return

    peak, peak_src = measured_peak()
    ms_step = ms_total / n_timed
    stages = {}
    for k, v in stage_ms.items():
        ms = v / nb
        gbs = alg[k] / (ms * 1e-3) / 1e9 if ms > 0 else 0.0
        stages[k] = {"ms_per_step": ms, "share": v / max(sum(stage_ms.values()), 1e-12), "alg_bytes": int(alg[k]),
                     "gbs": gbs, "frac_of_hbm_peak": gbs / peak}
    dom = max(stage_ms, key=lambda k: stage_ms[k])
    traffic, traffic_src = None, None
    try:  # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel from the committed ncu --set full capture
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        if tj.get("stage") == dom and tj.get("workload_pages") == P and tj.get("page") == S:
            traffic, traffic_src = tj["dram_bytes_per_launch"], tj["source"]
    except Exception:
        pass
    roofline = {"kernel": dom, "bound": "hbm", "achieved": stages[dom]["gbs"], "peak": peak, "unit": "GB/s",
                "frac": stages[dom]["gbs"] / peak, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": peak_src,
                "alg_bytes_per_launch": int(alg[dom]), "ms_per_launch": stages[dom]["ms_per_step"]}
    whole = sum(alg.values()) / (ms_step * 1e-3) / 1e9
    line = {
        "metric": METRIC, "value": world * P * n_timed / (ms_total * 1e-3), "unit": "pages/s", "n_gpus": world,
        "steps": a.steps, "warmup": W, "ms_per_step": ms_step, "higher_is_better": True,
        "timed_region_ms": ms_total,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64 (NMS) / f32 (boxes) / u8 (crops)", "data": "synthetic",
        "config": {"workload": workload_name(a), "pages_per_gpu": P, "page": S, "map": M, "words_per_page": a.words,
                   "candidates_per_page": n_cand / P, "boxes_per_page": n_boxes / P, "crops_per_page": n_crops / P,
                   "candidates_note": "synthdata scales every word to its grid cell (87 % x 68 % of it: 44 x 28 px at this "
                                      "density) and shrinks the score region by 0.3 of the shorter side like "
                                      "dataset.py:180-199, which leaves ~7.5 quantisation cells per word; SURVEY 8d's "
                                      "probe (~12 per word, 24k per page) used larger words -- variants.dense_candidates "
                                      "times that load",
                   "l2": "inputs (maps + pages) of one step exceed L2 (no flush needed)",
                   "timing": f"the {a.steps} timed steps run back to back inside one CUDA-event bracket; ms_per_step is "
                             "their mean; the repeated call is replayed as a CUDA graph by the library (MS_B200_NO_GRAPHS=1: "
                             "direct launches)",
                   "reading_order": bool(a.reading_order), "host_cpus_rank0": (len(cpus) if cpus else None),
                   "numa_node_rank0": numa_node,
                   "parallelism": f"pages sharded over {world} GPU(s), no collective"},
        "boxes_per_sec": total_boxes * n_timed / (ms_total * 1e-3),
        "gpu_launches": int(round(launches)),
        "parity_checked": parity is not None, "parity": parity,
        "roofline": roofline,
        "whole_step": {"alg_bytes": int(sum(alg.values())), "gbs": whole, "frac_of_hbm_peak": whole / peak},
        "stages": stages,
        "stage_pass": {"ms_per_step": ms_staged, "steps": int(nb),
                       "note": "`stages`, `roofline.ms_per_launch` and the shares come from a second pass of the same steps, "
                               "run right after the timed region with the library's stage events on the launch stream "
                               "(direct launches: events between the stages cannot be part of the replayed graph); "
                               "`value` / `ms_per_step` are the timed region itself (graph replay, what a caller gets)"},
        "clocks": sampler.summary(t_wall0, t_wall2),
    }
    if dumped is not None:
        line["outputs_dumped"] = dumped
    if e2e is not None:
        line["e2e"] = e2e
    if corpus is not None:
        line["corpus"] = corpus
    if variants:
        for v in variants.values():
            if "gbs" in v:
                v["frac_of_hbm_peak"] = v["gbs"] / peak
        line["variants"] = variants
    if world == 1 and not a.no_cpu_baseline:
        pps, _, dt = cpu_baseline(a, a.cpu_pages, 1)
        line["cpu_baseline"] = {"value": pps, "unit": "pages/s", "cores": 1, "kind": "port",
                                "sample": f"{a.cpu_pages} pages of the same workload through the C oracle "
                                          f"(oracle/oracle.c), 1 thread, {dt:.1f} s"}
    print(json.dumps(line), file=_REAL_STDOUT or sys.stdout, flush=True)
    if dist is not None:
        dist.destroy_process_group()


def run_variants(a, mb, torch, dev, local, ctx, res, counts, d_score, d_geo, d_pages, h_pages, imgs_np, cap_boxes,
                 crops_cap, stream):
    """Paths next to the BASELINE metric, timed on one GPU after the main regions: reading order on the device, rotated
    crops, the other BASELINE shapes (configs[1], configs[3]), a denser candidate load, and Pipeline.predict."""
    import ctypes as C

    P, S = a.pages, a.page_size
    variants = {}

    def timed(fn, reps=5, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(reps):
            fn()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    if not a.reading_order:  # the step as Pipeline.predict runs it: boxes and crops in reading order
        ro = mb.PageBatch(device=local, params=mb.EastParams.default(target_size=S, sort_reading_order=1),
                          cap_boxes=cap_boxes, crops_cap=crops_cap, out_hw=(OUT_H, OUT_W))
        ms_ro = timed(lambda: ro.run(d_score, d_geo, d_pages))
        variants["with_reading_order"] = {"ms_per_step": ms_ro, "pages_per_s": P / (ms_ro * 1e-3),
                                          "note": "ms_east_params.sort_reading_order = 1 (utils.py:610-644 + "
                                                  "_pipeline.py:105-123 on the device)"}
        del ro
    # rotated-quad crops (SURVEY 8f-4 extension): this step's boxes, each turned by up to +-0.15 rad about its centre
    bx = res.boxes.cpu().numpy()
    quads, page_of = [], []
    rng = np.random.default_rng(1)
    for pg in range(P):
        q = bx[pg, : counts[pg], :8].reshape(-1, 4, 2).astype(np.float64)
        c = q.mean(axis=1, keepdims=True)
        ang = rng.uniform(-0.15, 0.15, len(q))
        rot = np.stack([np.stack([np.cos(ang), -np.sin(ang)], -1), np.stack([np.sin(ang), np.cos(ang)], -1)], -2)
        quads.append((np.einsum("nij,nkj->nki", rot, q - c) + c).reshape(-1, 8))
        page_of.append(np.full(len(q), pg, np.int32))
    quads = torch.from_numpy(np.concatenate(quads).astype(np.float32)).to(dev)
    page_of = torch.from_numpy(np.concatenate(page_of)).to(dev)
    nq = int(quads.shape[0])
    qbatch = torch.empty((nq, 3, OUT_H, OUT_W), dtype=torch.float32, device=dev)
    qsizes = torch.zeros((nq, 2), dtype=torch.int32, device=dev)

    def quad_run():
        mb._cabi.check(ctx.lib.ms_quad_crop_resize_pad(
            ctx.handle, d_pages.data_ptr(), P, S, S, quads.data_ptr(), 8, page_of.data_ptr(), nq, 5, 1, 0, OUT_H,
            OUT_W, qbatch.data_ptr(), None, qsizes.data_ptr(), C.c_void_p(stream.cuda_stream)))

    ms_q = timed(quad_run)
    sz = qsizes.cpu().numpy().astype(np.int64)
    q_bytes = 3 * int((sz[:, 0] * sz[:, 1]).sum()) + 3 * OUT_H * OUT_W * 4 * nq
    variants["rotated_quad_crop"] = {"ms_per_launch": ms_q, "quads": nq, "patches": int((sz[:, 0] > 0).sum()),
                                     "alg_bytes": q_bytes, "gbs": q_bytes / (ms_q * 1e-3) / 1e9,
                                     "note": "ms_quad_crop_resize_pad: cv2.warpPerspective-exact rectified crops "
                                             "(extension, not a reference behaviour)"}
    del qbatch, quads
    # one 1280x1280 page (BASELINE configs[1]): ~50 short launches, so the call is launch-bound; a repeated call is
    # replayed as a CUDA graph (second occurrence on), MS_B200_NO_GRAPHS=1 keeps direct launches
    s1, g1, i1 = synthdata.make_batch([7], 1280, 500)
    d1 = [torch.from_numpy(x).to(dev) for x in (s1, g1, i1)]
    one = mb.PageBatch(device=local, params=mb.EastParams.default(target_size=1280), cap_boxes=2048,
                       out_hw=(OUT_H, OUT_W))
    ms_graph = timed(lambda: one.run(*d1), reps=20)
    os.environ["MS_B200_NO_GRAPHS"] = "1"  # read when a context is created
    one_d = mb.PageBatch(device=local, params=mb.EastParams.default(target_size=1280), cap_boxes=2048,
                         out_hw=(OUT_H, OUT_W))
    del os.environ["MS_B200_NO_GRAPHS"]
    ms_direct = timed(lambda: one_d.run(*d1), reps=20)
    variants["single_page_1280"] = {"ms_graph_replay": ms_graph, "ms_direct_launches": ms_direct,
                                    "note": "BASELINE configs[1]: device-resident, one page per call, 500 words"}
    del one, one_d, d1
    # BASELINE configs[3]: 4096x4096 pages with ~10 000 quads (~63 000 candidates) each, NMS-bound; 8 pages per step
    s4, g4, i4 = synthdata.make_batch([3, 4], 4096, 10000)
    reps8 = [0, 1, 0, 1, 0, 1, 0, 1]
    d4 = [torch.from_numpy(np.ascontiguousarray(x[reps8])).to(dev) for x in (s4, g4, i4)]
    big = mb.PageBatch(device=local, params=mb.EastParams.default(target_size=4096), cap_boxes=16384,
                       crops_cap=8 * 12000, out_hw=(OUT_H, OUT_W))
    r4 = big.run(*d4, sync=True)
    ms4 = timed(lambda: big.run(*d4), reps=5)
    big.ctx.stage_timing(True)
    big.run(*d4)
    _, st4 = big.ctx.stage_times()
    big.ctx.stage_timing(False)
    variants["stress_4096"] = {"ms_per_step": ms4, "pages_per_step": 8, "pages_per_s": 8 / (ms4 * 1e-3),
                               "boxes_per_page": float(r4.box_counts.float().mean().item()),
                               "crops": int(r4.n_crops.item()), "stage_ms": st4,
                               "note": "BASELINE configs[3]: 8 pages of 4096x4096 (2 distinct, repeated), ~10 000 quads and "
                                       "~63 000 candidates per page; parity of this shape: tests/test_gpu_batch.py::"
                                       "test_stress_4096_page against the committed oracle digests"}
    # the same with the reading-order sort (10 000 boxes per page: the global-memory reading-order kernel)
    del big
    big_ro = mb.PageBatch(device=local, params=mb.EastParams.default(target_size=4096, sort_reading_order=1),
                          cap_boxes=16384, crops_cap=8 * 12000, out_hw=(OUT_H, OUT_W))
    r4o = big_ro.run(*d4, sync=True)
    assert int(r4o.n_crops.item()) == int(r4.n_crops.item())
    ms4o = timed(lambda: big_ro.run(*d4), reps=5)
    variants["stress_4096"]["with_reading_order_ms_per_step"] = ms4o
    del big_ro, r4o, d4, r4, s4, g4, i4
    # a denser candidate load (SURVEY 8d expected ~24k candidates per 2048^2 page): the score regions shrunk by 0.2 instead
    # of 0.3 of the shorter side, 16 pages
    sd, gd, _ = synthdata.make_batch(list(range(500, 516)), S, a.words, with_images=False, shrink=0.2)
    dd = [torch.from_numpy(x).to(dev) for x in (sd, gd)]
    dense = mb.PageBatch(device=local, params=mb.EastParams.default(target_size=S), cap_boxes=cap_boxes,
                         crops_cap=16 * (a.words + a.words // 4 + 64), out_hw=(OUT_H, OUT_W))
    rd = dense.run(dd[0], dd[1], d_pages[:16], sync=True)
    ccnt = torch.zeros((16,), dtype=torch.int32, device=dev)
    cflg = torch.zeros((16,), dtype=torch.int32, device=dev)
    M = S // 4
    cand = torch.empty((16, (M // 2) * (M // 2), 9), dtype=torch.float32, device=dev)
    mb._cabi.check(ctx.lib.ms_decode_quads(ctx.handle, dd[0].data_ptr(), dd[1].data_ptr(), 16, M, M, 0.6, 4.0, 2,
                                           cand.data_ptr(), cand.shape[1], ccnt.data_ptr(), cflg.data_ptr(),
                                           stream.cuda_stream))
    msd = timed(lambda: dense.run(dd[0], dd[1], d_pages[:16]), reps=5)
    dense.ctx.stage_timing(True)
    dense.run(dd[0], dd[1], d_pages[:16])
    _, std = dense.ctx.stage_times()
    dense.ctx.stage_timing(False)
    variants["dense_candidates"] = {"ms_per_step": msd, "pages_per_step": 16, "pages_per_s": 16 / (msd * 1e-3),
                                    "candidates_per_page": float(ccnt.float().mean().item()),
                                    "boxes_per_page": float(rd.box_counts.float().mean().item()), "stage_ms": std}
    del dense, dd, cand, rd
    # Pipeline.predict page by page through the public classes (fused route): stub networks -- the detector replays the
    # synthetic maps of page 0 from HBM, the recogniser returns constants -- so the time is the path's, not a network's
    class Net:
        def __call__(self, x):
            return {"score": d_score[0:1, None], "geometry": d_geo[0:1]}

    det = mb.EAST(model=Net(), target_size=S, device=local)
    rec = mb.TRBA(model=lambda batch: [("w", 0.5)] * len(batch), img_h=OUT_H, img_w=OUT_W, device=local)
    pipe = mb.Pipeline(detector=det, recognizer=rec)
    img0 = imgs_np[0]
    page = pipe.predict(img0)
    assert pipe.last_route == "fused"
    n_words = sum(len(b.words) for b in page.blocks)
    reps = 10
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        pipe.predict(img0)
    torch.cuda.synchronize()
    ms_pp = 1e3 * (time.perf_counter() - t0) / reps
    variants["pipeline_predict_2048"] = {
        "ms_per_page": ms_pp, "pages_per_s": 1e3 / ms_pp, "words": n_words, "h2d_bytes_per_page": int(img0.nbytes),
        "d2h_bytes_per_page": int(n_words * 36 + n_words * 20 + 16),
        "note": "mb.Pipeline(mb.EAST, mb.TRBA).predict(image) on one 2048x2048 page, wall clock incl. building the Page "
                "of ~2000 Word objects on the host: ONE upload of the page image, zero downloads of pixels; the network "
                "input, maps, boxes, reading order and the recogniser batch stay on the device"}
    return variants


def main():
    a = parse_args()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_b200(a)


if __name__ == "__main__":
    main()
