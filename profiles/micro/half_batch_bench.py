"""The recogniser batch in float32, float16 and bfloat16 on the benchmark workload:
    python profiles/micro/half_batch_bench.py [out.json]

Workload: bench.py's default (BASELINE configs[2]): 64 synthetic 2048 x 2048 pages, ~2000 words each, 32 x 128 canvases,
the same device buffers every step.  Arms, alternated in one process for three rounds, 250 CUDA-event-timed steps each:
  f32, f16, bf16      PageBatch(batch_dtype=...).run: the whole step, the crop kernels writing that dtype
  f32+cast            the f32 step followed by batch[:n].to(torch.bfloat16): what a 16-bit recogniser needs without
                      the 16-bit batch
Then, per dtype, the crop stage alone (ms_stage_timing events, direct launches) with its algorithmic bytes
(3 * sum(w * h) read + 3 * 32 * 128 * element size * n_crops written) against the measured 6 557 GB/s copy peak, and the
benchmark's word boxes as rotated quads (~128 000, turned by up to +-0.15 rad) through ms_quad_crop_resize_pad_ex.
Every 16-bit batch is checked bit for bit against the f32 batch cast with .to(dtype)."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "manuscript-ocr_b200")]
import manuscript_b200 as mb  # noqa: E402
import synthdata  # noqa: E402

P, S, WORDS, OUT_H, OUT_W = 64, 2048, 2000, 32, 128
STEPS, ROUNDS = 250, 3
PEAK_GBS = 6557.0  # measured device-to-device copy peak of one B200 (profiles/README.md)
DTYPES = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    dev = torch.device("cuda:0")
    score, geo, imgs = synthdata.make_batch(list(range(P)), S, WORDS)
    d_score, d_geo, d_pages = (torch.from_numpy(x).to(dev) for x in (score, geo, imgs))
    params = mb.EastParams.default(target_size=S)
    kw = dict(device=0, params=params, cap_boxes=max(4096, 2 * WORDS), crops_cap=P * (WORDS + WORDS // 4 + 64),
              out_hw=(OUT_H, OUT_W))
    runners = {k: mb.PageBatch(batch_dtype=dt, **kw) for k, dt in DTYPES.items()}
    stream = torch.cuda.current_stream()

    res = {k: r.run(d_score, d_geo, d_pages, sync=True) for k, r in runners.items()}
    n = int(res["f32"].n_crops.item())
    crops = res["f32"].crops[:n].cpu().numpy().astype(np.int64)
    src_px = int(((crops[:, 3] - crops[:, 1]) * (crops[:, 4] - crops[:, 2])).sum())
    parity = {}
    for k in ("f16", "bf16"):
        ok = torch.equal(res[k].crops[:n], res["f32"].crops[:n]) and torch.equal(
            res[k].batch[:n].view(torch.int16), res["f32"].batch[:n].to(DTYPES[k]).view(torch.int16))
        parity[k] = bool(ok)

    arms = {k: (lambda r=r: r.run(d_score, d_geo, d_pages)) for k, r in runners.items()}
    arms["f32+cast"] = lambda: runners["f32"].run(d_score, d_geo, d_pages).batch[:n].to(torch.bfloat16)
    for f in arms.values():  # warm-up, graph capture
        for _ in range(3):
            f()
    torch.cuda.synchronize()

    def timed(f, steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record(stream)
        for _ in range(steps):
            f()
        e1.record(stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    step_ms = {k: [] for k in arms}
    for _ in range(ROUNDS):
        for k, f in arms.items():
            step_ms[k].append(timed(f, STEPS))

    crop_ms = {k: [] for k in DTYPES}
    for _ in range(ROUNDS):
        for k, r in runners.items():
            r.ctx.stage_timing(True)
            for _ in range(STEPS):
                r.run(d_score, d_geo, d_pages)
            nb, st = r.ctx.stage_times()
            r.ctx.stage_timing(False)
            crop_ms[k].append(st["crop"] / nb)
    crop_bytes = {k: 3 * src_px + 3 * OUT_H * OUT_W * DTYPES[k].itemsize * n for k in DTYPES}

    # the benchmark's boxes as rotated quads (profiles/micro/quad_bench.py's construction, all 64 pages)
    counts = res["f32"].box_counts.cpu().numpy()
    bx = res["f32"].boxes.cpu().numpy()
    rng = np.random.default_rng(1)
    quads, page_of = [], []
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
    ctx = mb.Context(0)
    qout = {k: torch.empty((nq, 3, OUT_H, OUT_W), dtype=dt, device=dev) for k, dt in DTYPES.items()}
    sizes = torch.zeros((nq, 2), dtype=torch.int32, device=dev)

    def quad_run(k):
        mb._cabi.check(ctx.lib.ms_quad_crop_resize_pad_ex(
            ctx.handle, d_pages.data_ptr(), P, S, S, quads.data_ptr(), 8, page_of.data_ptr(), nq, 5, 1, 0, OUT_H, OUT_W,
            qout[k].data_ptr(), mb.batch_dtype_code(DTYPES[k]), None, sizes.data_ptr(), C.c_void_p(stream.cuda_stream)))

    for k in DTYPES:
        quad_run(k)
    qc = (C.c_int32 * 2)()
    mb._cabi.check(ctx.lib.ms_quad_crop_last_counts(ctx.handle, qc))
    for k in ("f16", "bf16"):
        parity["quad_" + k] = bool(torch.equal(qout[k].view(torch.int16), qout["f32"].to(DTYPES[k]).view(torch.int16)))
    quad_ms = {k: [] for k in DTYPES}
    for _ in range(ROUNDS):
        for k in DTYPES:
            quad_ms[k].append(timed(lambda k=k: quad_run(k), 20))

    med = lambda v: float(np.median(v))  # noqa: E731
    out = {
        "gpu": gpu_identity(),
        "workload": f"{P} pages {S}x{S}, {WORDS} words each (BASELINE configs[2]), {OUT_H}x{OUT_W} canvases, "
                    f"{n} crops per step, {src_px} source pixels",
        "steps_per_arm": STEPS, "rounds": ROUNDS,
        "parity_bit_exact_vs_f32_cast": parity,
        "step_ms": {k: {"rounds": v, "median": med(v)} for k, v in step_ms.items()},
        "crop_stage": {k: {"ms_rounds": crop_ms[k], "ms_median": med(crop_ms[k]), "alg_bytes": crop_bytes[k],
                           "alg_GBs": crop_bytes[k] / med(crop_ms[k]) / 1e6,
                           "share_of_copy_peak": crop_bytes[k] / med(crop_ms[k]) / 1e6 / PEAK_GBS} for k in DTYPES},
        "cast_to_bf16_ms": med(step_ms["f32+cast"]) - med(step_ms["f32"]),
        "rotated_quads": {"quads": nq, "staged": int(qc[0]), "generic": int(qc[1]),
                          "ms": {k: {"rounds": v, "median": med(v)} for k, v in quad_ms.items()}},
        "copy_peak_GBs": PEAK_GBS,
    }
    text = json.dumps(out, indent=1)
    print(text)
    if out_path:
        with open(out_path, "w") as f:
            f.write(text + "\n")
    if not all(parity.values()):
        sys.exit(1)


if __name__ == "__main__":
    main()
