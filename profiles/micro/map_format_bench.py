"""Detector maps in the formats a B200 network returns them in, on the benchmark workload:
    python profiles/micro/map_format_bench.py [out.json]

Workload: bench.py's default (BASELINE configs[2]): 64 synthetic 2048 x 2048 pages, ~2000 words each, 512 x 512 maps,
32 x 128 float32 canvases, the same device buffers every step (graph replay).  The seeded maps are rounded to bfloat16
once, so that every arm sees the same values.  Arms, alternated in one process for three rounds, CUDA-event-timed steps,
each arm on its own context (its own arena and graph cache):
  A  f32 NCHW maps                        ms_page_batch_ex                      (a float32 network today)
  B  bf16 NCHW maps                       .float() of both maps, ms_page_batch_ex (a bfloat16 network today)
  C  bf16 NCHW maps                       ms_page_batch_maps
  D  bf16 maps, channels_last geometry    ms_page_batch_maps
  E  f32 maps, channels_last geometry     .contiguous(), ms_page_batch_ex    (E_copy)
                                          against ms_page_batch_maps          (E_maps)
Then the decode stage of every arm (ms_stage_timing events, direct launches, as bench.py reads it) and the peak of
torch.cuda.max_memory_allocated above the inputs for one step of B and of C.  Every arm's boxes, counts, flags, crop
list and batch are checked against arm A before timing."""
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
STEPS, ROUNDS = 200, 3


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip().splitlines()[:1]}


class Arm:
    """One page-batch call with its own context and output buffers; prep(score, geo) -> the maps the call is given
    (inside the timed region), maps=True: through ms_page_batch_maps."""

    def __init__(self, score, geo, pages, prep, maps):
        dev = pages.device
        self.ctx = mb.Context(0)
        self.score, self.geo, self.pages, self.prep, self.maps = score, geo, pages, prep, maps
        self.params = mb.EastParams.default(target_size=S)
        self.cap_boxes, self.crops_cap = max(4096, 2 * WORDS), P * (WORDS + WORDS // 4 + 64)
        self.boxes = torch.empty((P, self.cap_boxes, 9), dtype=torch.float32, device=dev)
        self.counts = torch.zeros((P,), dtype=torch.int32, device=dev)
        self.crops = torch.zeros((self.crops_cap, 5), dtype=torch.int32, device=dev)
        self.n_crops = torch.zeros((1,), dtype=torch.int32, device=dev)
        self.batch = torch.empty((self.crops_cap, 3, OUT_H, OUT_W), dtype=torch.float32, device=dev)
        self.flags = torch.zeros((P,), dtype=torch.int32, device=dev)

    def __call__(self):
        s, g = self.prep(self.score, self.geo)
        H, W = s.shape[1:]
        lib, stream = self.ctx.lib, torch.cuda.current_stream().cuda_stream
        tail = (self.pages.data_ptr(), P, H, W, S, S, C.byref(self.params), 5, OUT_H, OUT_W, self.cap_boxes,
                self.boxes.data_ptr(), self.counts.data_ptr(), self.crops.data_ptr(), self.crops_cap,
                self.n_crops.data_ptr(), self.batch.data_ptr(), mb._cabi.MS_DTYPE_F32, None, self.flags.data_ptr(),
                C.c_void_p(stream))
        if self.maps:
            d = mb._cabi.maps_descriptor(s, g)
            mb._cabi.check(lib.ms_page_batch_maps(self.ctx.handle, C.byref(d), *tail))
        else:
            mb._cabi.check(lib.ms_page_batch_ex(self.ctx.handle, s.data_ptr(), g.data_ptr(), *tail))
        return s, g  # (kept alive until the call is queued)

    def outputs(self):
        torch.cuda.synchronize()
        counts = self.counts.cpu().numpy()
        n = int(self.n_crops.item())
        return ([counts, self.flags.cpu().numpy(), self.crops[:n].cpu().numpy(), self.batch[:n].view(torch.int32).cpu().numpy()]
                + [self.boxes[p, : counts[p]].view(torch.int32).cpu().numpy() for p in range(P)])


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    dev = torch.device("cuda:0")
    score, geo, imgs = synthdata.make_batch(list(range(P)), S, WORDS)
    pages = torch.from_numpy(imgs).to(dev)
    s_bf = torch.from_numpy(score).to(dev).to(torch.bfloat16)
    g_bf = torch.from_numpy(geo).to(dev).to(torch.bfloat16)
    del score, geo, imgs
    s32, g32 = s_bf.float(), g_bf.float()
    g_bf_cl = g_bf.contiguous(memory_format=torch.channels_last)
    g32_cl = g32.contiguous(memory_format=torch.channels_last)
    same = lambda s, g: (s, g)  # noqa: E731
    arms = {
        "A_f32_nchw_ex": Arm(s32, g32, pages, same, False),
        "B_bf16_nchw_float_ex": Arm(s_bf, g_bf, pages, lambda s, g: (s.float(), g.float()), False),
        "C_bf16_nchw_maps": Arm(s_bf, g_bf, pages, same, True),
        "D_bf16_cl_maps": Arm(s_bf, g_bf_cl, pages, same, True),
        "E_copy_f32_cl_contiguous_ex": Arm(s32, g32_cl, pages, lambda s, g: (s, g.contiguous()), False),
        "E_maps_f32_cl_maps": Arm(s32, g32_cl, pages, same, True),
    }
    assert g_bf_cl.stride() == (8 * 512 * 512, 1, 8 * 512, 8) and not g32_cl.is_contiguous()

    # parity against arm A, before timing (direct launches)
    for a in arms.values():
        a()
    want = arms["A_f32_nchw_ex"].outputs()
    assert not want[1].any(), "flags on the benchmark workload"
    parity = {}
    for k, a in arms.items():
        got = a.outputs()
        parity[k] = all(np.array_equal(x, y) for x, y in zip(got, want))

    # memory above the inputs: one step of B against C (each after a step that settled its arena)
    mem = {}
    for k in ("B_bf16_nchw_float_ex", "C_bf16_nchw_maps"):
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated()
        torch.cuda.reset_peak_memory_stats()
        arms[k]()
        torch.cuda.synchronize()
        mem[k] = torch.cuda.max_memory_allocated() - base

    stream = torch.cuda.current_stream()

    def timed(f, steps):
        for _ in range(3):  # graph capture at the second call
            f()
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
        for k, a in arms.items():
            step_ms[k].append(timed(a, STEPS))

    decode_ms = {k: [] for k in arms}
    for _ in range(ROUNDS):
        for k, a in arms.items():
            a.ctx.stage_timing(True)
            for _ in range(STEPS // 4):
                a()
            nb, st = a.ctx.stage_times()
            a.ctx.stage_timing(False)
            decode_ms[k].append(st["decode"] / nb)

    med = lambda v: float(np.median(v))  # noqa: E731
    out = {
        "gpu": gpu_identity(),
        "workload": f"{P} pages {S}x{S}, {WORDS} words each (BASELINE configs[2]), maps {P}x(1+8)x512x512 rounded to "
                    f"bfloat16, {OUT_H}x{OUT_W} float32 canvases, {int(want[3].shape[0])} crops per step",
        "steps_per_arm": STEPS, "rounds": ROUNDS,
        "parity_bit_exact_vs_A": parity,
        "step_ms": {k: {"rounds": v, "median": med(v)} for k, v in step_ms.items()},
        "decode_stage_ms": {k: {"rounds": v, "median": med(v), "note": "direct launches, the front half on the "
                                "caller's stream"} for k, v in decode_ms.items()},
        "peak_bytes_above_inputs": mem,
        "map_bytes": {"f32": int(s32.numel() + g32.numel()) * 4, "bf16": int(s_bf.numel() + g_bf.numel()) * 2},
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
