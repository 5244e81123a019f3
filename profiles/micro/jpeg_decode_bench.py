"""Device JPEG decode (ms_jpeg_decode_batch) against cv2.imread, and Pipeline.process_batch(paths) against a parent tree.

    python profiles/micro/jpeg_decode_bench.py [--rounds 7] [--parent-tree DIR] [--out profiles/jpeg_decode_bench.json]

1. 64 pages of 2048 x 2048 per set (document-like at q75 and q90, synthdata.make_page_image at q90; 4:2:0), each set
   decoded by one ms_jpeg_decode_batch call, the H2D copy of the compressed bytes included.  Sets alternate within
   every round; medians over rounds.  Stage times come from a separate torch.profiler run (kernel durations summed
   per stage).  The IDCT / colour stages' algorithmic bytes: coefficients read (128 B per block) + planes written and
   read (64 B per block, twice) + RGB written.
2. cv2.imread of the same files on one host core and on a thread pool of every host core.
3. With --parent-tree (a checkout of the parent commit, e.g. `git worktree add DIR HEAD~1`): Pipeline.process_batch on
   the same 64 files of one set with bench.py's stub networks, in a child process per tree, alternating; the Pages of
   the two trees must be equal.
The card's name and power limit are read in the same run.  Files are written to a temporary directory.
"""
import argparse
import concurrent.futures as cf
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path[:0] = [ROOT, os.path.join(ROOT, "manuscript-ocr_b200")]
N, SIDE = 64, 2048


def doc_page(seed):
    rng = np.random.default_rng(seed)
    a = np.full((SIDE, SIDE, 3), 244, np.uint8) + rng.integers(0, 8, (SIDE, SIDE, 3), dtype=np.uint8)
    for _ in range(SIDE * SIDE // 3000):
        y, x = int(rng.integers(0, SIDE)), int(rng.integers(0, SIDE))
        a[y:y + 12, x:x + 50] = int(rng.integers(0, 70))
    return a


def make_sets(tmp):
    import cv2

    import synthdata

    sets = {}
    for name, make, q in (("doc_q75", doc_page, 75), ("doc_q90", doc_page, 90),
                          ("synth_q90", lambda s: synthdata.make_page_image(s, SIDE), 90)):
        paths = []
        for i in range(N):
            p = os.path.join(tmp, f"{name}_{i}.jpg")
            img = make(1000 + i)
            cv2.imwrite(p, cv2.cvtColor(img, cv2.COLOR_RGB2BGR),
                        [cv2.IMWRITE_JPEG_QUALITY, q, cv2.IMWRITE_JPEG_SAMPLING_FACTOR,
                         cv2.IMWRITE_JPEG_SAMPLING_FACTOR_420])
            paths.append(p)
        sets[name] = paths
    return sets


STAGES = {"unstuff": ("jpg_end", "jpg_count", "jpg_scan", "jpg_emit"),
          "huffman_sync": ("jpg_guess", "jpg_sync", "jpg_fix", "jpg_base"),
          "huffman_write": ("jpg_write",), "dc": ("jpg_dc",), "idct": ("jpg_idct",), "color": ("jpg_color",)}


def device_part(sets, rounds):
    import torch

    import manuscript_b200 as mb

    ctx = mb.Context(0)
    lib = ctx.lib
    datas = {k: [open(p, "rb").read() for p in v] for k, v in sets.items()}
    outs = [torch.empty((SIDE, SIDE, 3), dtype=torch.uint8, device="cuda") for _ in range(N)]
    status = torch.empty((N,), dtype=torch.int32, pin_memory=True)
    stream = torch.cuda.current_stream()

    def call(ds):
        keep = [C.c_char_p(d) for d in ds]
        files = (C.c_void_p * N)(*[C.cast(k, C.c_void_p).value for k in keep])
        sizes = (C.c_int64 * N)(*[len(d) for d in ds])
        ptrs = (C.c_void_p * N)(*[o.data_ptr() for o in outs])
        mb._cabi.check(lib.ms_jpeg_decode_batch(ctx.handle, files, sizes, N, ptrs, status.data_ptr(),
                                                C.c_void_p(stream.cuda_stream)))
        stream.synchronize()

    import cv2

    for k, ds in datas.items():  # warm-up and correctness of a sample of pages
        call(ds)
        assert (status.numpy() == 0).all(), (k, status.numpy())
        for i in (0, N - 1):
            want = cv2.cvtColor(cv2.imread(sets[k][i]), cv2.COLOR_BGR2RGB)
            assert np.array_equal(outs[i].cpu().numpy(), want), (k, i)
    times = {k: [] for k in datas}
    for _ in range(rounds):
        for k, ds in datas.items():
            t0 = time.perf_counter()
            call(ds)
            times[k].append((time.perf_counter() - t0) * 1e3)
    stages = {}
    from torch.profiler import ProfilerActivity, profile

    for k, ds in datas.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call(ds)
        per = {s: 0.0 for s in STAGES}
        h2d = 0.0
        for ev in prof.events():
            name, dur = ev.name, ev.device_time_total / 1e3 if hasattr(ev, "device_time_total") else 0.0
            if "Memcpy HtoD" in name:
                h2d += dur
            for s, pref in STAGES.items():
                if any(name.startswith(p) or f" {p}" in name or name.startswith("void " + p) for p in pref):
                    per[s] += dur
        stages[k] = {"h2d_ms": round(h2d, 3), **{f"{s}_ms": round(v, 3) for s, v in per.items()}}
    res = {}
    for k, ds in datas.items():
        med = float(np.median(times[k]))
        mbytes = sum(len(d) for d in ds) / 1e6
        blocks = N * (SIDE // 8) ** 2 * 6 // 4  # 4:2:0: 6 blocks per 16 x 16 MCU
        algo = blocks * 128 + blocks * 64 * 2 + N * SIDE * SIDE * 3
        st = stages[k]
        idct_color = st["idct_ms"] + st["color_ms"]
        res[k] = {"ms_per_64_pages": round(med, 3), "spread_ms": [round(min(times[k]), 3), round(max(times[k]), 3)],
                  "compressed_MB": round(mbytes, 2), "compressed_MB_per_s": round(mbytes / med * 1e3, 1),
                  "output_MP_per_s": round(N * SIDE * SIDE / 1e6 / med * 1e3, 1), "stages": st,
                  "idct_color_algorithmic_GB": round(algo / 1e9, 3),
                  "idct_color_share_of_6557_GBps": round(algo / 1e9 / (idct_color / 1e3) / 6557, 3)
                  if idct_color > 0 else None}
    return res


def _read(p):
    import cv2

    return cv2.imread(p)


def host_part(sets):
    import cv2

    cv2.setNumThreads(1)
    out = {"host_cores": os.cpu_count()}
    for k, paths in sets.items():
        t0 = time.perf_counter()
        for p in paths:
            _read(p)
        one = (time.perf_counter() - t0) * 1e3
        with cf.ThreadPoolExecutor(os.cpu_count()) as ex:
            t0 = time.perf_counter()
            list(ex.map(_read, paths))
            allc = (time.perf_counter() - t0) * 1e3
        out[k] = {"imread_1_core_ms_per_64": round(one, 1), "imread_all_cores_ms_per_64": round(allc, 1)}
    return out


def pipeline_part(parent, paths, rounds, tmp):
    """process_batch(paths) in a child process per tree (this one and the parent), alternating"""
    lst = os.path.join(tmp, "paths.json")
    json.dump(paths, open(lst, "w"))
    child = os.path.join(tmp, "child.py")
    with open(child, "w") as f:
        f.write(CHILD_SRC)
    trees = {"this": ROOT, "parent": os.path.abspath(parent)}
    for t in trees.values():  # build each tree's library in place first
        subprocess.run([sys.executable, os.path.join(t, "manuscript-ocr_b200", "build.py")], check=True,
                       stdout=subprocess.DEVNULL)
    walls = {k: [] for k in trees}
    digests = {}
    for _ in range(rounds):
        for k, t in trees.items():
            r = subprocess.run([sys.executable, child, t, lst], check=True, capture_output=True, text=True)
            line = json.loads(r.stdout.strip().splitlines()[-1])
            walls[k].append(line["wall_ms"])
            digests.setdefault(k, line["digest"])
            assert digests[k] == line["digest"]
    return {"pages": len(paths), "pages_equal": digests["this"] == digests["parent"],
            **{f"{k}_process_batch_ms": round(float(np.median(v)), 1) for k, v in walls.items()},
            **{f"{k}_spread_ms": [round(min(v), 1), round(max(v), 1)] for k, v in walls.items()}}


CHILD_SRC = r'''
import hashlib, json, sys, time
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/manuscript-ocr_b200"]
import numpy as np, torch
import manuscript_b200 as mb
paths = json.load(open(sys.argv[2]))
T = 1280


class StubEAST:  # bench.py's stub detector: fixed maps per row, made once
    def __init__(self):
        import synthdata
        s, g, _ = synthdata.make_batch([7], T, 200)
        self.s = torch.from_numpy(s).cuda()[:, None] if s.ndim == 3 else torch.from_numpy(s).cuda()
        self.g = torch.from_numpy(g).cuda()

    def __call__(self, x):
        P = x.shape[0]
        return {"score": self.s.expand(P, *self.s.shape[1:]), "geometry": self.g.expand(P, *self.g.shape[1:])}


class StubTRBA:
    def __call__(self, batch):
        m = batch.float().mean(dim=(1, 2, 3)).cpu().numpy()
        return [(f"w{i % 97}", float(v)) for i, v in enumerate(m)]


det = mb.EAST(model=StubEAST(), target_size=T)
rec = mb.TRBA(model=StubTRBA(), img_h=32, img_w=128, batch_size=256)
pipe = mb.Pipeline(detector=det, recognizer=rec)
pipe.process_batch(paths[:2], max_pages=32)  # warm-up: library load, buffers
torch.cuda.synchronize()
t0 = time.perf_counter()
pages = pipe.process_batch(paths, max_pages=32)
torch.cuda.synchronize()
wall = (time.perf_counter() - t0) * 1e3
h = hashlib.sha256()
for p in pages:
    for b in p.blocks:
        for w in b.words:
            h.update(repr((w.polygon, w.detection_confidence, w.text, w.recognition_confidence)).encode())
print(json.dumps({"wall_ms": wall, "digest": h.hexdigest()}))
'''


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--parent-tree", default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "jpeg_decode_bench.json"))
    a = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        raise SystemExit("jpeg_decode_bench needs a CUDA device")
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
    with tempfile.TemporaryDirectory() as tmp:
        sets = make_sets(tmp)
        result = {"gpu": gpu, "pages_per_set": N, "page": [SIDE, SIDE], "sampling": "4:2:0",
                  "device_decode": device_part(sets, a.rounds), "host_imread": host_part(sets)}
        if a.parent_tree:
            result["process_batch_paths"] = pipeline_part(a.parent_tree, sets["doc_q90"], max(3, a.rounds // 2), tmp)
    line = json.dumps(result)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(json.dumps(result, indent=1) + "\n")


if __name__ == "__main__":
    main()
