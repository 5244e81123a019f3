"""BASELINE configs[0]: "Pipeline().predict on example/ocr_example_image.jpg with default EAST+TRBA, weights-free random
init on CPU (reference post-process path)" -- the plumbing run, as a golden fixture.

Run in the build container only (needs /root/reference, torchvision, cv2):

    python tests/golden/make_golden_cfg0.py

The reference's OWN network module (detectors/_east/east.py:99-139, loaded by file path) is built with random weights
under a fixed seed and run on the CPU on the reference's example image, prepared exactly as EAST.predict prepares it
(infer.py:301-313: cv2.resize to target_size^2, ToTensor, Normalize(0.5, 0.5)).  Random init puts the whole score map at
~0.45-0.46 (SURVEY 8c), far below the default threshold 0.6, so the run is made at score_thresh = the median of the map:
about half of the map's cells become candidates.  The reference's post-processing functions (decode_quads_from_maps,
locality_aware_nms, expand_boxes, the EAST box filters) are then run on those maps.

The fixture holds the network INPUT hash, the maps (float32, exactly as the network produced them) and the reference's
outputs, so that the GPU box -- which has neither /root/reference nor the example image -- can replay the maps through
mb.EAST / mb.Pipeline and compare.  target_size = 640 keeps the fixture small (160 x 160 maps); the example
image itself is 4250 x 5390 and is replaced by its 640 x 640 network-input resize (stored as uint8).  The geometry map
is stored only at the pixels a quantisation-2 decode reads (geo[:, 1::2, 1::2], the centre of every 2 x 2 cell), which
keeps the file under 1 MB; the outputs are checked to be the same with every other pixel set to zero.
"""
import hashlib
import importlib.util
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import cpu, refload  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "cfg0_example.npz")
TARGET = 640


def sha(*arrs):
    h = hashlib.sha256()
    for a in arrs:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def main():
    import cv2
    import torch

    spec = importlib.util.spec_from_file_location("_ref_east_model", os.path.join(refload._SRC, "detectors/_east/east.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    torch.manual_seed(0)
    torch.set_num_threads(8)
    model = mod.EAST(pretrained_backbone=False).eval()  # random init, no weights anywhere
    img = cv2.cvtColor(cv2.imread(os.path.join(refload.REF_ROOT, "example", "ocr_example_image.jpg")), cv2.COLOR_BGR2RGB)
    resized = cv2.resize(img, (TARGET, TARGET))                                         # infer.py:304
    t = torch.from_numpy(resized).permute(2, 0, 1).float().div(255.0)                   # ToTensor
    t = (t - 0.5) / 0.5                                                                 # Normalize(0.5, 0.5)
    with torch.no_grad():
        out = model(t.unsqueeze(0))
    score = out["score"][0].numpy().squeeze(0).astype(np.float32)
    geo = out["geometry"][0].numpy().astype(np.float32)
    thr = float(np.median(score))
    ru, rs = refload.utils(), refload.lanms_stable()
    quads = ru.decode_quads_from_maps(score, geo.transpose(1, 2, 0), thr, 4.0, 2)
    nms = rs.locality_aware_nms(quads, 0.2)
    ep = refload.EastPost(target_size=TARGET)
    orig_hw = img.shape[:2]
    e = ru.expand_boxes(nms, 0.9, 0.9)
    final = ep._convert_to_axis_aligned(ep._remove_area_anomalies(ep._remove_fully_contained_boxes(
        ep._scale_boxes_to_original(e, orig_hw))))
    # the C oracle agrees with the reference on these network-made maps as well
    oq = cpu.decode_quads_from_maps(score, geo, thr, 4.0, 2)
    assert np.array_equal(oq, quads)
    assert np.array_equal(cpu.locality_aware_nms(oq, 0.2), nms)
    assert np.array_equal(cpu.east_postprocess(nms, orig_hw, target_size=TARGET), final)
    centres = np.ascontiguousarray(geo[:, 1::2, 1::2])
    sparse = np.zeros_like(geo)
    sparse[:, 1::2, 1::2] = centres
    assert np.array_equal(cpu.decode_quads_from_maps(score, sparse, thr, 4.0, 2), quads)
    np.savez_compressed(OUT, target=TARGET, orig_hw=np.array(orig_hw), resized=resized, input_sha=sha(t.numpy()),
                        score=score, geo_centres=centres, score_thresh=thr, n_candidates=len(quads), quads_sha=sha(quads),
                        lanms=nms, final=final, score_min=float(score.min()), score_max=float(score.max()))
    print("score range", score.min(), score.max(), "thr", thr, "candidates", len(quads), "kept", len(nms), "final",
          len(final), "bytes", os.path.getsize(OUT))


if __name__ == "__main__":
    if not refload.available():
        sys.exit("reference not found: run in the build container")
    main()
