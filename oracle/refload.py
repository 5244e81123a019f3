"""Load the REAL reference hot-path modules (olegiy/manuscript-ocr v0.1.8) by file path.

The reference source tree is not part of this repository: it is looked for in oracle/_ref/ (kept out of git) or in
the directory MANUSCRIPT_REFERENCE_ROOT names.  TEST INFRASTRUCTURE ONLY, so nothing marked `gpu`, smoke() or
bench.py may call this.  It is used by tests/golden/make_golden*.py (fixture generation) and by `not gpu` tests that
cross-check the oracle against the live reference when it is present (skipped otherwise).

The reference package cannot be imported as a whole here (gdown / shapely / albumentations are
not installed, SURVEY 8c), so the two self-contained modules are loaded directly:
  * detectors/_east/lanms.py   -- needs only numpy + numba
  * detectors/_east/utils.py   -- needs a stub `shapely.geometry.Polygon` (eval helpers only)
  * recognizers/_trba/data/transforms.py -- needs stub `albumentations` (ImageOnlyTransform base)
infer.py / _pipeline.py methods that are plain functions of numpy arrays are extracted from the
source with `ast` and executed against a tiny stand-in `self` (no model, no weights).
"""
import ast
import importlib.util
import os
import sys
import types

REF_ROOT = os.environ.get("MANUSCRIPT_REFERENCE_ROOT") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")
_SRC = os.path.join(REF_ROOT, "src", "manuscript")


def available() -> bool:
    return os.path.isfile(os.path.join(_SRC, "detectors", "_east", "lanms.py"))


def _load(name, relpath):
    spec = importlib.util.spec_from_file_location(name, os.path.join(_SRC, relpath))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


_cache = {}


def lanms():
    if "lanms" not in _cache:
        _cache["lanms"] = _load("_ref_lanms", "detectors/_east/lanms.py")
    return _cache["lanms"]


class _StableNumpy:
    """numpy proxy whose argsort is stable: the documented tie rule (SURVEY 8c)."""

    def __init__(self, np):
        self._np = np

    def __getattr__(self, k):
        return getattr(self._np, k)

    def argsort(self, a, *args, **kw):
        kw.setdefault("kind", "stable")
        return self._np.argsort(a, *args, **kw)


def lanms_stable():
    """The reference lanms module with np.argsort forced to kind='stable' in the two pure-Python
    functions (standard_nms, locality_aware_nms).  The njit primitives are untouched (they were
    compiled at import)."""
    if "lanms_stable" not in _cache:
        import numpy as np

        mod = _load("_ref_lanms_stable", "detectors/_east/lanms.py")
        mod.np = _StableNumpy(np)
        _cache["lanms_stable"] = mod
    return _cache["lanms_stable"]


def utils():
    if "utils" not in _cache:
        if "shapely" not in sys.modules:
            sh = types.ModuleType("shapely")
            geo = types.ModuleType("shapely.geometry")

            class Polygon:  # only the offline eval helpers touch it
                def __init__(self, *a, **k):
                    raise RuntimeError("shapely stub")

            geo.Polygon = Polygon
            sh.geometry = geo
            sys.modules["shapely"] = sh
            sys.modules["shapely.geometry"] = geo
        _cache["utils"] = _load("_ref_east_utils", "detectors/_east/utils.py")
    return _cache["utils"]


def transforms():
    if "transforms" not in _cache:
        if "albumentations" not in sys.modules:
            A = types.ModuleType("albumentations")

            class ImageOnlyTransform:
                def __init__(self, always_apply=True, p=1.0):
                    pass

            A.ImageOnlyTransform = ImageOnlyTransform
            A.Compose = lambda *a, **k: None
            A.Normalize = lambda *a, **k: None
            A.ShiftScaleRotate = A.RandomBrightnessContrast = A.InvertImg = lambda *a, **k: None
            Ap = types.ModuleType("albumentations.pytorch")
            Ap.ToTensorV2 = lambda *a, **k: None
            A.pytorch = Ap
            sys.modules["albumentations"] = A
            sys.modules["albumentations.pytorch"] = Ap
        _cache["transforms"] = _load("_ref_trba_transforms", "recognizers/_trba/data/transforms.py")
    return _cache["transforms"]


def _extract_methods(relpath, class_name, method_names, extra_globals):
    """Compile selected methods of a reference class without importing its module."""
    with open(os.path.join(_SRC, relpath), "r", encoding="utf-8") as f:
        tree = ast.parse(f.read())
    out = {}
    for node in tree.body:
        if isinstance(node, ast.ClassDef) and node.name == class_name:
            for item in node.body:
                if isinstance(item, ast.FunctionDef) and item.name in method_names:
                    item.decorator_list = []
                    item.returns = None
                    for a in item.args.args + item.args.kwonlyargs:
                        a.annotation = None
                    m = ast.Module(body=[item], type_ignores=[])
                    ast.fix_missing_locations(m)
                    ns = dict(extra_globals)
                    exec(compile(m, relpath, "exec"), ns)
                    out[item.name] = ns[item.name]
    missing = set(method_names) - set(out)
    if missing:
        raise RuntimeError(f"reference methods not found: {missing}")
    return out


class EastPost:
    """Stand-in `self` carrying only the attributes the EAST box filters read
    (infer.py:134-233); the methods themselves are the reference's own code."""

    def __init__(self, target_size=1280, remove_area_anomalies=True, anomaly_sigma_threshold=5.0,
                 anomaly_min_box_count=30):
        import cv2
        import numpy as np

        self.target_size = target_size
        self.remove_area_anomalies = remove_area_anomalies
        self.anomaly_sigma_threshold = anomaly_sigma_threshold
        self.anomaly_min_box_count = anomaly_min_box_count
        names = ["_scale_boxes_to_original", "_convert_to_axis_aligned", "_polygon_area_batch",
                 "_is_quad_inside", "_remove_fully_contained_boxes", "_remove_area_anomalies"]
        fns = _extract_methods("detectors/_east/infer.py", "EAST", names, {"np": np, "cv2": cv2})
        for k, fn in fns.items():
            if k == "_polygon_area_batch":
                setattr(self, k, fn)  # staticmethod in the reference
            else:
                setattr(self, k, types.MethodType(fn, self))


class PipelineCrop:
    """Stand-in for Pipeline carrying `_extract_word_image` (_pipeline.py:204-221)."""

    def __init__(self, min_text_size=5):
        import numpy as np

        self.min_text_size = min_text_size
        fns = _extract_methods("_pipeline.py", "Pipeline", ["_extract_word_image"], {"np": np})
        self._extract_word_image = types.MethodType(fns["_extract_word_image"], self)
