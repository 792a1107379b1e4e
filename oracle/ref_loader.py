"""Loader for the UNMODIFIED reference hot-path modules (test infrastructure only).

This file is part of ``oracle/`` — the checker, never the product.  It imports the
reference's own Python files (``REF_ROOT``) *by file path* so that

  * ``oracle/make_golden.py`` can generate the golden vectors in ``tests/golden/`` and
  * ``tests/test_oracle_vs_reference.py`` can pin the numpy restatement (``oracle/np_oracle.py``)
    against the executed reference (skipped when the reference tree is absent).

Nothing under ``litehandnet_b200/`` imports this module.

Why by file path: site-packages holds HuggingFace ``datasets`` which shadows the reference's
``datasets/`` namespace package, and several reference modules import names that no longer exist
(``config.DATASET``, ``config.config_dict``) or third-party modules that are absent here
(``addict``, ``matplotlib``, ``mmcv``, ``munkres``) — none of which take part in the hot-path
arithmetic (SURVEY.md §8c).
"""
import importlib.util
import os
import sys
import types

# the original project's source tree: LHN_REFERENCE_ROOT, else the copy oracle/build_ref.py stages in oracle/_ref
REF_ROOT = os.environ.get("LHN_REFERENCE_ROOT", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))

_LOADED = {}


def available():
    return os.path.isdir(os.path.join(REF_ROOT, "utils"))


class _AttrDict(dict):
    """Minimal stand-in for addict.Dict (attribute access + .get)."""

    def __init__(self, *a, **k):
        super().__init__()
        for key, val in dict(*a, **k).items():
            self[key] = _AttrDict(val) if isinstance(val, dict) else val

    def __getattr__(self, key):
        try:
            return self[key]
        except KeyError:
            return _AttrDict()

    def __setattr__(self, key, val):
        self[key] = val


def _stub(name, **attrs):
    if name in sys.modules and not getattr(sys.modules[name], "__lhn_stub__", False):
        return sys.modules[name]
    m = types.ModuleType(name)
    m.__lhn_stub__ = True
    for k, v in attrs.items():
        setattr(m, k, v)
    sys.modules[name] = m
    return m


def _shell(name):
    """Register an empty package shell (shadows e.g. HuggingFace ``datasets``)."""
    m = types.ModuleType(name)
    m.__path__ = []
    m.__lhn_shell__ = True
    sys.modules[name] = m
    return m


def _load(dotted, relpath):
    if dotted in _LOADED:
        return _LOADED[dotted]
    path = os.path.join(REF_ROOT, relpath)
    spec = importlib.util.spec_from_file_location(dotted, path)
    mod = importlib.util.module_from_spec(spec)
    sys.modules[dotted] = mod
    spec.loader.exec_module(mod)
    _LOADED[dotted] = mod
    parent, _, leaf = dotted.rpartition(".")
    if parent and parent in sys.modules:
        setattr(sys.modules[parent], leaf, mod)
    return mod


class Ref:
    """Namespace holding the loaded reference modules."""


def load():
    """Load every hot-path module of the reference.  Returns a namespace:

    ref.loss (package), ref.generateTarget, ref.generate_simder, ref.post_transforms,
    ref.heatmap_post_processing, ref.evaluation, ref.top_down_eval, ref.decoder, ref.transforms,
    ref.result_parser, ref.SPheatmapParser, ref.HeatmapParser, ref.config
    """
    if "ref" in _LOADED:
        return _LOADED["ref"]
    if not available():
        raise RuntimeError(f"reference tree not found at {REF_ROOT}")

    saved = {k: sys.modules.get(k) for k in ("datasets", "utils", "config", "loss")}

    try:
        import matplotlib  # noqa: F401
    except Exception:
        _stub("matplotlib", rc=lambda *a, **k: None)
    try:
        import addict  # noqa: F401
    except Exception:
        _stub("addict", Dict=_AttrDict)
    try:
        import mmcv  # noqa: F401
    except Exception:
        _stub("mmcv")
    try:
        import munkres  # noqa: F401
    except Exception:
        _stub("munkres", Munkres=object)

    for pkg in ("datasets", "datasets.data_pipeline", "utils", "utils.post_processing",
                "utils.post_processing.evaluation"):
        _shell(pkg)

    ref = Ref()
    ref.config = _load("config", "config/__init__.py")
    # injected dummies for names the legacy parsers import but config/ no longer defines
    ref.config.DATASET = {}
    ref.config.config_dict = {}
    ref.post_transforms = _load("datasets.data_pipeline.post_transforms",
                                "datasets/data_pipeline/post_transforms.py")
    ref.generateTarget = _load("datasets.data_pipeline.generateTarget",
                               "datasets/data_pipeline/generateTarget.py")
    ref.generate_simder = _load("datasets.data_pipeline.generate_simder",
                                "datasets/data_pipeline/generate_simder.py")
    ref.bbox_metric = _load("utils.bbox_metric", "utils/bbox_metric.py")
    ref.heatmap_post_processing = _load("utils.heatmap_post_processing",
                                        "utils/heatmap_post_processing.py")
    ref.evaluation = _load("utils.evaluation", "utils/evaluation.py")
    ref.top_down_eval = _load("utils.post_processing.evaluation.top_down_eval",
                              "utils/post_processing/evaluation/top_down_eval.py")
    ref.decoder = _load("utils.post_processing.decoder", "utils/post_processing/decoder.py")
    ref.transforms = _load("utils.transforms", "utils/transforms.py")
    ref.result_parser = _load("utils.result_parser", "utils/result_parser.py")
    ref.SPheatmapParser = _load("utils.SPheatmapParser", "utils/SPheatmapParser.py")
    ref.HeatmapParser = _load("utils.HeatmapParser", "utils/HeatmapParser.py")

    # loss/ is a regular package; load it under a private name so it cannot collide
    spec = importlib.util.spec_from_file_location(
        "loss", os.path.join(REF_ROOT, "loss/__init__.py"),
        submodule_search_locations=[os.path.join(REF_ROOT, "loss")])
    loss_pkg = importlib.util.module_from_spec(spec)
    sys.modules["loss"] = loss_pkg
    spec.loader.exec_module(loss_pkg)
    ref.loss = loss_pkg

    # un-shadow the packages we displaced so the rest of the process is unaffected
    ref._modules = {k: sys.modules.get(k) for k in list(sys.modules)
                    if k.split(".")[0] in ("datasets", "utils", "config", "loss")}
    for k in list(sys.modules):
        if k.split(".")[0] in ("datasets", "utils", "config", "loss"):
            del sys.modules[k]
    for k, v in saved.items():
        if v is not None:
            sys.modules[k] = v

    # bbox_metric.py changed global print options and cv2 threading at import; keep the cv2
    # setting (it is the reference's behaviour) but restore numpy/torch print options.
    import numpy as np
    import torch
    np.set_printoptions(linewidth=75, formatter=None)
    torch.set_printoptions(profile="default")

    ref.AttrDict = _AttrDict
    _LOADED["ref"] = ref
    return ref


def make_result_parser(ref, image_size=(256, 256), hm_size=(64, 64), dark=False, k=2):
    """ResultParser without running its heavy __init__ dependencies on missing cfg keys
    (utils/result_parser.py:19-48)."""
    cfg = dict(image_size=list(image_size), hm_size=list(hm_size), model="litehandnet",
               simdr_split_ratio=k, bbox_alpha=1.0, with_region_map=False,
               cycle_detection_reduction=1, DARK=dark)
    return ref.result_parser.ResultParser(cfg)


if __name__ == "__main__":
    r = load()
    print("loaded:", [k for k in vars(r) if not k.startswith("_")])
