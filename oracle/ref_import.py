"""ORACLE helper — path-import of the reference's own torch-only modules.

Only usable where the reference tree exists (``REF_ROOT``), i.e. by ``tests/golden/make_golden.py``,
which stores what the reference computes as fixtures for the tests.  A normal
``import wild_visual_navigation`` fails here (pytorch_lightning / omegaconf / pandas are absent),
so stub packages are registered and the individual files are loaded with importlib, exactly as
SURVEY.md §8c describes.  Nothing is copied: the modules execute from the read-only tree.
"""
from __future__ import annotations

import importlib.util
import os
import sys
import types

REF_ROOT = os.environ.get("WVN_REFERENCE_ROOT", "/root/reference")


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "wild_visual_navigation"))


def _load(name: str, rel: str):
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF_ROOT, rel))
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def load():
    """Returns a namespace with the reference classes: Data, Batch, KalmanFilter,
    ConfidenceGenerator, SimpleMLP, TraversabilityLoss, SegmentExtractor."""
    if "wild_visual_navigation" in sys.modules and getattr(sys.modules["wild_visual_navigation"], "_wvn_stub", False):
        return sys.modules["wild_visual_navigation"]._ns
    root = types.ModuleType("wild_visual_navigation")
    root.__path__ = []
    root._wvn_stub = True
    root.WVN_ROOT_DIR = "/tmp/wvn_ref_root"
    sys.modules["wild_visual_navigation"] = root
    utils = types.ModuleType("wild_visual_navigation.utils")
    utils.__path__ = []
    sys.modules["wild_visual_navigation.utils"] = utils
    data = _load("wild_visual_navigation.utils.data", "wild_visual_navigation/utils/data.py")
    utils.Data, utils.Batch = data.Data, data.Batch
    kf = _load("wild_visual_navigation.utils.kalman_filter", "wild_visual_navigation/utils/kalman_filter.py")
    utils.KalmanFilter = kf.KalmanFilter
    cg = _load("wild_visual_navigation.utils.confidence_generator", "wild_visual_navigation/utils/confidence_generator.py")
    utils.ConfidenceGenerator = cg.ConfidenceGenerator
    loss = _load("wild_visual_navigation.utils.loss", "wild_visual_navigation/utils/loss.py")
    mlp = _load("wild_visual_navigation.model.simple_mlp", "wild_visual_navigation/model/simple_mlp.py")
    seg = _load(
        "wild_visual_navigation.feature_extractor.segment_extractor",
        "wild_visual_navigation/feature_extractor/segment_extractor.py",
    )
    ns = types.SimpleNamespace(
        Data=data.Data,
        Batch=data.Batch,
        KalmanFilter=kf.KalmanFilter,
        ConfidenceGenerator=cg.ConfidenceGenerator,
        TraversabilityLoss=loss.TraversabilityLoss,
        SimpleMLP=mlp.SimpleMLP,
        SegmentExtractor=seg.SegmentExtractor,
        root=REF_ROOT,
    )
    root._ns = ns
    return ns
