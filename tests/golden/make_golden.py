"""Generate the golden fixtures in tests/golden/ by running the REFERENCE's own code.

Run in the build container (``/root/reference`` present):  ``python tests/golden/make_golden.py``

The reference is pure Python; its torch-only modules are path-imported from the read-only tree
(oracle/ref_import.py) and executed on seeded inputs.  The results are stored as small fixtures
so that the GPU box (which has no ``/root/reference``) can still check the oracle — and through
it the CUDA path — against what the reference computes.

Fixtures
  mlp_train.pt      reference SimpleMLP + TraversabilityLoss + torch.optim.Adam, 3 steps (small dims)
  mlp_init_384.pt   checksum of the seed-42 init of the real-size SimpleMLP(384,[256,32,1],True)
  confidence.pt     ConfidenceGenerator.inference_without_update / update (latest_measurement)
  supervision.pt    MissionNode.update_supervision_signal (the reference's method source, executed from the reference file)
  sparsify.pt       FeatureExtractor.sparsify_features (loop + cumsum variants) and segment_stego's relabel loop,
                    the reference's method sources executed from the reference file
  checkpoint_ref.pt a checkpoint as TraversabilityEstimator.save_checkpoint writes it, from the reference's classes
  tmp_state_dict.pt the weight hand-off file as wvn_learning_node.py:381-394 writes it (reference SimpleMLP + ConfidenceGenerator)
  simple_mlp_ref_state.pt  state dict of a fresh reference SimpleMLP(16, [8, 4, 1], True), the model the hand-off
                    file is loaded into
  segments.npz      reference SegmentExtractor on a synthetic map + the reference's shipped
                    known-answer assets/graph/{seg,center}.pt and graph.pt edge_index
  extract_stego.pt  reference FeatureExtractor.extract end to end (stego segmentation + stego features) over the
                    shimmed StegoInterface and the reference SegmentExtractor
  stego_wrapper.pt  reference StegoInterface.inference (its real transform / interpolation code) around a shim Stego
                    model made of the oracle's restated head + backbone (tiny config)
  dino_wrapper.pt   reference DinoInterface.inference (its real transform / upsample code) wrapped
                    around the oracle's restated ViT (tiny config) via omegaconf/stego shims
"""
from __future__ import annotations

import io
import os
import sys
import types

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import ref_import  # noqa: E402
from oracle.dino_vit import ViTConfig, synthetic_state_dict, vit_feature_map  # noqa: E402


def make_mlp_train(ns):
    D, hidden = 32, [16, 8, 1]
    torch.manual_seed(42)
    model = ns.SimpleMLP(D, list(hidden), True)
    init_sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    loss_fn = ns.TraversabilityLoss(
        w_trav=0.03, w_reco=0.5, w_temp=0.0, anomaly_balanced=True, model=model, method="latest_measurement",
        confidence_std_factor=0.5, log_enabled=False, log_folder="/tmp",
    )
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    g = torch.Generator().manual_seed(7)
    R = 96
    x = torch.randn(R, D, generator=g)
    y_valid = torch.rand(R, generator=g) < 0.25
    y = torch.where(y_valid, torch.rand(R, generator=g).clamp(min=0.001), torch.zeros(R))
    steps = []
    for step in range(3):
        graph = ns.Data(x=x, y=y, y_valid=y_valid)
        res = model(graph)
        loss, aux, _ = loss_fn(graph, res, step=step, log_step=False)
        opt.zero_grad()
        loss.backward()
        grads = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
        opt.step()
        steps.append(
            {
                "loss_total": loss.item(),
                "loss_trav": aux["loss_trav"].item(),
                "loss_reco": aux["loss_reco"].item(),
                "loss_trav_confidence": aux["loss_trav_confidence"].item(),
                "confidence": aux["confidence"].detach().clone(),
                "cg_mean": loss_fn._confidence_generator.mean.detach().clone(),
                "cg_std": loss_fn._confidence_generator.std.detach().clone(),
                "grads": grads,
                "state_dict": {k: v.detach().clone() for k, v in model.state_dict().items()},
            }
        )
    # forward of the final model on fresh rows (inference semantics incl. in-place sigmoid)
    xq = torch.randn(10, D, generator=g)
    with torch.no_grad():
        pred = model(ns.Data(x=xq.clone()))
    torch.save(
        {"dim": D, "hidden": hidden, "init_state_dict": init_sd, "x": x, "y": y, "y_valid": y_valid, "steps": steps,
         "xq": xq, "pred": pred},
        os.path.join(HERE, "mlp_train.pt"),
    )


def make_mlp_init(ns):
    torch.manual_seed(42)
    model = ns.SimpleMLP(384, [256, 32, 1], True)
    sd = model.state_dict()
    torch.save(
        {"sums": {k: v.double().sum().item() for k, v in sd.items()},
         "abs_sums": {k: v.double().abs().sum().item() for k, v in sd.items()},
         "shapes": {k: tuple(v.shape) for k, v in sd.items()},
         "first8": {k: v.flatten()[:8].clone() for k, v in sd.items()}},
        os.path.join(HERE, "mlp_init_384.pt"),
    )


def make_handoff(ns):
    """.tmp_state_dict.pt exactly as the reference's learning node writes it (wvn_learning_node.py:381-394),
    from the reference's own SimpleMLP / ConfidenceGenerator (small dims)."""
    torch.manual_seed(7)
    model = ns.SimpleMLP(16, [8, 4, 1], True)
    cg = ns.ConfidenceGenerator(std_factor=0.5, method="latest_measurement")
    with torch.no_grad():
        cg.mean[0], cg.std[0], cg.var[0, 0] = 0.37, 0.21, 0.0441
    new_model_state_dict = model.state_dict()
    new_model_state_dict["confidence_generator"] = cg.get_dict()
    torch.save(new_model_state_dict, os.path.join(HERE, "tmp_state_dict.pt"))


def make_reference_mlp_state(ns):
    """State dict of a freshly built reference SimpleMLP(16, [8, 4, 1], True): the parameter names, order, shapes and
    init values the reference's inference node loads a hand-off file into."""
    torch.manual_seed(5)
    torch.save(ns.SimpleMLP(16, [8, 4, 1], True).state_dict(), os.path.join(HERE, "simple_mlp_ref_state.pt"))


def make_checkpoint(ns):
    """last_checkpoint.pt exactly as TraversabilityEstimator.save_checkpoint writes it
    (traversability_estimator.py:377-399: step / model_state_dict / optimizer_state_dict /
    traversability_loss_state_dict / loss) from the reference's own SimpleMLP, TraversabilityLoss (which registers the
    model as a sub-module: its state dict carries ``_model.layers.*``) and torch.optim.Adam after two steps."""
    torch.manual_seed(42)
    model = ns.SimpleMLP(16, [8, 4, 1], True)   # small dims: the FORMAT is what this fixture pins
    loss_fn = ns.TraversabilityLoss(w_trav=0.03, w_reco=0.5, w_temp=0.0, anomaly_balanced=True, model=model,
                                    method="latest_measurement", confidence_std_factor=0.5, log_enabled=False,
                                    log_folder="/tmp")
    opt = torch.optim.Adam(model.parameters(), lr=1e-3)
    g = torch.Generator().manual_seed(11)
    x = torch.randn(48, 16, generator=g)
    yv = torch.rand(48, generator=g) < 0.3
    y = torch.where(yv, torch.rand(48, generator=g).clamp(min=0.001), torch.zeros(48))
    loss = None
    for step in range(2):
        graph = ns.Data(x=x, y=y, y_valid=yv)
        loss, _, _ = loss_fn(graph, model(graph), step=step, log_step=False)
        opt.zero_grad()
        loss.backward()
        opt.step()
    torch.save({"step": 2, "model_state_dict": model.state_dict(), "optimizer_state_dict": opt.state_dict(),
                "traversability_loss_state_dict": loss_fn.state_dict(), "loss": loss.item()},
               os.path.join(HERE, "checkpoint_ref.pt"))
    torch.save({"x": x, "y": y, "y_valid": yv}, os.path.join(HERE, "checkpoint_ref_batch.pt"))


def make_supervision():
    """Runs the reference's OWN ``MissionNode.update_supervision_signal`` (nodes.py:400-440).  nodes.py cannot be
    imported here (liegroups / kornia / networkx are absent), so the method's source is taken from the reference
    file with ``ast`` and executed against a bare namespace object — nothing is copied into this repository."""
    import ast

    path = os.path.join(ref_import.REF_ROOT, "wild_visual_navigation/traversability_estimator/nodes.py")
    src = open(path).read()
    fn = next(n for n in ast.walk(ast.parse(src)) if isinstance(n, ast.FunctionDef) and n.name == "update_supervision_signal")
    import textwrap

    code = "import torch\n" + textwrap.dedent("\n".join(src.splitlines()[fn.lineno - 1 : fn.end_lineno]))
    scope = {}
    exec(compile(code, path, "exec"), scope)
    g = torch.Generator().manual_seed(13)
    seg = synthetic_segments(48, 48, 9, seed=6).long()
    mask = torch.rand(3, 48, 48, generator=g)
    mask[torch.rand(3, 48, 48, generator=g) < 0.55] = float("nan")
    mask[:, seg == 4] = float("nan")       # one segment without any label
    mask[1:, seg == 2] = float("nan")      # one segment labelled in a single channel only
    node = types.SimpleNamespace(_supervision_mask=mask.clone(), _features=torch.zeros(9, 4), _feature_segments=seg.clone())
    scope["update_supervision_signal"](node)
    torch.save({"seg": seg, "mask": mask, "signal": node._supervision_signal, "valid": node._supervision_signal_valid},
               os.path.join(HERE, "supervision.pt"))


def make_image_projector():
    """Runs the reference's OWN ``ImageProjector`` (image_projector/image_projector.py:16-200: scaled camera matrix,
    project / check_validity, project_and_render, resize_image) and ``make_polygon_from_points`` (utils/meshes.py:156-165).
    kornia / liegroups / pytictac are absent here, so the three kornia routines the class calls are provided by the
    oracle's restatement (oracle/image_projector.py, [EXTERNAL-RECALLED]) through stub modules: the golden pins the
    reference's in-repo logic; the kornia part stays unpinned against kornia itself."""
    import importlib.util
    from oracle import image_projector as oip

    class _PinholeCamera:
        def __init__(self, intrinsics, extrinsics, height, width):
            self.intrinsics, self.extrinsics, self.height, self.width = intrinsics, extrinsics, height, width

        batch_size = property(lambda self: self.intrinsics.shape[0])
        camera_matrix = property(lambda self: self.intrinsics[..., :3, :3])

        def project(self, point_3d):
            P = self.intrinsics @ self.extrinsics
            return oip.convert_points_from_homogeneous(oip.transform_points(P, point_3d))

    def _mod(name, **attrs):
        m = types.ModuleType(name)
        m.__dict__.update(attrs)
        sys.modules[name] = m
        return m

    names = ["pytictac", "kornia", "kornia.geometry", "kornia.geometry.camera", "kornia.geometry.camera.pinhole",
             "kornia.geometry.linalg", "kornia.utils", "kornia.utils.draw", "liegroups", "liegroups.torch"]
    _mod("pytictac", Timer=object)
    for n in names[1:]:
        _mod(n)
    sys.modules["kornia.geometry.camera.pinhole"].PinholeCamera = _PinholeCamera
    sys.modules["kornia.geometry.linalg"].transform_points = oip.transform_points
    sys.modules["kornia.utils.draw"].draw_convex_polygon = oip.draw_convex_polygon
    sys.modules["liegroups.torch"].SE3 = sys.modules["liegroups.torch"].SO3 = object
    spec = importlib.util.spec_from_file_location(
        "ref_image_projector", os.path.join(ref_import.REF_ROOT, "wild_visual_navigation/image_projector/image_projector.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    spec = importlib.util.spec_from_file_location(
        "ref_meshes", os.path.join(ref_import.REF_ROOT, "wild_visual_navigation/utils/meshes.py"))
    meshes = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(meshes)

    B = 7
    K, poses, fp = oip.synthetic_footprints(B, seed=3, image=48)
    K[:, 0, 0] *= 1.1            # fx != fy: the square-crop branch of the constructor overwrites fx with fy * s
    K[:, 0, 2] += 12             # 48 x 72 camera, principal point off-centre
    corners = torch.tensor([[0.4, 0.3, 0.0], [0.4, -0.3, 0.0], [1.3, -0.35, 0.0], [1.3, 0.25, 0.0]])
    poly_ref = meshes.make_polygon_from_points(corners, grid_size=10)
    out = {"K": K, "poses": poses, "corners": corners, "polygon": poly_ref, "h": 48, "w": 72}
    g = torch.Generator().manual_seed(5)
    img = torch.rand(2, 3, 48, 72, generator=g)
    for tag, kw in (("square", dict(new_h=32)), ("rect", dict(new_h=24, new_w=40)), ("native", dict())):
        im = mod.ImageProjector(K.clone(), torch.tensor(48), torch.tensor(72), **kw)
        colors = torch.tensor([0.0, 1.0, 0.5]) if tag == "rect" else torch.ones(3)
        masks, _, proj, valid = im.project_and_render(poses.clone(), fp.clone(), colors)
        out[tag] = {"kw": kw, "sK": im.camera.intrinsics.clone(), "colors": colors, "masks": masks.clone(),
                    "projected": proj.clone(), "valid": valid.clone(), "resized": im.resize_image(img)}
    out["img"] = img
    torch.save(out, os.path.join(HERE, "image_projector.pt"))
    for n in names:
        sys.modules.pop(n, None)


def _reference_method(rel_path, name):
    """A method of a reference class whose module cannot be imported here: its source is read from the reference file
    with ``ast`` and compiled as a free function (nothing is copied into this repository)."""
    import ast
    import textwrap

    path = os.path.join(ref_import.REF_ROOT, rel_path)
    src = open(path).read()
    fn = next(n for n in ast.walk(ast.parse(src)) if isinstance(n, ast.FunctionDef) and n.name == name)
    code = "import torch\n" + textwrap.dedent("\n".join(src.splitlines()[fn.lineno - 1 : fn.end_lineno]))
    scope = {}
    exec(compile(code, path, "exec"), scope)
    return scope[name]


def make_sparsify():
    """The reference's OWN ``FeatureExtractor.sparsify_features`` (default loop and cumsum variant,
    feature_extractor.py:310-398) and the relabel loop of ``segment_stego`` (:237-249)."""
    fe = "wild_visual_navigation/feature_extractor/feature_extractor.py"
    sparsify, segment_stego = _reference_method(fe, "sparsify_features"), _reference_method(fe, "segment_stego")
    g = torch.Generator().manual_seed(17)
    seg = synthetic_segments(24, 24, 5, seed=8).long()
    dense = torch.randn(1, 6, 24, 24, generator=g)
    me = types.SimpleNamespace(_feature_type="dino", _segmentation_type="stego")
    feat = sparsify(me, dense, seg)
    feat_cumsum = sparsify(me, dense.clone(), seg.clone(), cumsum_trick=True)
    # cluster ids as the STEGO probe emits them (arbitrary subset of 0..26), relabelled to 0..S-1
    labels = torch.tensor([3, 7, 19, 20, 26])
    raw = labels[seg][None, None]
    extractor = types.SimpleNamespace(inference=lambda img: None, cluster_segments=raw.clone())
    me2 = types.SimpleNamespace(_extractor=extractor, _device="cpu")
    relabelled = segment_stego(me2, torch.zeros(1, 3, 24, 24))
    torch.save({"dense": dense, "seg": seg, "feat": feat, "feat_cumsum": feat_cumsum, "raw_clusters": raw,
                "relabelled": relabelled}, os.path.join(HERE, "sparsify.pt"))


def make_confidence(ns):
    cg = ns.ConfidenceGenerator(std_factor=0.5, method="latest_measurement")
    g = torch.Generator().manual_seed(11)
    x = torch.rand(200, generator=g) * 2.0
    xp = x[:40]
    with torch.no_grad():
        conf_update = cg.update(x, xp, step=0)
        mean, std = cg.mean.detach().clone(), cg.std.detach().clone()
        conf_infer = cg.inference_without_update(x * 1.3)
    # zero-interval-at-zero clamp case: mean small so that lo clamps to 0
    cg2 = ns.ConfidenceGenerator(std_factor=1.0, method="latest_measurement")
    with torch.no_grad():
        cg2.mean[0], cg2.std[0] = 0.05, 0.2
        conf_clamped = cg2.inference_without_update(x)
    torch.save(
        {"x": x, "x_positive": xp, "conf_update": conf_update, "mean": mean, "std": std, "conf_infer": conf_infer,
         "conf_clamped": conf_clamped},
        os.path.join(HERE, "confidence.pt"),
    )


def make_confidence_methods(ns):
    """The reference's OWN ConfidenceGenerator for all four methods (confidence_generator.py:78-145): five consecutive
    ``update`` calls with growing / shrinking positive sets, including an empty one for the Kalman filter."""
    g = torch.Generator().manual_seed(23)
    seq = []
    for i, (n, npos) in enumerate(((300, 50), (280, 31), (310, 2), (290, 77), (305, 40), (300, 64), (150, 9))):
        x = torch.rand(n, generator=g) * (1.5 + 0.3 * i) + 0.05 * i
        pos = torch.rand(n, generator=g) < npos / n
        pos[:2] = True
        seq.append((x, pos))
    out = {"seq": seq, "std_factor": 0.5}
    for method in ("latest_measurement", "running_mean", "moving_average", "kalman_filter"):
        cg = ns.ConfidenceGenerator(std_factor=0.5, method=method)
        steps = []
        with torch.no_grad():
            for i, (x, pos) in enumerate(seq):
                xp = x[pos] if not (method == "kalman_filter" and i == 2) else x[:0]   # empty positives: KF keeps its state
                conf = cg.update(x, xp, step=i)
                steps.append({"conf": conf.clone(), "mean": cg.mean.detach().clone(), "std": cg.std.detach().clone(),
                              "var": cg.var.detach().clone()})
        out[method] = steps
        out[method + "_keys"] = sorted(cg.state_dict().keys())
    torch.save(out, os.path.join(HERE, "confidence_methods.pt"))


def synthetic_segments(h=48, w=48, n=9, seed=5):
    g = torch.Generator().manual_seed(seed)
    cy = torch.rand(n, generator=g) * h
    cx = torch.rand(n, generator=g) * w
    yy, xx = torch.meshgrid(torch.arange(h).float(), torch.arange(w).float(), indexing="ij")
    d = (yy[None] - cy[:, None, None]) ** 2 + (xx[None] - cx[:, None, None]) ** 2
    return d.argmin(0)


def make_segments(ns):
    se = ns.SegmentExtractor()
    seg = synthetic_segments()[None, None]
    edges = se.adjacency_list(seg)
    cent = se.centers(seg)
    out = {"syn_seg": seg[0, 0].numpy().astype(np.uint8), "syn_edges": edges.numpy(), "syn_centers": cent.numpy()}
    # shipped known-answer fixture of the reference (SURVEY.md §8c): assets/graph/{seg,center}.pt, graph.pt
    adir = os.path.join(ns.root, "assets", "graph")
    aseg = torch.load(os.path.join(adir, "seg.pt"), map_location="cpu")
    acen = torch.load(os.path.join(adir, "center.pt"), map_location="cpu")
    out["asset_seg"] = aseg.numpy().astype(np.uint8)
    out["asset_centers"] = acen.numpy()
    # graph.pt pickles a torch_geometric Data: unpickle with a stub class
    tg = types.ModuleType("torch_geometric"); tgd = types.ModuleType("torch_geometric.data")
    tgdd = types.ModuleType("torch_geometric.data.data"); tgds = types.ModuleType("torch_geometric.data.storage")

    class _Any:
        def __init__(self, *a, **k): pass
        def __setstate__(self, st): self.__dict__.update(st if isinstance(st, dict) else {"state": st})

    def _mod_getattr(name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Any

    for m in (tgdd, tgds, tgd):
        m.__getattr__ = _mod_getattr  # type: ignore
    for name in ("Data", "DataEdgeAttr", "DataTensorAttr", "GlobalStorage"):
        setattr(tgdd, name, type(name, (_Any,), {}))
        setattr(tgds, name, type(name, (_Any,), {}))
    sys.modules.update({"torch_geometric": tg, "torch_geometric.data": tgd, "torch_geometric.data.data": tgdd,
                        "torch_geometric.data.storage": tgds})
    try:
        graph = torch.load(os.path.join(adir, "graph.pt"), map_location="cpu", weights_only=False)

        def find(obj, key, depth=0):
            if depth > 6: return None
            d = getattr(obj, "__dict__", obj if isinstance(obj, dict) else None)
            if not isinstance(d, dict): return None
            if key in d and torch.is_tensor(d[key]): return d[key]
            for v in d.values():
                r = find(v, key, depth + 1)
                if r is not None: return r
            return None

        ei = find(graph, "edge_index")
        if ei is not None:
            out["asset_edge_index"] = ei.numpy()
    except Exception as e:  # pragma: no cover
        print("graph.pt not decodable:", e)
    finally:
        for k in ("torch_geometric", "torch_geometric.data", "torch_geometric.data.data", "torch_geometric.data.storage"):
            sys.modules.pop(k, None)
    # reference outputs on its own asset (what the restatement must reproduce)
    out["asset_ref_edges"] = se.adjacency_list(aseg[None, None]).numpy()
    out["asset_ref_centers"] = se.centers(aseg[None, None]).numpy()
    np.savez_compressed(os.path.join(HERE, "segments.npz"), **out)


def make_dino_wrapper():
    # shims for the two absent imports of dino_interface.py
    class _Cfg(dict):
        def is_empty(self): return len(self) == 0
        __getattr__ = dict.__getitem__

    om = types.ModuleType("omegaconf")
    om.OmegaConf = types.SimpleNamespace(create=lambda d: _Cfg(d))
    sys.modules["omegaconf"] = om
    cfg = ViTConfig(image_size=32, patch_size=8, dim=32, depth=2, heads=2, mlp_dim=64, pretrain_grid=2)
    sd = synthetic_state_dict(cfg, seed=21, attn_std=0.3)

    class _Backbone(torch.nn.Module):
        def forward(self, x): return vit_feature_map(x, sd, cfg)

    st = types.ModuleType("stego"); stb = types.ModuleType("stego.backbones"); stbb = types.ModuleType("stego.backbones.backbone")
    stbb.get_backbone = lambda c: _Backbone()
    sys.modules.update({"stego": st, "stego.backbones": stb, "stego.backbones.backbone": stbb})
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "ref_dino_interface", os.path.join(ref_import.REF_ROOT, "wild_visual_navigation/feature_extractor/dino_interface.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    di = mod.DinoInterface(device="cpu", backbone="dino", input_size=32, backbone_type="vit_small", patch_size=8)
    g = torch.Generator().manual_seed(9)
    img = torch.rand(1, 3, 40, 52, generator=g)
    out = di.inference(img.clone())
    img2 = torch.rand(2, 3, 32, 32, generator=g)
    out2 = di.inference(img2.clone())
    torch.save({"vit_seed": 21, "attn_std": 0.3, "cfg": cfg.__dict__, "img": img, "out": out, "img2": img2, "out2": out2},
               os.path.join(HERE, "dino_wrapper.pt"))


def make_extract(ns, stego_interface, cfg):
    """End to end: the reference's OWN ``FeatureExtractor.extract`` orchestration (extract / compute_segments /
    segment_stego / compute_features / compute_stego / sparsify_features, feature_extractor.py:95-128,151-177,237-271,
    310-398 — method sources compiled from the reference file) over the reference's StegoInterface (shimmed external
    nets) and the reference's SegmentExtractor, configuration segmentation_type = feature_type = "stego"."""
    fe = "wild_visual_navigation/feature_extractor/feature_extractor.py"
    names = ["extract", "compute_segments", "segment_stego", "compute_features", "compute_stego", "sparsify_features"]
    cls = type("RefFeatureExtractor", (), {n: _reference_method(fe, n) for n in names})
    me = cls()
    me._device, me._segmentation_type, me._feature_type, me._input_size = "cpu", "stego", "stego", cfg.image_size
    me._stego_features_already_computed_in_segmentation = False
    me.segment_extractor = ns.SegmentExtractor()
    me._extractor = stego_interface
    g = torch.Generator().manual_seed(12)
    img = torch.rand(1, 3, 32, 32, generator=g)
    edges, feat, seg, center, dense = me.extract(img, return_dense_features=True)
    torch.save({"img": img, "edges": edges, "feat": feat, "seg": seg, "center": center, "dense": dense},
               os.path.join(HERE, "extract_stego.pt"))


def make_stego_wrapper(ns):
    """The reference's own ``StegoInterface.inference`` (stego_interface.py:73-111: transform, code -> bilinear
    align_corners=True to (H, H), predictions -> nearest (H, H) int, return order) around a shim ``Stego`` model whose
    ``get_code`` / ``postprocess`` are the oracle's restated head on the oracle's restated backbone."""
    from oracle import stego_head

    cfg = ViTConfig(image_size=32, patch_size=8, dim=32, depth=2, heads=2, mlp_dim=64, pretrain_grid=2)
    sd = synthetic_state_dict(cfg, seed=21, attn_std=0.3)
    hd = stego_head.synthetic_head(32, code_dim=10, n_clusters=6, n_classes=5, seed=4)

    class _Stego(torch.nn.Module):
        def get_code(self, img):  # Stego.get_code: horizontal-flip TTA
            code = stego_head.head_code(vit_feature_map(img, sd, cfg), hd)
            code_f = stego_head.head_code(vit_feature_map(img.flip(dims=[3]), sd, cfg), hd)
            return (code + code_f.flip(dims=[3])) / 2

        def postprocess(self, code, img, use_crf_cluster, use_crf_linear, image_clustering):
            assert not (use_crf_cluster or use_crf_linear or image_clustering)
            return stego_head.postprocess(code, tuple(img.shape[-2:]), hd)

        @classmethod
        def load_from_checkpoint(cls, path, n_image_clusters=None):
            return cls()

    class _Cfg(dict):
        def is_empty(self): return len(self) == 0
        __getattr__ = dict.__getitem__

    om = types.ModuleType("omegaconf")
    om.OmegaConf = types.SimpleNamespace(create=lambda d: _Cfg(d))
    pt = types.ModuleType("pytictac"); pt.Timer = object
    st = types.ModuleType("stego"); st.STEGO_ROOT_DIR = "/nonexistent"
    sts = types.ModuleType("stego.stego"); sts.Stego = _Stego
    std = types.ModuleType("stego.data"); std.create_cityscapes_colormap = lambda: None
    sys.modules.update({"omegaconf": om, "pytictac": pt, "stego": st, "stego.stego": sts, "stego.data": std})
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        "ref_stego_interface", os.path.join(ref_import.REF_ROOT, "wild_visual_navigation/feature_extractor/stego_interface.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    si = mod.StegoInterface(device="cpu", input_size=32, n_image_clusters=6, run_crf=False, run_clustering=False)
    make_extract(ns, si, cfg)
    g = torch.Generator().manual_seed(10)
    img = torch.rand(2, 3, 40, 52, generator=g)  # non-square: the transform resizes (NEAREST) and crops
    linear, cluster = si.inference(img.clone())
    torch.save({"vit_seed": 21, "attn_std": 0.3, "cfg": cfg.__dict__, "head_seed": 4, "head_dims": (32, 10, 6, 5),
                "img": img, "linear": linear, "cluster": cluster, "features": si.features},
               os.path.join(HERE, "stego_wrapper.pt"))
    for k in ("omegaconf", "pytictac", "stego", "stego.stego", "stego.data"):
        sys.modules.pop(k, None)


if __name__ == "__main__":
    assert ref_import.available(), "needs /root/reference"
    ns = ref_import.load()
    make_mlp_train(ns)
    make_mlp_init(ns)
    make_confidence(ns)
    make_confidence_methods(ns)
    make_handoff(ns)
    make_reference_mlp_state(ns)
    make_checkpoint(ns)
    make_supervision()
    make_image_projector()
    make_sparsify()
    make_segments(ns)
    make_dino_wrapper()
    make_stego_wrapper(ns)
    for f in sorted(os.listdir(HERE)):
        print(f, os.path.getsize(os.path.join(HERE, f)))
