"""CPU tests of the learner -> inference weight hand-off file (SURVEY.md §8f rank 2): format compatibility with
the file the reference's learning node writes (golden ``tmp_state_dict.pt``, produced by the reference's own
classes) and the reader's change-detection semantics (wvn_feature_extractor_node.py:407-446)."""
import os

import torch

from wild_visual_navigation_b200.model.simple_mlp import SimpleMLP
from wild_visual_navigation_b200.utils import ConfidenceGenerator, read_tmp_state_dict, write_tmp_state_dict, TMP_STATE_DICT_NAME


def _pair(seed):
    torch.manual_seed(seed)
    return SimpleMLP(16, [8, 4, 1], True), ConfidenceGenerator(std_factor=0.5, method="latest_measurement")


def test_reads_the_file_the_reference_node_writes(golden_dir):
    path = os.path.join(golden_dir, "tmp_state_dict.pt")
    want = torch.load(path, weights_only=False)
    model, cg = _pair(0)
    flat_before = model.flat_params.data_ptr()
    assert read_tmp_state_dict(model, cg, path)
    for k, v in model.state_dict().items():
        assert torch.equal(v, want[k]), k
    assert model.flat_params.data_ptr() == flat_before  # kernels keep pointing at the same storage
    assert torch.equal(torch.cat([p.reshape(-1) for p in model.layers.parameters()]), model.flat_params)
    assert abs(cg.mean.item() - 0.37) < 1e-7 and abs(cg.std.item() - 0.21) < 1e-7 and abs(cg.var.item() - 0.0441) < 1e-7
    # same weights again -> "model has not changed" -> nothing loaded
    assert not read_tmp_state_dict(model, cg, path)


def test_roundtrip_and_change_detection(tmp_path):
    src_model, src_cg = _pair(1)
    with torch.no_grad():
        src_cg.mean[0], src_cg.std[0] = 0.5, 0.25
    f = write_tmp_state_dict(src_model, src_cg, str(tmp_path))  # directory -> .tmp_state_dict.pt inside it
    assert os.path.basename(f) == TMP_STATE_DICT_NAME and os.path.exists(f)
    dst_model, dst_cg = _pair(2)
    assert read_tmp_state_dict(dst_model, dst_cg, str(tmp_path))
    assert torch.equal(dst_model.flat_params, src_model.flat_params)
    assert dst_cg.mean.item() == 0.5 and dst_cg.std.item() == 0.25
    assert not read_tmp_state_dict(dst_model, dst_cg, f)          # unchanged
    assert not read_tmp_state_dict(dst_model, dst_cg, str(tmp_path / "missing.pt"))
    # a file from another model family (last key absent) is ignored
    torch.save({"something.else": torch.zeros(1)}, f)
    assert not read_tmp_state_dict(dst_model, dst_cg, f)


def _module_with_state(state_dict):
    """A module whose parameters have exactly the names, order and values of ``state_dict``."""
    root = torch.nn.Module()
    for name, v in state_dict.items():
        *path, leaf = name.split(".")
        m = root
        for p in path:
            if not hasattr(m, p):
                m.add_module(p, torch.nn.Module())
            m = getattr(m, p)
        m.register_parameter(leaf, torch.nn.Parameter(v.clone()))
    return root


def test_reference_classes_load_our_file(tmp_path, golden_dir):
    """The reference's inference node loads the hand-off file into its SimpleMLP with ``load_state_dict(strict=False)``;
    that model's parameter layout and init come from the reference's own class (golden ``simple_mlp_ref_state.pt``)."""
    model, cg = _pair(3)
    with torch.no_grad():
        cg.mean[0], cg.std[0] = 0.11, 0.07
    f = write_tmp_state_dict(model, cg, str(tmp_path))
    new_model_state_dict = torch.load(f, weights_only=False)
    ref_model = _module_with_state(torch.load(os.path.join(golden_dir, "simple_mlp_ref_state.pt")))
    k = list(ref_model.state_dict().keys())[-1]
    assert k in new_model_state_dict and (ref_model.state_dict()[k] != new_model_state_dict[k]).any()
    ref_model.load_state_dict(new_model_state_dict, strict=False)
    for name, v in ref_model.state_dict().items():
        assert torch.equal(v, model.state_dict()[name])
    c = new_model_state_dict["confidence_generator"]
    assert abs(c["mean"].item() - 0.11) < 1e-7 and abs(c["std"].item() - 0.07) < 1e-7 and tuple(c["var"].shape) == (1, 1)


def test_image_features_wire_roundtrip():
    """ImageFeatures.msg field layout (wvn_feature_extractor_node.py:373-393) and the learning node's decode
    (wvn_learning_node.py:651-656): bit-identical round trip."""
    from wild_visual_navigation_b200.utils import decode_image_features, encode_image_features

    g = torch.Generator().manual_seed(4)
    feat = torch.randn(7, 90, generator=g) * 3
    seg = torch.randint(0, 7, (24, 32), generator=g)
    msg = encode_image_features(feat, seg, header={"seq": 5, "frame_id": "cam"})
    dim = msg["features"]["layout"]["dim"]
    assert [(d["label"], d["size"], d["stride"]) for d in dim] == [("n", 7, 630), ("feat", 90, 90)]
    assert isinstance(msg["features"]["data"], list) and len(msg["features"]["data"]) == 630
    assert msg["feature_segments"]["step"] == 32 * 4 and len(msg["feature_segments"]["data"]) == 24 * 32 * 4
    f2, s2 = decode_image_features(msg)
    assert torch.equal(f2, feat) and torch.equal(s2.long(), seg) and s2.dtype == torch.int32
