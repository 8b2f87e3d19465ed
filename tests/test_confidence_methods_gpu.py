"""GPU parity of the fused train step under every ConfidenceGenerator method (utils/confidence_generator.py:49-145):
TraversabilityEstimator configured with running_mean / kalman_filter / moving_average (and the default) against the
oracle's autograd + Adam step driven by the oracle's ConfidenceState, which tests/test_oracle.py pins to the reference's
own class.  Tolerance: the train step's 2e-5 (relative) of tests/test_path_gpu.py; confidence per row 1e-4 absolute.
"""
import pytest
import torch

pytestmark = pytest.mark.gpu


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30)).item()


@pytest.mark.parametrize("method", ["latest_measurement", "running_mean", "kalman_filter", "moving_average"])
def test_fused_train_step_confidence_methods_vs_oracle(method):
    from oracle import wvn_path
    from wild_visual_navigation_b200 import TraversabilityEstimator
    from wild_visual_navigation_b200.traversability_estimator.traversability_estimator import default_params

    params = default_params()
    params["loss"]["method"] = method
    te = TraversabilityEstimator(params=params, device="cuda", min_samples_for_training=0, max_rows=512)
    cg_mod = te._traversability_loss._confidence_generator
    assert cg_mod.method == method
    sd = wvn_path.mlp_init(384, (256, 32), seed=42)
    cg = wvn_path.ConfidenceState(0.5, method)
    opt_state = None
    g = torch.Generator().manual_seed(31)
    for step in range(7):          # > 5 steps: the moving-average window wraps around
        n = 200 + 37 * step
        x = torch.randn(n, 384, generator=g) * (1.0 + 0.2 * step)
        y, yv = wvn_path.synthetic_supervision(n, seed=40 + step, p_valid=0.2)
        if method == "kalman_filter" and step == 3:
            yv = torch.zeros_like(yv)     # no positive sample: the filter keeps its state (confidence_generator.py:133)
            y = torch.zeros_like(y)
        conf = te._trainer.step(x.cuda(), y.cuda(), yv.cuda())
        m = te._trainer.metrics.tolist()
        if method == "kalman_filter" and step == 3:
            # loss_reco over an empty set is NaN in the reference too (mean of empty) and poisons the weights from here
            # on; only the generator's behaviour is compared for this step, then both sides restart from the same state
            cg.update(torch.zeros(1), torch.zeros(0))
            assert abs(cg_mod.mean.item() - cg.mean.item()) <= 1e-6 and abs(cg_mod.var.item() - cg.var.item()) <= 1e-6
            return
        sd, opt_state, ref = wvn_path.train_step(sd, opt_state, x, y, yv, lr=1e-3, cg=cg)
        got = torch.cat([v.reshape(-1) for v in te._model.state_dict().values()]).cpu()
        want = torch.cat([v.reshape(-1) for v in sd.values()])
        print(f"{method} step {step}: loss {m[0]:.7f} vs {ref['loss_total']:.7f}; mean {m[4]:.6f} vs {ref['mean']:.6f}; "
              f"std {m[5]:.6f} vs {ref['std']:.6f}; conf |d| {(conf.cpu() - ref['confidence']).abs().max().item():.1e}; "
              f"param rel {rel_l2(got, want):.2e}")
        assert abs(m[0] - ref["loss_total"]) <= 2e-5 * max(1.0, abs(ref["loss_total"]))
        assert abs(m[4] - ref["mean"]) <= 2e-5 * max(1.0, abs(ref["mean"])) and abs(m[5] - ref["std"]) <= 2e-5 * max(1.0, abs(ref["std"]))
        assert (conf.cpu() - ref["confidence"]).abs().max() <= 1e-4
        assert rel_l2(got, want) <= 2e-5
        # the module's parameters ARE the state the kernels update
        assert abs(cg_mod.mean.item() - ref["mean"]) <= 2e-5 * max(1.0, abs(ref["mean"]))
        assert abs(cg_mod.var.item() - cg.var.item()) <= 1e-5 * max(1.0, abs(cg.var.item()))
        if method == "running_mean":
            assert abs(cg_mod.running_n.item() - cg.running[0].item()) < 0.5
            assert abs(cg_mod.running_sum.item() - cg.running[1].item()) <= 1e-5 * abs(cg.running[1].item())


def test_confidence_state_in_checkpoint_roundtrip(tmp_path):
    """running_mean's sums and the Kalman filter's parameters ride in the checkpoint's traversability_loss_state_dict."""
    from wild_visual_navigation_b200 import TraversabilityEstimator
    from wild_visual_navigation_b200.traversability_estimator.traversability_estimator import default_params

    for method, key in (("running_mean", "_confidence_generator.running_sum"),
                        ("kalman_filter", "_confidence_generator._kalman_filter.proc_cov")):
        params = default_params()
        params["loss"]["method"] = method
        te = TraversabilityEstimator(params=params, device="cuda", min_samples_for_training=0, max_rows=256)
        x = torch.randn(100, 384, device="cuda")
        yv = torch.rand(100, device="cuda") < 0.3
        y = torch.where(yv, torch.rand(100, device="cuda"), torch.zeros(100, device="cuda"))
        te._trainer.step(x, y, yv)
        te.save_checkpoint(str(tmp_path), f"{method}.pt")
        ck = torch.load(str(tmp_path / f"{method}.pt"))
        assert key in ck["traversability_loss_state_dict"]
        params2 = default_params()   # a fresh dict: SimpleMLP mutates its hidden_sizes list, as the reference's does
        params2["loss"]["method"] = method
        te2 = TraversabilityEstimator(params=params2, device="cuda", min_samples_for_training=0, max_rows=256)
        te2.load_checkpoint(str(tmp_path / f"{method}.pt"))
        a, b = te._traversability_loss._confidence_generator, te2._traversability_loss._confidence_generator
        assert torch.equal(a.mean.data, b.mean.data) and torch.equal(a.var.data, b.var.data)
        sa, sb = a.state_dict(), b.state_dict()
        assert list(sa) == list(sb) and all(torch.equal(sa[k], sb[k]) for k in sa)   # the whole state, bit for bit
        # the step's per-row loss_reco is summed with shared-memory float atomics, so two runs of it on the same state
        # differ in the last bits; the confidence's slope 1 / (2 std) turns one ulp of loss_reco into ~1e-6
        # (test_bench_path_gpu.py::test_padded_step_equals_compacted_step holds this output to the same 1e-5)
        c1, c2 = te._trainer.step(x, y, yv).clone(), te2._trainer.step(x, y, yv).clone()
        assert torch.allclose(c1, c2, atol=1e-5)
