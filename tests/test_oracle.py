"""CPU: the oracle restatement against the golden vectors produced by the unmodified reference: (a) with the oracle's
initialisers (tests/golden/<config>.pt) and (b) with perturbed BatchNorm statistics (Swin: also bias tables and biases),
checked against summaries of the reference's outputs and signatures of its parameter names
(tests/golden/reference_checks.pt, `python -m oracle.make_golden refchecks`). The state-dict sharing of accelerate()
needs a live instance of the reference's classes and runs where the reference tree is present."""
import os

import pytest
import torch

from oracle import configs, ref_loader
from oracle import taskprompter_ref as TPR
from oracle import invpt_ref as IPR
from oracle.make_golden import max_abs_error, perturb, sd_checksum, signature

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def reference_case(name):
    return torch.load(os.path.join(GOLD, "reference_checks.pt"), weights_only=False)["cases"][name]


@pytest.mark.parametrize("name", ["tp_tiny", "tp_tiny1", "tp_tiny_de"])
def test_taskprompter_oracle_vs_golden(name):
    fx = torch.load(os.path.join(GOLD, f"{name}.pt"), weights_only=False)
    cfg = configs.taskprompter(fx["cfg"])
    sd = TPR.init_state_dict(cfg, seed=fx["seed"])
    assert sd_checksum(sd) == fx["sd_sha256"], "deterministic initialiser drifted from the fixture"
    with torch.no_grad():
        out = TPR.forward(sd, cfg, fx["x"])
    for t, ref in fx["out"].items():
        # same algorithm, same fp32 library kernels, different op order: rounding-level agreement
        assert (out[t] - ref).abs().max() <= 2e-6 * ref.abs().max().clamp_min(1.0) + 2e-6, t
        if t in ("semseg", "human_parts"):
            assert torch.equal(out[t].argmax(1), ref.argmax(1))


@pytest.mark.parametrize("name", ["tp_tiny", "tp_tiny1", "tp_tiny_de"])
def test_taskprompter_oracle_vs_reference(name):
    rec = reference_case(name)
    cfg = configs.taskprompter(name)
    sd = perturb(TPR.init_state_dict(cfg, seed=rec["seed"]), rec["seed"] + 1)
    assert signature(sorted((k, v.shape) for k, v in sd.items())) == rec["sorted_param_signature"]   # the reference's names
    x = torch.randn(rec["batch"], 3, *cfg["img_size"], generator=torch.Generator().manual_seed(rec["seed"] + 1000))
    with torch.no_grad():
        out = TPR.forward(sd, cfg, x)
    for t in cfg["tasks"]:
        assert max_abs_error(out[t], rec["out"][t]) <= 2e-6, t


@pytest.mark.skipif(not ref_loader.available(), reason="reference tree not present")
@pytest.mark.parametrize("name", ["tp_tiny", "tp_tiny_de"])
def test_accelerate_shares_reference_state_dict(name):
    import mtt_b200  # noqa: F401
    from mtt_b200 import taskprompter as TP

    cfg = configs.taskprompter(name)
    ref = ref_loader.build_taskprompter(cfg).eval()
    mine = TP.accelerate(ref)
    a, b = ref.state_dict(), mine.state_dict()
    assert list(a.keys()) == list(b.keys())
    assert all(torch.equal(a[k], b[k]) for k in a)


@pytest.mark.parametrize("name", ["ip_tiny", "ip_cfg1"])
def test_invpt_oracle_vs_golden(name):
    fx = torch.load(os.path.join(GOLD, f"{name}.pt"), weights_only=False)
    cfg = configs.invpt(fx["cfg"])
    sd = IPR.init_state_dict(cfg, seed=fx["seed"])
    assert sd_checksum(sd) == fx["sd_sha256"], "deterministic initialiser drifted from the fixture"
    with torch.no_grad():
        out = IPR.forward(sd, cfg, fx["x"])
    for t, ref in fx["out"].items():
        assert (out[t] - ref).abs().max() <= 5e-6 * ref.abs().max().clamp_min(1.0), t
        if fx["inter_preds"] is not None:
            assert (out["inter_preds"][t] - fx["inter_preds"][t]).abs().max() <= 5e-6, t


@pytest.mark.parametrize("name", ["ip_tiny", "ip_cfg1"])
def test_invpt_oracle_vs_reference(name):
    rec = reference_case(name)
    cfg = configs.invpt(name)
    sd = perturb(IPR.init_state_dict(cfg, seed=rec["seed"]), rec["seed"] + 1)
    assert signature(sorted((k, v.shape) for k, v in sd.items())) == rec["sorted_param_signature"]
    x = torch.randn(rec["batch"], 3, *cfg["img_size"], generator=torch.Generator().manual_seed(rec["seed"] + 1000))
    with torch.no_grad():
        out = IPR.forward(sd, cfg, x)
    for t in cfg["tasks"]:
        assert max_abs_error(out[t], rec["out"][t]) <= 5e-6, t
        assert max_abs_error(out["inter_preds"][t], rec["inter_preds"][t]) <= 5e-6, t


@pytest.mark.skipif(not ref_loader.available(), reason="reference tree not present")
def test_invpt_accelerate_shares_reference_state_dict():
    import mtt_b200  # noqa: F401
    from mtt_b200 import invpt as IP

    cfg = configs.invpt("ip_tiny")
    ref = ref_loader.build_invpt(cfg).eval()
    mine = IP.accelerate(ref)
    a, b = ref.state_dict(), mine.state_dict()
    assert set(a.keys()) == set(b.keys())
    assert all(torch.equal(a[k], b[k]) for k in a)


# ---- Swin-backbone TaskPrompter (SURVEY.md section 8f N2): oracle only, no CUDA path yet -------------------------
@pytest.mark.parametrize("name", ["tps_tiny", "tps_tiny4"])
def test_swin_oracle_vs_golden(name):
    from oracle import taskprompter_swin_ref as SR

    fx = torch.load(os.path.join(GOLD, f"{name}.pt"), weights_only=False)
    cfg = configs.taskprompter_swin(fx["cfg"])
    sd = SR.init_state_dict(cfg, seed=fx["seed"])
    assert sd_checksum(sd) == fx["sd_sha256"], "deterministic initialiser drifted from the fixture"
    with torch.no_grad():
        out = SR.forward(sd, cfg, fx["x"])
    for t, ref in fx["out"].items():
        assert out[t].shape == ref.shape
        assert (out[t] - ref).abs().max() <= 5e-6 * ref.abs().max().clamp_min(1.0) + 2e-6, t
        if t == "semseg":
            assert torch.equal(out[t].argmax(1), ref.argmax(1))


@pytest.mark.parametrize("name", ["tps_tiny", "tps_tiny4", "tps_mid"])
def test_swin_oracle_vs_reference(name):
    """Against the unmodified reference's outputs with non-trivial biases, bias tables and BatchNorm statistics: shifted
    and padded windows, 2x2 channel windows, patch merging of the logit maps. The parameter names and shapes the oracle
    expects are the reference module's (signature of the sorted list, derived index / mask buffers excluded)."""
    from oracle import taskprompter_swin_ref as SR

    rec = reference_case(name)
    cfg = configs.taskprompter_swin(name)
    assert signature(sorted(SR.param_shapes(cfg).items())) == rec["sorted_param_signature"]
    sd = perturb(SR.init_state_dict(cfg, seed=rec["seed"]), rec["seed"] + 1, swin=True)
    x = torch.randn(rec["batch"], 3, *cfg["img_size"], generator=torch.Generator().manual_seed(rec["seed"] + 1000))
    with torch.no_grad():
        out = SR.forward(sd, cfg, x)
    for t in cfg["tasks"]:
        assert max_abs_error(out[t], rec["out"][t]) <= 5e-6, t


def test_swin_window_tables_match_definitions():
    """The derived tables the oracle recomputes (instead of reading the reference's buffers)."""
    from oracle import taskprompter_swin_ref as SR

    idx = SR.relative_position_index(3)
    assert idx.shape == (9, 9) and idx.min() == 0 and idx.max() == 24 and idx[0, 0] == 12      # centre of a 5x5 table
    assert idx[0, 8] == 0 and idx[8, 0] == 24
    m = SR.shifted_window_mask(8, 8, 4, 2)
    assert m.shape == (4, 16, 16) and set(m.unique().tolist()) == {-100.0, 0.0}
    assert (m[0] == 0).all()                      # the top-left window holds one region only
    assert (m[3] != 0).any() and torch.equal(m[3], m[3].t())


def test_swin_param_shapes_at_the_reference_config():
    """The reference's Cityscapes-3D Swin-B model (cs_swinB_taskprompter.yml: 1024x2048, img_ds_ratio 0.75, window 12,
    depths 2-2-18-2): every parameter name and shape the oracle expects equals the reference module's (274.6 M
    parameters; construction only, no forward; the reference's list is stored as a signature)."""
    from oracle import taskprompter_swin_ref as SR

    cfg = configs.taskprompter_swin("tps_swinB")
    ref = torch.load(os.path.join(GOLD, "reference_checks.pt"), weights_only=False)["tps_swinB"]
    shapes = SR.param_shapes(cfg)
    assert len(shapes) == ref["n_params"] == 732
    assert signature(sorted(shapes.items())) == ref["sorted_param_signature"]
    assert [SR.stage_geometry(cfg, i)[1] for i in range(4)] == [(192, 384), (96, 192), (48, 96), (24, 48)]
    assert [SR.level_resolution(cfg, i) for i in range(4)] == [(96, 192), (48, 96), (24, 48), (24, 48)]
