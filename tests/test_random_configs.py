"""CPU: randomly drawn TaskPrompter geometries -- task subsets, image shapes, widths, depths, tapped blocks, decoder
widths, 1 or 4 channel-attention windows, with / without cross-task reweighting, ConvHead / DEConvHead, batch 1..3 --
through (a) the oracle restatement against the UNMODIFIED reference's outputs (tests/golden/reference_checks.pt, made by
`python -m oracle.make_golden refchecks`) and (b) the product's
launch plan, kernels emulated by tests/emul_ops.py, against the oracle. The named configurations pin particular shapes;
this pins the bookkeeping (offsets, paddings of e / f to multiples of 8, level selection, per-task slices) in general."""
import os
import random

import pytest
import torch

from oracle import ref_loader
from oracle import taskprompter_ref as TPR
from oracle.make_golden import max_abs_error, perturb, rel_l2_error

REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.pt")


def reference_checks():
    return torch.load(REF, weights_only=False)

N_OUT = {"semseg": None, "human_parts": None, "sal": 2, "normals": 3, "edge": 1, "depth": 1}


def draw(seed):
    rng = random.Random(seed)
    tasks = rng.sample(list(N_OUT), rng.randint(1, 5))
    cn = rng.choice([1, 1, 4])
    step = 32 if cn == 4 else 16                         # the token grid must split into sqrt(cn) x sqrt(cn) windows
    C = rng.choice([64, 128, 192])
    depth = rng.choice([4, 5, 6])
    cfg = dict(tasks=tasks, num_output={t: (N_OUT[t] or rng.randint(2, 9)) for t in tasks},
               img_size=(step * rng.randint(1, 3) + (16 if cn == 1 else 0), step * rng.randint(1, 3) + (16 if cn == 1 else 0)),
               patch=16, C=C, depth=depth, heads=C // 64, select=sorted(rng.sample(range(1, depth), 3)),
               e=rng.choice([12, 20, 24, 30, 36]), f=rng.choice([16, 28, 32, 44]), chan_nheads=cn,
               use_ctr=rng.random() < 0.5, name=f"random{seed}", prompt_len=1, head=rng.choice(["conv", "conv", "deconv"]))
    return cfg, rng.choice([1, 2, 3])


@pytest.mark.parametrize("seed", range(6))
def test_oracle_vs_reference_on_random_geometries(seed):
    """The reference's outputs for these weights (BatchNorm statistics perturbed) are in the fixture."""
    rec = reference_checks()["cases"][f"random_tp{seed}"]
    cfg, B = draw(seed)
    sd = perturb(TPR.init_state_dict(cfg, seed=seed), seed + 1)
    x = torch.randn(B, 3, *cfg["img_size"], generator=torch.Generator().manual_seed(seed + 1000))
    with torch.no_grad():
        out = TPR.forward(sd, cfg, x)
    for t in cfg["tasks"]:
        ref = rec["out"][t]
        assert max_abs_error(out[t], ref) <= 3e-6 * max(ref["absmax"], 1.0), (cfg, t)


@pytest.mark.parametrize("seed", range(10))
def test_launch_plan_vs_oracle_on_random_geometries(monkeypatch, seed):
    import mtt_b200  # noqa: F401
    from mtt_b200 import taskprompter as TP
    import emul_ops

    emul_ops.install(monkeypatch)
    cfg, B = draw(seed)
    sd = TPR.init_state_dict(cfg, seed=seed)
    model = TP.build_from_config(cfg, nsplit=2, use_graph=False).eval()
    model.load_state_dict(sd, strict=True)
    torch.manual_seed(seed)
    x = torch.randn(B, 3, *cfg["img_size"])
    with torch.no_grad():
        ref = TPR.forward(sd, cfg, x)
        got = model.plan(B, torch.device("cpu")).run(x, graph=False)
    for t in cfg["tasks"]:
        assert got[t].shape == ref[t].shape
        err = float((got[t] - ref[t]).norm() / ref[t].norm())
        assert err < 2e-4, (cfg, t, err)


# ---- InvPT -----------------------------------------------------------------------------------------------------------------
def draw_invpt(seed):
    rng = random.Random(1000 + seed)
    tasks = rng.sample(list(N_OUT), rng.randint(1, 4))
    C = rng.choice([128, 192])
    depth = rng.choice([4, 5, 6])
    cfg = dict(tasks=tasks, num_output={t: (N_OUT[t] or rng.randint(2, 9)) for t in tasks},
               img_size=(64 * rng.randint(1, 2), 64 * rng.randint(1, 2)), patch=16, C=C, depth=depth, heads=C // 64,
               select=sorted(rng.sample(range(1, depth), 3)), embed_dim=rng.choice([32, 48, 64]),
               pred_const=rng.choice([8, 16]), down=2, name=f"random_ip{seed}")
    return cfg, rng.choice([1, 2])


@pytest.mark.parametrize("seed", range(6))
def test_invpt_launch_plan_and_oracle_on_random_geometries(monkeypatch, seed):
    """InvPT (IP transformer_net.py:22-38): launch plan (kernels emulated) against the oracle, and the oracle against the
    unmodified reference's outputs for the same weights and input (fixture)."""
    import mtt_b200  # noqa: F401
    from mtt_b200 import invpt as IP
    from oracle import invpt_ref as IPR
    import emul_ops

    emul_ops.install(monkeypatch)
    cfg, B = draw_invpt(seed)
    sd = IPR.init_state_dict(cfg, seed=seed)
    model = IP.build_from_config(cfg, nsplit=2, use_graph=False).eval()
    model.load_state_dict(sd, strict=True)
    torch.manual_seed(seed)
    x = torch.randn(B, 3, *cfg["img_size"])
    with torch.no_grad():
        ref = IPR.forward(sd, cfg, x)
        got = model.plan(B, torch.device("cpu")).run(x, graph=False)
    for t in cfg["tasks"]:
        assert got[t].shape == ref[t].shape
        assert float((got[t] - ref[t]).norm() / ref[t].norm()) < 2e-4, (cfg, t)
        ri, gi = ref["inter_preds"][t], got["inter_preds"][t]
        assert float((gi - ri).norm() / ri.norm()) < 2e-4, (cfg, t, "inter_preds")
    rec = reference_checks()["cases"][f"random_ip{seed}"]
    for t in cfg["tasks"]:
        assert max_abs_error(ref[t], rec["out"][t]) <= 5e-6 * max(rec["out"][t]["absmax"], 1.0), (cfg, t)


def test_invpt_rejects_the_sizes_the_reference_rejects(monkeypatch):
    """A 6 x 6 token grid (96 x 96 image): the reference's decoder concatenates maps of different sizes and raises; the
    oracle restates that; the product says so explicitly before it launches anything."""
    import mtt_b200  # noqa: F401
    from mtt_b200 import invpt as IP
    from oracle import invpt_ref as IPR
    import emul_ops

    emul_ops.install(monkeypatch)
    cfg = dict(tasks=["edge", "semseg"], num_output={"edge": 1, "semseg": 5}, img_size=(96, 96), patch=16, C=128, depth=4,
               heads=2, select=[1, 2, 3], embed_dim=32, pred_const=16, down=2, name="ip_6x6")
    x = torch.randn(1, 3, 96, 96)
    sd = IPR.init_state_dict(cfg, seed=0)
    with pytest.raises(RuntimeError), torch.no_grad():
        IPR.forward(sd, cfg, x)
    assert reference_checks()["raises"]["ip_6x6"] == "RuntimeError"
    model = IP.build_from_config(cfg, nsplit=2, use_graph=False).eval()
    with pytest.raises(ValueError, match="multiple of 4 x 4"):
        model.plan(1, torch.device("cpu"))


# ---- error behaviour and odd-but-legal arguments -----------------------------------------------------------------------
_TP_BASE = dict(tasks=["semseg", "depth"], num_output={"semseg": 5, "depth": 1}, img_size=(64, 64), patch=16, C=128, depth=4,
                heads=2, select=[1, 2, 3], e=24, f=32, use_ctr=True, chan_nheads=1, name="edge", prompt_len=1, head="conv")


@pytest.mark.parametrize("change,match", [(dict(img_size=(48, 80), chan_nheads=4), "chan_nheads=4 must be a perfect square"),
                                          (dict(chan_nheads=2), "chan_nheads=2 must be a perfect square"),
                                          (dict(C=96, heads=2), "must be 64")])
def test_taskprompter_says_what_it_does_not_support(monkeypatch, change, match):
    """Geometries the kernels are not built for (or that fail inside the reference's rearrange, taskprompter.py:236) are
    refused when the model is built / planned, with the reason -- never by a kernel reading out of bounds."""
    import mtt_b200  # noqa: F401
    from mtt_b200 import taskprompter as TP
    import emul_ops

    emul_ops.install(monkeypatch)
    cfg = dict(_TP_BASE, **change)
    with pytest.raises(ValueError, match=match):
        TP.build_from_config(cfg, nsplit=2, use_graph=False).eval().plan(1, torch.device("cpu"))


def test_taskprompter_refuses_inputs_of_another_size(monkeypatch):
    import mtt_b200  # noqa: F401
    from mtt_b200 import taskprompter as TP
    import emul_ops

    emul_ops.install(monkeypatch)
    model = TP.build_from_config(dict(_TP_BASE), nsplit=2, use_graph=False).eval()
    for shape in ((1, 3, 64, 96), (1, 3, 50, 64)):          # the reference asserts on these in PatchEmbed (timm)
        with pytest.raises(ValueError, match="expected fp32 input"):
            model.plan(1, torch.device("cpu")).run(torch.randn(*shape), graph=False)


@pytest.mark.parametrize("select", [[1, 2, 4], [0, 2, 3], [2, 2, 3], [3, 2, 1]])
def test_unusual_select_lists_follow_the_reference(monkeypatch, select):
    """select_list entries past the depth, repeated, zero or out of order: the reference taps a level when
    `idx + 1 in select_list` (taskprompter.py:404-411), so such lists simply tap fewer / other blocks. Same here
    (the reference's outputs for these weights are in the fixture)."""
    import mtt_b200  # noqa: F401
    from mtt_b200 import taskprompter as TP
    import emul_ops

    emul_ops.install(monkeypatch)
    rec = reference_checks()["cases"]["select_" + "-".join(map(str, select))]
    cfg = dict(_TP_BASE, select=select)
    sd = perturb(TPR.init_state_dict(cfg, seed=5), 6)
    x = torch.randn(2, 3, 64, 64, generator=torch.Generator().manual_seed(1005))
    model = TP.build_from_config(cfg, nsplit=2, use_graph=False).eval()
    model.load_state_dict(sd, strict=True)
    with torch.no_grad():
        got = model.plan(2, torch.device("cpu")).run(x, graph=False)
    for t in cfg["tasks"]:
        assert rel_l2_error(got[t], rec["out"][t]) < 2e-4, t


# ---- Swin TaskPrompter ------------------------------------------------------------------------------------------------------
def draw_swin(seed):
    rng = random.Random(2000 + seed)
    tasks = rng.sample(["semseg", "sal", "normals", "edge", "depth"], rng.randint(1, 3))
    ed = rng.choice([16, 32])
    hd = rng.choice([16, ed])                               # head dim 16 or 32 (the two window-attention instantiations)
    cn = rng.choice([1, 1, 4])
    cnh = 2 if cn == 4 else 1
    ratio = rng.choice([1.0, 1.0, 0.75])
    # token maps (image x ratio / 4) must stay even through three PatchMergings and split into cnh x cnh windows at every level:
    # image multiples of 32 cnh at ratio 1, of 128 cnh at ratio 0.75 (x 0.75 -> multiples of 96 = 4 * 8 * 3)
    if ratio == 1.0:
        img = (32 * cnh * rng.randint(1, 3), 32 * cnh * rng.randint(1, 4))
    else:
        img = (128 * cnh * rng.randint(1, 2), 128 * cnh * rng.randint(1, 2))
    cfg = dict(tasks=tasks, num_output={t: (N_OUT[t] or rng.randint(2, 7)) for t in tasks}, img_size=img, patch=4,
               embed_dim=ed, depths=(2, 2, rng.choice([2, 4]), 2), heads=tuple(max(1, (ed * 2 ** i) // hd) for i in range(4)),
               window=rng.choice([4, 6, 8]), img_ds_ratio=ratio, level_embed_dim=rng.choice([10, 12, 16]),
               f=rng.choice([20, 24]), chan_embed_dim=16, chan_nheads=cn, head=rng.choice(["conv", "deconv"]),
               name=f"random_swin{seed}", prompt_len=1)
    return cfg, rng.choice([1, 2])


@pytest.mark.parametrize("seed", range(8))
def test_swin_launch_plan_and_oracle_on_random_geometries(monkeypatch, seed):
    """Swin TaskPrompter (TP taskprompter_swin.py:542-774): shifted windows clipped / padded to the map, 0.75 input
    down-scaling, 1 or 4 channel windows, both head types. Plan (kernels emulated) against the oracle; the oracle against the
    unmodified reference's outputs for the same weights and input (fixture)."""
    import mtt_b200  # noqa: F401
    from mtt_b200 import taskprompter_swin as TS
    from oracle import taskprompter_swin_ref as TSR
    import emul_ops

    emul_ops.install(monkeypatch)
    cfg, B = draw_swin(seed)
    sd = TSR.init_state_dict(cfg, seed=seed)
    torch.manual_seed(seed)
    x = torch.randn(B, 3, *cfg["img_size"])
    model = TS.build_from_config(cfg, nsplit=2, use_graph=False).eval()
    model.load_state_dict(sd, strict=False)              # index / mask buffers are derived, not parameters
    with torch.no_grad():
        ref = TSR.forward(sd, cfg, x)
        got = model.plan(B, torch.device("cpu")).run(x, graph=False)
    for t in cfg["tasks"]:
        assert got[t].shape == ref[t].shape
        assert float((got[t] - ref[t]).norm() / ref[t].norm()) < 2e-4, (cfg, t)
    rec = reference_checks()["cases"][f"random_swin{seed}"]
    for t in cfg["tasks"]:
        assert max_abs_error(ref[t], rec["out"][t]) <= 5e-6 * max(rec["out"][t]["absmax"], 1.0), (cfg, t)


SWIN_BAD = dict(tasks=["depth"], num_output={"depth": 1}, img_size=(64, 96), patch=4, embed_dim=16, depths=(2, 2, 2, 2),
                heads=(1, 2, 4, 8), window=4, img_ds_ratio=1.0, level_embed_dim=12, f=24, chan_embed_dim=16, chan_nheads=1,
                head="conv", name="swin_bad", prompt_len=1)
SWIN_REJECTS = [(dict(img_size=(128, 96), img_ds_ratio=0.75), "must be even on both axes"),
                (dict(img_size=(96, 64), chan_nheads=4), "chan_nheads=4 must be a perfect square")]


@pytest.mark.parametrize("change,match", SWIN_REJECTS)
def test_swin_rejects_the_sizes_the_reference_rejects(change, match):
    """PatchMerging asserts even maps (TP taskprompter_swin.py:438) and the channel gate needs every level's map to split into
    sqrt(chan_nheads)^2 windows (the reference's torch.cat fails at :763 otherwise): refused when the model is built."""
    import mtt_b200  # noqa: F401
    from mtt_b200 import taskprompter_swin as TS
    from oracle import taskprompter_swin_ref as TSR

    cfg = dict(SWIN_BAD, **change)
    with pytest.raises(ValueError, match=match):
        TS.build_from_config(cfg, nsplit=2, use_graph=False)
    x = torch.randn(1, 3, *cfg["img_size"])
    with pytest.raises((RuntimeError, AssertionError)), torch.no_grad():
        TSR.forward(TSR.init_state_dict(cfg, seed=0), cfg, x)
    assert reference_checks()["raises"][match] in ("RuntimeError", "AssertionError")


# ---- the training step ---------------------------------------------------------------------------------------------------
def draw_train(seed):
    rng = random.Random(3000 + seed)
    tasks = rng.sample(list(N_OUT), rng.randint(1, 4))
    cn = rng.choice([1, 1, 4])
    step = 32 if cn == 4 else 16
    C = rng.choice([64, 128])
    depth = rng.choice([4, 5])
    cfg = dict(tasks=tasks, num_output={t: (N_OUT[t] or rng.randint(2, 7)) for t in tasks},
               img_size=(step * rng.randint(1, 2) + (16 if cn == 1 else 0), step * rng.randint(1, 2) + (16 if cn == 1 else 0)),
               patch=16, C=C, depth=depth, heads=C // 64, select=sorted(rng.sample(range(1, depth), 3)),
               e=rng.choice([12, 20, 24]), f=rng.choice([16, 28, 36]), chan_nheads=cn, use_ctr=rng.random() < 0.5,
               name=f"random_train{seed}", prompt_len=1, head="conv", drop_path_rate=0.2)
    return cfg, rng.choice([2, 3])


@pytest.mark.parametrize("seed", [0, 4, 6, 7])
def test_training_step_on_random_geometries(monkeypatch, seed):
    """TrainStep (train-mode forward with replayed DropPath draws, hand-scheduled reverse pass; kernels emulated) against
    torch autograd of the oracle's train-mode restatement, for the same upstream gradient: forward 2e-4, every parameter
    gradient 5e-3 of max(|g|, 1e-4 |all gradients|)."""
    import mtt_b200  # noqa: F401
    from mtt_b200 import taskprompter as TP
    from mtt_b200.train import TrainStep
    import emul_ops

    emul_ops.install(monkeypatch)
    cfg, B = draw_train(seed)
    sd = TPR.init_state_dict(cfg, seed=seed)
    model = TP.build_from_config(cfg, use_graph=False)
    model.load_state_dict(sd, strict=True)
    ts = TrainStep(model, lr=1e-4)
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(B, 3, *cfg["img_size"], generator=g)
    masks = [torch.rand(B, 1, 1, generator=g) for _ in range(4 * cfg["depth"])]
    ts.zero_grad()
    with torch.no_grad():
        out = ts.forward(x, drop_rand=masks)
    gout = {t: torch.randn(out[t].shape, generator=g) for t in cfg["tasks"]}
    with torch.no_grad():
        ts.backward(gout)
    sdo = {k: v.clone() for k, v in sd.items()}
    params = {k: v.requires_grad_(True) for k, v in sdo.items() if v.is_floating_point() and "running_" not in k}
    sdo.update(params)
    with TPR.train_mode(0.2, rand=masks):
        ref = TPR.forward(sdo, cfg, x)
    for t in cfg["tasks"]:
        assert float((out[t] - ref[t].detach()).norm() / ref[t].detach().norm()) < 2e-4, (cfg, t)
    torch.autograd.backward([ref[t] for t in cfg["tasks"]], [gout[t] for t in cfg["tasks"]])
    total = float(torch.sqrt(sum((v.grad ** 2).sum() for v in params.values() if v.grad is not None)))
    for k, v in params.items():
        want = v.grad if v.grad is not None else torch.zeros_like(v)
        err = float((ts.G_(k).detach().cpu() - want).norm()) / max(float(want.norm()), 1e-4 * total)
        assert err < 5e-3, (cfg, k, err)


# ---- accelerate(live reference model) end to end -----------------------------------------------------------------------
@pytest.mark.skipif(not ref_loader.available(), reason="reference tree not present")
@pytest.mark.parametrize("family,name", [("tp", "tp_tiny"), ("tp", "tp_tiny_de"), ("ip", "ip_tiny")])
def test_accelerate_runs_a_live_reference_model_end_to_end(monkeypatch, family, name):
    """accelerate(ref_model) on an instance of the UNMODIFIED reference (its own random initialisation, BatchNorm statistics
    perturbed): the accelerated model's forward (launch plan, kernels emulated) reproduces the reference model's own
    forward on the same input -- the drop-in claim of INTEGRATION.md section 1, not only equal state dicts."""
    import mtt_b200  # noqa: F401
    from mtt_b200 import configs
    import emul_ops

    emul_ops.install(monkeypatch)
    if family == "tp":
        from mtt_b200 import taskprompter as M
        cfg = configs.taskprompter(name)
        ref = ref_loader.build_taskprompter(cfg)
    else:
        from mtt_b200 import invpt as M
        cfg = configs.invpt(name)
        ref = ref_loader.build_invpt(cfg)
    torch.manual_seed(5)
    for m in ref.modules():
        if isinstance(m, (torch.nn.BatchNorm2d, torch.nn.SyncBatchNorm)):
            m.running_mean.normal_(0, 0.1)
            m.running_var.uniform_(0.8, 1.2)
    ref.eval()
    mine = M.accelerate(ref, use_graph=False).eval()
    x = torch.randn(2, 3, *cfg["img_size"])
    with torch.no_grad():
        want = ref(x)
        got = {t: v.clone() for t, v in mine.plan(2, torch.device("cpu")).run(x, graph=False).items() if t in cfg["tasks"]}
    for t in cfg["tasks"]:
        assert got[t].shape == want[t].shape
        assert float((got[t] - want[t]).norm() / want[t].norm()) < 2e-4, t
    # accelerate() COPIES the parameters (DESIGN.md section 1): a later in-place update of the reference is not seen ...
    with torch.no_grad():
        next(ref.parameters()).add_(1.0)
        again = mine.plan(2, torch.device("cpu")).run(x, graph=False)
    for t in cfg["tasks"]:
        assert torch.equal(again[t], got[t])
