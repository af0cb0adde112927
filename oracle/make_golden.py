"""Generates tests/golden/*.pt by running the UNMODIFIED reference (imported from /root/reference through
oracle/shim) in the build container. TEST INFRASTRUCTURE.

Weights come from the deterministic oracle initialisers (oracle.taskprompter_ref.init_state_dict,
oracle.invpt_ref.init_state_dict: fixed torch CPU generator seeds) loaded into the reference model
with strict=True, so a fixture only needs to carry the input, the reference's outputs and a checksum
of the parameters -- the GPU box regenerates identical weights without /root/reference.

    python -m oracle.make_golden            # rewrites tests/golden/
"""
import hashlib
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import configs, ref_loader  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def sd_checksum(sd):
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].detach().cpu().contiguous().numpy().tobytes())
    return h.hexdigest()


def make_taskprompter(name, seed, batch):
    from oracle import taskprompter_ref as R

    cfg = configs.taskprompter(name)
    sd = R.init_state_dict(cfg, seed=seed)
    model = ref_loader.build_taskprompter(cfg).eval()
    model.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(seed + 1000)
    x = torch.randn(batch, 3, *cfg["img_size"], generator=g)
    with torch.no_grad():
        y = model(x)
    return {"family": "taskprompter", "cfg": name, "seed": seed, "x": x, "out": {k: v.clone() for k, v in y.items()},
            "sd_sha256": sd_checksum(sd), "torch": torch.__version__,
            "made_by": "oracle/make_golden.py from the unmodified reference forward (eval, fp32, CPU)"}


def make_taskprompter_swin(name, seed, batch):
    from oracle import taskprompter_swin_ref as R

    cfg = configs.taskprompter_swin(name)
    sd = R.init_state_dict(cfg, seed=seed)
    model = ref_loader.build_taskprompter_swin(cfg).eval()
    missing, unexpected = model.load_state_dict(sd, strict=False)   # index / mask buffers are derived, not stored
    assert not unexpected and all("relative_position_index" in k or "attn_mask" in k for k in missing), (missing, unexpected)
    g = torch.Generator().manual_seed(seed + 1000)
    x = torch.randn(batch, 3, *cfg["img_size"], generator=g)
    with torch.no_grad():
        y = model(x)
    return {"family": "taskprompter_swin", "cfg": name, "seed": seed, "x": x, "out": {k: v.clone() for k, v in y.items()},
            "sd_sha256": sd_checksum(sd), "torch": torch.__version__,
            "made_by": "oracle/make_golden.py from the unmodified reference Swin TaskPrompter forward (eval, fp32, CPU)"}


def make_invpt(name, seed, batch):
    from oracle import invpt_ref as R

    cfg = configs.invpt(name)
    sd = R.init_state_dict(cfg, seed=seed)
    model = ref_loader.build_invpt(cfg).eval()
    model.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(seed + 1000)
    x = torch.randn(batch, 3, *cfg["img_size"], generator=g)
    with torch.no_grad():
        y = model(x)
    out = {k: v.clone() for k, v in y.items() if k != "inter_preds"}
    # inter_preds kept only for the tiny config (fixture size)
    inter = {k: v.clone() for k, v in y["inter_preds"].items()} if name == "ip_tiny" else None
    return {"family": "invpt", "cfg": name, "seed": seed, "x": x, "out": out, "inter_preds": inter,
            "sd_sha256": sd_checksum(sd), "torch": torch.__version__,
            "made_by": "oracle/make_golden.py from the unmodified reference forward (eval, fp32, CPU)"}


def make_preproc():
    """Golden vectors for the inference pre-processing: the reference's OWN Normalize / ToTensor classes
    (TaskPrompter/data/transforms.py) around cv2.cvtColor + cv2.resize exactly as TaskPrompter/inference.py:66-81,
    :93-115, :127-133 chains them (inference.py itself parses argv and loads a checkpoint at import, so its three-line
    DirectResize is restated here around the same cv2 call)."""
    import cv2
    import numpy as np

    ref_loader._activate("TaskPrompter")
    from data import transforms as T

    rng = np.random.default_rng(7)
    cases = []
    for (h, w, H, W) in [(37, 53, 64, 48), (96, 120, 64, 80), (50, 70, 50, 70)]:
        bgr = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        img = cv2.cvtColor(bgr.astype(np.float32), cv2.COLOR_BGR2RGB)          # inference.py:127-128
        sample = T.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])({"image": img})
        sample["image"] = cv2.resize(sample["image"], (W, H), interpolation=cv2.INTER_LINEAR)   # DirectResize
        out = T.ToTensor()(sample)["image"].unsqueeze(0)
        cases.append({"bgr_u8": torch.from_numpy(bgr), "out_hw": (H, W), "out": out.clone()})
    return {"family": "preproc", "cases": cases, "cv2": cv2.__version__,
            "made_by": "oracle/make_golden.py: reference Normalize/ToTensor + cv2.resize (TP/inference.py pipeline)"}


LOSS_WEIGHTS = {"semseg": 1.0, "human_parts": 2.0, "sal": 5.0, "edge": 50.0, "normals": 10.0, "depth": 1.0}  # the ymls


def synthetic_labels(tasks, num_output, B, H, W, g):
    """Labels of the shapes the reference's datasets produce, with ignore regions (255; depth: -1)."""
    lab = {}
    hole = lambda frac: torch.rand(B, 1, H, W, generator=g) < frac
    for t in tasks:
        if t in ("semseg", "human_parts"):
            y = torch.randint(0, num_output[t], (B, 1, H, W), generator=g).float()
            y[hole(0.1)] = 255.0
        elif t == "sal":
            y = (torch.rand(B, 1, H, W, generator=g) < 0.3).float()
            y[hole(0.05)] = 255.0
        elif t == "edge":
            y = (torch.rand(B, 1, H, W, generator=g) < 0.1).float()
            y[hole(0.05)] = 255.0
        elif t == "normals":
            y = torch.nn.functional.normalize(torch.randn(B, 3, H, W, generator=g), dim=1)
            y = torch.where(hole(0.1).expand(-1, 3, -1, -1), torch.full_like(y, 255.0), y)
        elif t == "depth":
            y = torch.rand(B, 1, H, W, generator=g) * 9 + 0.5
            y[hole(0.15)] = -1.0
        lab[t] = y
    return lab


def make_losses():
    """Golden vectors for the training losses and for the backward pass they drive: (a) every task loss and the
    weighted total of the reference's criterion (utils/common_config.py:211-244 -> losses/) on random predictions,
    with d total / d prediction; (b) the tp_tiny reference model in eval mode -> criterion -> autograd: total loss
    and, per parameter, the gradient's L2 norm and sum (full gradients for a few small parameters)."""
    ref_loader._activate("TaskPrompter")
    from easydict import EasyDict
    from utils.common_config import get_criterion

    def criterion(tasks):
        p = EasyDict(TASKS=EasyDict(NAMES=list(tasks)), edge_w=0.95, ignore_index=255, ignore_invalid_area_depth=True,
                     loss_kwargs=EasyDict(loss_weights={t: LOSS_WEIGHTS[t] for t in tasks}))
        return get_criterion(p)

    g = torch.Generator().manual_seed(77)
    tasks = ["semseg", "human_parts", "sal", "edge", "normals", "depth"]
    nout = {"semseg": 7, "human_parts": 5, "sal": 2, "edge": 1, "normals": 3, "depth": 1}
    B, H, W = 2, 24, 32
    preds = {t: (torch.randn(B, nout[t], H, W, generator=g) * 2).requires_grad_() for t in tasks}
    labels = synthetic_labels(tasks, nout, B, H, W, g)
    out = criterion(tasks)(preds, labels, tasks=tasks)
    out["total"].backward()
    part_a = {"tasks": tasks, "preds": {t: preds[t].detach().clone() for t in tasks}, "labels": labels,
              "losses": {k: float(v.detach()) for k, v in out.items()},
              "dpreds": {t: preds[t].grad.clone() for t in tasks}}

    from oracle import taskprompter_ref as R
    cfg = configs.taskprompter("tp_tiny")
    sd = R.init_state_dict(cfg, seed=3)
    model = ref_loader.build_taskprompter(cfg).eval()
    model.load_state_dict(sd, strict=True)
    crit = criterion(cfg["tasks"])          # build_taskprompter re-activated the same reference root
    x = torch.randn(2, 3, *cfg["img_size"], generator=g)
    lab = synthetic_labels(cfg["tasks"], cfg["num_output"], 2, *cfg["img_size"], g)
    loss = crit(model(x), lab, tasks=cfg["tasks"])
    model.zero_grad()
    loss["total"].backward()
    grads = {k: v.grad for k, v in model.named_parameters()}
    full = ["backbone.task_prompts", "backbone.blocks.0.attn.qkv.bias", "backbone.blocks.3.attn.token_trans1.bias",
            "backbone.norm.weight", "heads.semseg.linear_pred.weight", "backbone.ctr_attn_conv.0.depth.0.weight"]
    part_b = {"cfg": "tp_tiny", "seed": 3, "x": x, "labels": lab, "losses": {k: float(v.detach()) for k, v in loss.items()},
              "grad_norm": {k: float(v.norm()) for k, v in grads.items()},
              "grad_sum": {k: float(v.double().sum()) for k, v in grads.items()},
              "grad_full": {k: grads[k].clone() for k in full}}
    return {"family": "losses", "criterion": part_a, "model": part_b, "weights": LOSS_WEIGHTS, "torch": torch.__version__,
            "made_by": "oracle/make_golden.py: reference get_criterion + autograd through the unmodified reference model"}


# ---------------------------------------------------------------------------------------------------------
# Full-size configurations (BASELINE.json configs[1..4]): the reference's outputs are hundreds of MB, so the
# fixture keeps (i) every output value on a stride-8 pixel lattice whose offset changes per (image, task) --
# the outputs are bilinear up-samplings of 4x / 8x coarser maps, so the lattice sees every coarse cell --
# (ii) the exact norms of the full tensors, and (iii) for multi-class tasks the full-resolution arg-max map
# (uint8) with the mask of pixels whose top-2 margin exceeds 1e-4 * max|logit| (where arg-max must be exact).
# The input is regenerated from the seed; its SHA-256 is stored.
BIG_STRIDE = 8
BIG_JOBS = [  # (family, config, seed, batch)
    ("taskprompter", "tp_cfg5_d4", 41, 1),   # N = 8195 tokens: 65 query tiles, ragged last key block
    ("taskprompter", "tp_cfg4", 42, 4),      # the bench configuration: 24 blocks, bs 4
    ("taskprompter", "tp_cfg2", 43, 4),      # BASELINE.json configs[1]
    ("invpt", "ip_cfg3", 44, 4),             # BASELINE.json configs[2]
    ("taskprompter", "tp_cfg5", 45, 1),      # BASELINE.json configs[4]: full 24-block, N = 8195
]


def big_input(cfg, seed, batch):
    g = torch.Generator().manual_seed(seed + 1000)
    return torch.randn(batch, 3, *cfg["img_size"], generator=g)


def lattice(b, ti, H, W, stride=BIG_STRIDE):
    """Row / column indices of the sampled pixels of image b, task index ti."""
    oy, ox = (3 * b + 5 * ti + 1) % stride, (5 * b + 3 * ti + 2) % stride
    return torch.arange(oy, H, stride), torch.arange(ox, W, stride)


def compress_output(y, ti, with_argmax=True):
    """y [B, n_out, H, W] fp32 -> the fixture record described above (`safe` is bit-packed, numpy.packbits order)."""
    B, n, H, W = y.shape
    samp = []
    for b in range(B):
        iy, ix = lattice(b, ti, H, W)
        samp.append(y[b][:, iy][:, :, ix].clone())
    rec = {"shape": tuple(y.shape), "samples": torch.stack(samp), "norm": float(y.double().norm()),
           "absmax": float(y.abs().max())}
    if n > 1 and with_argmax:
        import numpy as np
        top2 = y.topk(2, dim=1).values
        rec["argmax"] = y.argmax(1).to(torch.uint8)
        safe = (top2[:, 0] - top2[:, 1]) > 1e-4 * y.abs().max()
        rec["safe_bits"] = torch.from_numpy(np.packbits(safe.numpy().reshape(-1)))
    return rec


def make_big(family, name, seed, batch):
    if family == "taskprompter":
        from oracle import taskprompter_ref as R
        cfg = configs.taskprompter(name)
        model = ref_loader.build_taskprompter(cfg).eval()
    else:
        from oracle import invpt_ref as R
        cfg = configs.invpt(name)
        model = ref_loader.build_invpt(cfg).eval()
    sd = R.init_state_dict(cfg, seed=seed)
    model.load_state_dict(sd, strict=True)
    x = big_input(cfg, seed, batch)
    with torch.no_grad():
        y = model(x)
    out = {t: compress_output(y[t], ti) for ti, t in enumerate(cfg["tasks"])}
    inter = None
    if family == "invpt":
        inter = {t: compress_output(y["inter_preds"][t], ti, with_argmax=False) for ti, t in enumerate(cfg["tasks"])}
    return {"family": family, "cfg": name, "seed": seed, "batch": batch, "stride": BIG_STRIDE, "out": out,
            "inter_preds": inter, "x_sha256": hashlib.sha256(x.numpy().tobytes()).hexdigest(),
            "sd_sha256": sd_checksum(sd), "torch": torch.__version__,
            "made_by": "oracle/make_golden.py make_big: unmodified reference forward (eval, fp32, CPU), lattice-sampled"}


def main_big(only=None):
    import time
    for fam, name, seed, batch in BIG_JOBS:
        if only and name not in only:
            continue
        t0 = time.time()
        fx = make_big(fam, name, seed, batch)
        path = os.path.join(GOLD, f"big_{name}_b{batch}.pt")
        torch.save(fx, path)
        print(f"wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB, {time.time() - t0:.0f} s)", flush=True)


# ---------------------------------------------------------------------------------------------------------
# Training step (SURVEY.md 8f N1): the unmodified reference model in TRAIN mode (BatchNorm batch statistics, DropPath
# 0.15) -> the reference criterion -> autograd -> clip_grad_norm_ -> torch.optim.Adam (train_utils.py:34-51 with the
# yml's optimizer block). The fixture keeps the DropPath masks the reference drew (CPU generator; the product draws
# them with the same calls on its own device), the train-mode outputs, the losses, every parameter gradient (small
# models) or its norm / sum plus a few full ones (large models), the BatchNorm running statistics after the forward and
# the parameters after the optimizer step (same selection).
TRAIN_JOBS = [("tp_tiny", 21, 2, True), ("tp_tiny1", 22, 3, False), ("tp_cfg4_d4", 23, 2, False)]
TRAIN_HYPER = dict(lr=2e-5, weight_decay=1e-6, max_norm=10.0)      # configs/pascal/pascal_vitLp16_taskprompter.yml:18-23


def train_inputs(cfg, seed, batch):
    """The synthetic image batch and labels of a training fixture (CPU generator: identical wherever it runs)."""
    g = torch.Generator().manual_seed(seed + 500)
    x = torch.randn(batch, 3, *cfg["img_size"], generator=g)
    return x, synthetic_labels(cfg["tasks"], cfg["num_output"], batch, *cfg["img_size"], g)


def make_train(name, seed, batch, full):
    from oracle import taskprompter_ref as R

    cfg = configs.taskprompter(name)
    sd = R.init_state_dict(cfg, seed=seed)
    model = ref_loader.build_taskprompter(cfg)
    model.load_state_dict(sd, strict=True)
    model.train()
    from easydict import EasyDict
    from utils.common_config import get_criterion
    tasks = cfg["tasks"]
    p = EasyDict(TASKS=EasyDict(NAMES=list(tasks)), edge_w=0.95, ignore_index=255, ignore_invalid_area_depth=True,
                 loss_kwargs=EasyDict(loss_weights={t: LOSS_WEIGHTS[t] for t in tasks}))
    crit = get_criterion(p)
    x, lab = train_inputs(cfg, seed, batch)
    masks, real_rand = [], torch.rand

    def rand(*a, **k):
        r = real_rand(*a, **k)
        if tuple(r.shape) == (batch, 1, 1):
            masks.append(r.clone())
        return r
    torch.manual_seed(seed + 900)
    torch.rand = rand
    try:
        out = model(x)
    finally:
        torch.rand = real_rand
    loss = crit(out, lab, tasks=tasks)
    opt = torch.optim.Adam(model.parameters(), lr=TRAIN_HYPER["lr"], weight_decay=TRAIN_HYPER["weight_decay"])
    opt.zero_grad()
    loss["total"].backward()
    grads = {k: v.grad.detach().clone() for k, v in model.named_parameters()}
    total_norm = float(torch.nn.utils.clip_grad_norm_(model.parameters(), max_norm=TRAIN_HYPER["max_norm"], norm_type=2))
    opt.step()
    after = {k: v.detach().clone() for k, v in model.named_parameters()}
    few = {
        "backbone.task_prompts", "backbone.patch_embed.proj.bias", "backbone.blocks.0.attn.qkv.bias",
        "backbone.blocks.0.norm1.weight", "backbone.blocks.1.mlp.fc1.bias", "backbone.blocks.3.attn.token_trans1.bias",
        "backbone.blocks.2.attn.token_trans.bias", "backbone.norm.weight", f"heads.{tasks[0]}.linear_pred.weight",
        f"backbone.ctr_attn_conv.0.{tasks[1]}.0.weight", f"backbone.fea_fuse.1.{tasks[0]}.2.weight",
        f"backbone.fea_fuse.2.{tasks[1]}.4.weight", f"backbone.fea_decode_spa.3.{tasks[2 % len(tasks)]}.0.weight",
        f"heads.{tasks[-1]}.mt_proj.1.bias"} & set(grads)
    keep = set(grads) if full else few
    bn = {k: v.detach().clone() for k, v in model.state_dict().items() if "running_" in k}
    lat = lambda v: v[..., ::8, ::8].clone() if not full else v.detach().clone()
    # the input and the labels are regenerated by the test from the seed (train_inputs below); only checksums travel
    sha = lambda t_: hashlib.sha256(t_.contiguous().numpy().tobytes()).hexdigest()
    return {"family": "train", "cfg": name, "seed": seed, "batch": batch, "x_sha256": sha(x),
            "labels_sha256": {k: sha(v) for k, v in lab.items()}, "masks": masks, "hyper": TRAIN_HYPER,
            "out": {k: lat(v.detach()) for k, v in out.items()}, "out_stride": 1 if full else 8,
            "losses": {k: float(v.detach()) for k, v in loss.items()}, "total_norm": total_norm,
            "grad_norm": {k: float(v.norm()) for k, v in grads.items()},
            "grad_sum": {k: float(v.double().sum()) for k, v in grads.items()},
            "grad_full": {k: grads[k] for k in sorted(keep)}, "param_after": {k: after[k] for k in sorted(few) if after[k].numel() <= 70000},
            "running": bn if full else {k: v for k, v in bn.items() if ".2.running" in k and ".0." in k},
            "sd_sha256": sd_checksum(sd), "weights": LOSS_WEIGHTS, "torch": torch.__version__,
            "made_by": "oracle/make_golden.py train: the unmodified reference model in train mode, the reference criterion, "
                       "torch autograd, clip_grad_norm_ and torch.optim.Adam"}


def main_train(only=None):
    for name, seed, batch, full in TRAIN_JOBS:
        if only and name not in only:
            continue
        fx = make_train(name, seed, batch, full)
        path = os.path.join(GOLD, f"train_{name}.pt")
        torch.save(fx, path)
        print(f"wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)", flush=True)


# ---------------------------------------------------------------------------------------------------------
# Reference checks (tests/golden/reference_checks.pt): the reference's outputs for the comparisons of
# tests/test_oracle.py and tests/test_random_configs.py, so those tests run where the reference is absent.
# Weights are the oracle initialisers plus the perturbations `perturb` draws from a fixed CPU generator
# (BatchNorm statistics; Swin also bias tables and biases), loaded into the reference with strict=True; the
# fixture stores a summary of each output (`summarize`) and signatures of the reference's parameter names.
SAMPLE_STRIDE = 1000003        # prime: the sampled flat indices are distinct for any output smaller than it


def signature(pairs):
    """SHA-256 over a sequence of (name, shape) pairs, in the order given."""
    h = hashlib.sha256()
    for k, shape in pairs:
        h.update(f"{k}:{tuple(shape)};".encode())
    return h.hexdigest()


def perturb(sd, seed, swin=False):
    """A copy of state dict `sd` (same order) with BatchNorm running statistics drawn around (0, 1); with `swin`, also
    relative-position bias tables ~ N(0, 0.5) and every bias ~ N(0, 0.05)."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for k, v in sd.items():
        if k.endswith("running_mean"):
            v = torch.randn(v.shape, generator=g) * 0.1
        elif k.endswith("running_var"):
            v = torch.rand(v.shape, generator=g) * 0.4 + 0.8
        elif swin and "relative_position_bias_table" in k:
            v = torch.randn(v.shape, generator=g) * 0.5
        elif swin and k.endswith(".bias"):
            v = torch.randn(v.shape, generator=g) * 0.05
        out[k] = v
    return out


def summarize(y, k=256):
    """Output tensor [B, C, ...] -> k elements at fixed flat indices, the per-(image, channel) means (float64), the norm."""
    y = y.detach().float().cpu()
    n = y.numel()
    assert n % SAMPLE_STRIDE, n
    idx = (torch.arange(min(k, n), dtype=torch.int64) * SAMPLE_STRIDE + 7) % n
    return {"shape": tuple(y.shape), "sample": y.reshape(-1)[idx].clone(),
            "channel_mean": y.double().flatten(2).mean(2), "norm": float(y.double().norm()), "absmax": float(y.abs().max())}


def max_abs_error(y, rec):
    """Largest |difference| of y against a `summarize` record, over the sampled elements and the channel means (each a
    lower bound of the largest elementwise |difference|)."""
    s = summarize(y)
    assert s["shape"] == rec["shape"], (s["shape"], rec["shape"])
    return max(float((s["sample"] - rec["sample"]).abs().max()), float((s["channel_mean"] - rec["channel_mean"]).abs().max()))


def rel_l2_error(y, rec):
    """Relative L2 difference of y against a `summarize` record: over the sampled elements, and | |y| - |ref| | / |ref|
    (a lower bound of |y - ref| / |ref|)."""
    s = summarize(y)
    assert s["shape"] == rec["shape"], (s["shape"], rec["shape"])
    return max(float((s["sample"] - rec["sample"]).norm() / rec["sample"].norm()), abs(s["norm"] - rec["norm"]) / rec["norm"])


# named configurations of tests/test_oracle.py: (family, config, seed, batch)
REF_NAMED = [("tp", "tp_tiny", 101, 2), ("tp", "tp_tiny1", 102, 2), ("tp", "tp_tiny_de", 103, 2), ("ip", "ip_tiny", 104, 2),
             ("ip", "ip_cfg1", 105, 2), ("tps", "tps_tiny", 106, 2), ("tps", "tps_tiny4", 107, 2), ("tps", "tps_mid", 108, 1)]
SELECT_LISTS = [[1, 2, 4], [0, 2, 3], [2, 2, 3], [3, 2, 1]]


def _reference_run(fam, cfg, sd, x):
    build = {"tp": ref_loader.build_taskprompter, "ip": ref_loader.build_invpt, "tps": ref_loader.build_taskprompter_swin}[fam]
    model = build(cfg).eval()
    ref_sd = model.state_dict()
    if fam == "tps":
        missing, unexpected = model.load_state_dict(sd, strict=False)   # index / mask buffers are derived, not stored
        assert not unexpected and all("relative_position_index" in k or "attn_mask" in k for k in missing)
    else:
        model.load_state_dict(sd, strict=True)
    with torch.no_grad():
        y = model(x)
    rec = {"out": {t: summarize(y[t]) for t in cfg["tasks"]},
           "inter_preds": {t: summarize(y["inter_preds"][t]) for t in cfg["tasks"]} if fam == "ip" else None}
    derived = ("relative_position_index", "attn_mask")
    params = [(k, v.shape) for k, v in ref_sd.items() if not any(d in k for d in derived)]
    return rec, params


def _reference_raises(fam, cfg, x):
    build = ref_loader.build_invpt if fam == "ip" else ref_loader.build_taskprompter_swin
    try:
        with torch.no_grad():
            build(cfg).eval()(x)
    except (RuntimeError, AssertionError) as ex:
        return type(ex).__name__
    return None


def make_reference_checks():
    import importlib

    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_random_configs as RC

    oracle_of = {"tp": "oracle.taskprompter_ref", "ip": "oracle.invpt_ref", "tps": "oracle.taskprompter_swin_ref"}
    cases = {}
    for fam, name, seed, batch in REF_NAMED:
        cfg = (configs.taskprompter if fam == "tp" else configs.invpt if fam == "ip" else configs.taskprompter_swin)(name)
        sd = perturb(importlib.import_module(oracle_of[fam]).init_state_dict(cfg, seed=seed), seed + 1, swin=fam == "tps")
        x = torch.randn(batch, 3, *cfg["img_size"], generator=torch.Generator().manual_seed(seed + 1000))
        rec, params = _reference_run(fam, cfg, sd, x)
        rec.update(seed=seed, batch=batch, sorted_param_signature=signature(sorted(params)))
        cases[name] = rec
    for seed in range(6):                   # test_oracle_vs_reference_on_random_geometries
        cfg, B = RC.draw(seed)
        sd = perturb(importlib.import_module(oracle_of["tp"]).init_state_dict(cfg, seed=seed), seed + 1)
        x = torch.randn(B, 3, *cfg["img_size"], generator=torch.Generator().manual_seed(seed + 1000))
        cases[f"random_tp{seed}"] = _reference_run("tp", cfg, sd, x)[0]
    for seed in range(6):                   # test_invpt_launch_plan_and_oracle_on_random_geometries: the test's own weights
        cfg, B = RC.draw_invpt(seed)
        torch.manual_seed(seed)
        x = torch.randn(B, 3, *cfg["img_size"])
        cases[f"random_ip{seed}"] = _reference_run("ip", cfg, importlib.import_module(oracle_of["ip"]).init_state_dict(cfg, seed=seed), x)[0]
    for seed in range(8):                   # test_swin_launch_plan_and_oracle_on_random_geometries: the test's own weights
        cfg, B = RC.draw_swin(seed)
        torch.manual_seed(seed)
        x = torch.randn(B, 3, *cfg["img_size"])
        sd = importlib.import_module(oracle_of["tps"]).init_state_dict(cfg, seed=seed)
        cases[f"random_swin{seed}"] = _reference_run("tps", cfg, sd, x)[0]
    for sel in SELECT_LISTS:                # test_unusual_select_lists_follow_the_reference
        cfg = dict(RC._TP_BASE, select=sel)
        sd = perturb(importlib.import_module(oracle_of["tp"]).init_state_dict(cfg, seed=5), 6)
        x = torch.randn(2, 3, 64, 64, generator=torch.Generator().manual_seed(1005))
        cases["select_" + "-".join(map(str, sel))] = _reference_run("tp", cfg, sd, x)[0]
    raises = {"ip_6x6": _reference_raises("ip", dict(tasks=["edge", "semseg"], num_output={"edge": 1, "semseg": 5},
                                                     img_size=(96, 96), patch=16, C=128, depth=4, heads=2, select=[1, 2, 3],
                                                     embed_dim=32, pred_const=16, down=2, name="ip_6x6"), torch.randn(1, 3, 96, 96))}
    for change, match in RC.SWIN_REJECTS:
        cfg = dict(RC.SWIN_BAD, **change)
        raises[match] = _reference_raises("tps", cfg, torch.randn(1, 3, *cfg["img_size"]))
    swin_b = ref_loader.build_taskprompter_swin(configs.taskprompter_swin("tps_swinB")).state_dict()
    params = sorted((k, v.shape) for k, v in swin_b.items() if "relative_position_index" not in k and "attn_mask" not in k)
    return {"family": "reference_checks", "cases": cases, "raises": raises,
            "tps_swinB": {"sorted_param_signature": signature(params), "n_params": len(params)}, "torch": torch.__version__,
            "made_by": "oracle/make_golden.py refchecks: the unmodified reference forward (eval, fp32, CPU), summarised"}


def main():
    if not ref_loader.available():
        raise SystemExit("reference not found (set MTT_REFERENCE or mount /root/reference)")
    os.makedirs(GOLD, exist_ok=True)
    jobs = [("taskprompter", "tp_tiny", 3, 2), ("taskprompter", "tp_tiny1", 4, 2), ("taskprompter", "tp_tiny_de", 8, 2),
            ("taskprompter_swin", "tps_tiny", 11, 2), ("taskprompter_swin", "tps_tiny4", 12, 2)]
    if os.environ.get("MTT_GOLDEN_ONLY") in ("tp_tiny_de", "tps_tiny", "tps_tiny4"):
        jobs = [j for j in jobs if j[1] == os.environ["MTT_GOLDEN_ONLY"]]
    elif os.path.exists(os.path.join(ROOT, "oracle", "invpt_ref.py")):
        jobs += [("invpt", "ip_tiny", 5, 2), ("invpt", "ip_cfg1", 6, 2)]
    path = os.path.join(GOLD, "preproc.pt")
    torch.save(make_preproc(), path)
    print(f"wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)")
    if os.environ.get("MTT_GOLDEN_ONLY") == "preproc":
        return
    if os.environ.get("MTT_GOLDEN_ONLY") in (None, "", "losses"):
        path = os.path.join(GOLD, "losses.pt")
        torch.save(make_losses(), path)
        print(f"wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)")
        if os.environ.get("MTT_GOLDEN_ONLY") == "losses":
            return
    for fam, name, seed, batch in jobs:
        fx = {"taskprompter": make_taskprompter, "taskprompter_swin": make_taskprompter_swin,
              "invpt": make_invpt}[fam](name, seed, batch)
        path = os.path.join(GOLD, f"{name}.pt")
        torch.save(fx, path)
        print(f"wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)")


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "big":      # python -m oracle.make_golden big [config ...]
        if not ref_loader.available():
            raise SystemExit("reference not found (set MTT_REFERENCE or mount /root/reference)")
        main_big(set(sys.argv[2:]) or None)
    elif len(sys.argv) > 1 and sys.argv[1] == "train":  # python -m oracle.make_golden train [config ...]
        if not ref_loader.available():
            raise SystemExit("reference not found (set MTT_REFERENCE or mount /root/reference)")
        main_train(set(sys.argv[2:]) or None)
    elif len(sys.argv) > 1 and sys.argv[1] == "refchecks":   # python -m oracle.make_golden refchecks
        if not ref_loader.available():
            raise SystemExit("reference not found (set MTT_REFERENCE to the reference tree)")
        path = os.path.join(GOLD, "reference_checks.pt")
        torch.save(make_reference_checks(), path)
        print(f"wrote {path} ({os.path.getsize(path) / 1024:.0f} KiB)")
    else:
        main()
