"""CPU: host-side pieces either side of the denoising path (SURVEY.md 8f) against what the unmodified reference
computes and writes (golden fixtures from tests/golden/make_golden.py): train_batch control flow
(trainer.py:13-97), checkpoint files (unet.py:794-832, model_ema.py:36-55) and the gradient-adoption contract of
the flat arena."""
import argparse
import copy
import os
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "..", "ml-mdm_b200"))
sys.path.insert(0, os.path.join(HERE, ".."))
from oracle.optim_ref import ema_update_  # noqa: E402

GOLD = os.path.join(HERE, "golden")


class _Ema:
    """The parts of the reference's ModelEma (model_ema.py:13-34) that train_batch uses: a deep copy in eval mode,
    update() with warm-up, counter."""

    def __init__(self, model, decay, warmup_steps=0):
        self.module = copy.deepcopy(model).eval()
        self.decay, self.warmup_steps, self.counter = decay, warmup_steps, 0

    def update(self, model):
        decay = (self.counter >= self.warmup_steps) * self.decay
        self.counter += 1
        with torch.no_grad():
            msd = model.state_dict()
            for k, v in self.module.state_dict().items():
                ema_update_(v, msd[k].detach(), decay)


def trainer_record(pipe, ema, out):
    """What the control-flow tests compare: per-step (loss, lr), the final parameters, the EMA copy, its counter."""
    rec = {"loss": np.array([o[0] for o in out], dtype=np.float64), "lr": np.array([o[1] for o in out], dtype=np.float64),
           "counter": np.array(ema.counter)}
    rec.update({"model__" + k: v.numpy().copy() for k, v in pipe.state_dict().items()})
    rec.update({"ema__" + k: v.numpy().copy() for k, v in ema.module.state_dict().items()})
    return rec


def assert_same_record(got, tag):
    """Against what the reference's train_batch + ModelEma produced. The learning rates and the EMA counter are pure
    control flow and must match exactly. Losses and weights come out of small CPU matmuls whose last bit may depend
    on the host's BLAS path; they are compared to 1e-5 relative, far below the 2e-3 or more that one missed,
    repeated or mis-scaled optimiser step moves them (lr 1e-2 decaying as 1 / (1 + step)). NaN losses compare
    equal."""
    gold = np.load(os.path.join(GOLD, "trainer_steps.npz"))
    want = {k[len(tag) + 1:]: gold[k] for k in gold.files if k.startswith(tag + "/")}
    assert sorted(got) == sorted(want)
    for k in want:
        if k in ("lr", "counter"):
            assert np.array_equal(got[k], want[k]), (tag, k)
        else:
            np.testing.assert_allclose(got[k], want[k], rtol=1e-5, atol=1e-6, equal_nan=True, err_msg=f"{tag} {k}")


# ------------------------------------------------------------------ train_batch
class _Vision(nn.Module):
    def __init__(self):
        super().__init__()
        torch.manual_seed(3)
        self.a = nn.Linear(6, 8)
        self.b = nn.Linear(8, 6)

    def forward(self, x):
        return self.b(torch.tanh(self.a(x)))


class _Inner(nn.Module):
    def __init__(self):
        super().__init__()
        self.vision_model = _Vision()


class _Pipe(nn.Module):
    """What train_batch touches of a Diffusion pipeline: .model.vision_model and .get_loss(sample)."""

    def __init__(self, weighted):
        super().__init__()
        self.model = _Inner()
        self.weighted = weighted

    def get_loss(self, sample):
        x = sample["x"]
        pred = self.model.vision_model(x)
        losses = ((pred - sample["y"]) ** 2).mean(dim=1)
        weights = sample["w"] if self.weighted else None
        return losses, torch.zeros(x.shape[0]), x, pred, sample["y"], weights


def _run(train_batch, ModelEma, weighted):
    pipe = _Pipe(weighted)
    opt = torch.optim.Adam(pipe.model.vision_model.parameters(), lr=1e-2, eps=1e-8)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda s: 1.0 / (1 + s))
    ema = ModelEma(pipe.model.vision_model, decay=0.9, warmup_steps=1)
    args = argparse.Namespace(fp16=False, gradient_clip_norm=0.05)
    g = torch.Generator().manual_seed(1)
    out = []
    for step in range(5):
        s = {"x": torch.randn(4, 6, generator=g), "y": torch.randn(4, 6, generator=g), "w": torch.rand(4, generator=g)}
        if step == 2:
            s["x"][0, 0] = float("nan")          # NaN loss: trainer.py:69-74
        accumulate = step == 3                  # no optimizer step / zero_grad on this one
        r = train_batch(pipe, s, opt, sched, None, args, accumulate_gradient=accumulate,
                        num_grad_accumulations=2 if accumulate else 1, ema_model=ema)
        out.append((r[0], sched.get_last_lr()[0]))
    return pipe, ema, out


@pytest.mark.parametrize("weighted", [False, True])
def test_train_batch_mirrors_reference_control_flow(weighted):
    from mdm_b200 import trainer as my_trainer

    assert_same_record(trainer_record(*_run(my_trainer.train_batch, _Ema, weighted)), f"weighted{int(weighted)}")


def _run_fp16(train_batch, ModelEma):
    """args.fp16 branch (trainer.py:29-61) with a disabled GradScaler (bf16 autocast needs no loss scaling; CPU has no
    CUDA scaler): loss_factor, pre-backward accumulation divide, NaN path without optimizer/scheduler step."""
    pipe = _Pipe(True)
    opt = torch.optim.Adam(pipe.model.vision_model.parameters(), lr=1e-2, eps=1e-8)
    sched = torch.optim.lr_scheduler.LambdaLR(opt, lambda s: 1.0 / (1 + s))
    ema = ModelEma(pipe.model.vision_model, decay=0.9, warmup_steps=1)
    args = argparse.Namespace(fp16=True, gradient_clip_norm=0.05)
    scaler = torch.amp.GradScaler("cuda", enabled=False)
    g = torch.Generator().manual_seed(1)
    out = []
    for step in range(6):
        s = {"x": torch.randn(4, 6, generator=g), "y": torch.randn(4, 6, generator=g), "w": torch.rand(4, generator=g)}
        if step == 2:
            s["x"][0, 0] = float("nan")
        accumulate = step == 3
        r = train_batch(pipe, s, opt, sched, None, args, grad_scaler=scaler, accumulate_gradient=accumulate,
                        num_grad_accumulations=2 if step in (3, 4) else 1, ema_model=ema, loss_factor=0.5)
        out.append((r[0], sched.get_last_lr()[0]))
    return pipe, ema, out


def test_train_batch_fp16_branch_mirrors_reference_control_flow():
    from mdm_b200 import trainer as my_trainer

    assert_same_record(trainer_record(*_run_fp16(my_trainer.train_batch, _Ema)), "fp16")


# ------------------------------------------------------------------ checkpoints
def checkpoint_layout(ck):
    """Top-level keys of a checkpoint dict and (name, shape, dtype) of every state_dict entry, in order."""
    return list(ck), [(k, "x".join(str(d) for d in v.shape), str(v.dtype)) for k, v in ck["state_dict"].items()]


def read_layout(kind):
    lines = open(os.path.join(GOLD, f"checkpoint_{kind}.txt")).read().strip().split("\n")
    return lines[0].split(), [tuple(l.split()) for l in lines[1:]]


@pytest.mark.parametrize("kind", ["unet", "nested"])
def test_checkpoint_files_interchange_with_reference(kind, tmp_path):
    """The file the reference's save() writes, {"state_dict": ..., **other_items} (golden: its layout for the tiny
    configs), loads into our module; our save() writes that same layout, so the reference's load() and ModelEma.load
    (which read ck["state_dict"] and hand back the other items) take it."""
    import tiny_configs as tc
    from mdm_b200 import config as mc
    from mdm_b200.models import NestedUNet, UNet

    top, entries = read_layout(kind)
    assert top == ["state_dict", "batch_num", "args"]
    def new_model():
        cfg = mc.unet_config_from_dict(copy.deepcopy(tc.TINY_UNET if kind == "unet" else tc.TINY_NESTED))
        cfg.conditioning_feature_dim = tc.LM_DIM
        return (UNet if kind == "unet" else NestedUNet)(3, 3, cfg)

    mine = new_model()
    # reference -> ours: a file in the reference's layout
    g = torch.Generator().manual_seed(0)
    sd = {k: (0.3 * torch.randn([int(d) for d in shape.split("x") if d], generator=g)).to(getattr(torch, dt[6:]))
          for k, shape, dt in entries}
    f1 = str(tmp_path / "vis_model_ref.pth")
    torch.save({"state_dict": sd, "batch_num": 41}, f1)
    items = mine.load(f1)
    assert items["batch_num"] == 41
    for (k, a), (k2, b) in zip(sd.items(), mine.state_dict().items()):
        assert k == k2 and torch.equal(a, b), k
    # ours -> reference: the model file, and the EMA file (ModelEma saves its deep copy's state_dict the same way)
    with torch.no_grad():
        for p in mine.parameters():
            p.mul_(1.5)
    f2 = str(tmp_path / "vis_model_mine.pth")
    mine.save(f2, other_items={"batch_num": 42, "args": {"lr": 1e-4}})
    ck = torch.load(f2, map_location="cpu")
    assert checkpoint_layout(ck) == (top, entries)
    assert ck["batch_num"] == 42 and ck["args"] == {"lr": 1e-4}
    for (k, a), (_, b) in zip(mine.state_dict().items(), ck["state_dict"].items()):
        assert torch.equal(a, b), k
    # EMA file: ModelEma deep-copies our module and saves {"state_dict": copy.state_dict(), **other_items}; the
    # averaged weights (0.5 * 1.5 w + 0.5 * 2.25 w) differ from the module's, and load back into a fresh module
    ema = _Ema(mine, decay=0.5)
    with torch.no_grad():
        for p in mine.parameters():
            p.mul_(1.5)
    ema.update(mine)
    f3 = str(tmp_path / "ema.pth")
    torch.save({"state_dict": ema.module.state_dict(), "batch_num": 42, "args": None}, f3)
    ck = torch.load(f3, map_location="cpu")
    assert checkpoint_layout(ck) == (top, entries)
    fresh = new_model()
    assert fresh.load(f3)["batch_num"] == 42
    for (k, a), (_, b), (_, c) in zip(ema.module.state_dict().items(), fresh.state_dict().items(),
                                      mine.state_dict().items()):
        assert torch.equal(a, b), k
        assert k.endswith("t_emb") or not torch.equal(a, c) or float(a.abs().max()) == 0, k


# ------------------------------------------------------------------ gradient adoption
def test_arena_views_are_adopted_not_cloned():
    """`.grad` must alias the flat arena after backward (one all-reduce, FusedAdam, GradientOverlap depend on it).
    autograd adopts an incoming gradient only if nothing else references it."""
    from mdm_b200.models.native import ARENA_ALIGN, _pad, arena_views

    ps = [nn.Parameter(torch.randn(3, 4)), nn.Parameter(torch.randn(5)), nn.Parameter(torch.randn(2, 2, 3))]
    offs, total = [], 0
    for p in ps:
        offs.append(total)
        total += _pad(p.numel())
    assert all(o % ARENA_ALIGN == 0 for o in offs)
    arena = torch.zeros(total)

    class Fn(torch.autograd.Function):
        @staticmethod
        def forward(ctx, x, *params):
            return x.sum() + 0 * sum(p.sum() for p in params)

        @staticmethod
        def backward(ctx, g):
            arena.fill_(2.0)
            return (None, *arena_views(arena, ps, offs))

    Fn.apply(torch.randn(3, requires_grad=True), *ps).backward()
    lo, hi = arena.data_ptr(), arena.data_ptr() + 4 * arena.numel()
    assert all(lo <= p.grad.data_ptr() < hi for p in ps)
    assert all(p.grad.shape == p.shape and float(p.grad.min()) == 2.0 for p in ps)
