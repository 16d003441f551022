"""Pins the oracle (oracle/*.py) against the golden fixtures generated from the unmodified reference
(tests/golden/make_golden.py)."""
import copy
import hashlib
import json
import os
import types

import numpy as np
import pytest
import torch

import tiny_configs as tc
from oracle import diffusion_ref as dref
from oracle import unet_ref

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def ns(d):
    if isinstance(d, dict):
        return types.SimpleNamespace(**{k: ns(v) for k, v in d.items()})
    return d


def tiny(kind):
    nested = kind == "nested"
    ucfg = copy.deepcopy(tc.TINY_NESTED if nested else tc.TINY_UNET)
    if nested:
        ucfg["initialize_inner_with_pretrained"] = None
    net = unet_ref.OracleNet(ns(ucfg), tc.LM_DIM)
    names = open(os.path.join(GOLD, f"tiny_{kind}_params.txt")).read().split()
    gold = np.load(os.path.join(GOLD, f"tiny_{kind}.npz"))
    return net, names, gold, nested


def params_for(kind, names, requires_grad=False):
    # shapes come from the golden fixture-independent module tree: rebuild through the product container
    from mdm_b200 import config as mc
    from mdm_b200.models import NestedUNet, UNet

    ucfg = copy.deepcopy(tc.TINY_NESTED if kind == "nested" else tc.TINY_UNET)
    cfg = mc.unet_config_from_dict(ucfg)
    cfg.conditioning_feature_dim = tc.LM_DIM
    m = (NestedUNet if kind == "nested" else UNet)(3, 3, cfg)
    assert [k for k, _ in m.named_parameters()] == names
    sd = tc.seeded_state_dict(m.state_dict(), 7)
    return {k: v.clone().requires_grad_(requires_grad) for k, v in sd.items()}


def close(a, b, tol=2e-5):
    a = torch.as_tensor(a).double()
    b = torch.as_tensor(b).double()
    err = float((a - b).abs().max() / b.abs().max().clamp_min(1e-30))
    assert err <= tol, err


@pytest.mark.parametrize("kind", ["unet", "nested"])
def test_forward_matches_reference_golden(kind):
    net, names, gold, nested = tiny(kind)
    P = params_for(kind, names)
    x, t, lm, mask = tc.seeded_inputs(3, 2, 32 if nested else 16, 6, nlevels=2 if nested else 1)
    with torch.no_grad():
        out = net.forward(P, x, t, lm, mask, {})
    for i, o in enumerate(out if nested else [out]):
        close(o, gold[f"fwd_out{i}"])


@pytest.mark.parametrize("kind", ["unet", "nested"])
def test_loss_and_gradients_match_reference_golden(kind):
    net, names, gold, nested = tiny(kind)
    P = params_for(kind, names, requires_grad=True)
    x, t, lm, mask = tc.seeded_inputs(3, 2, 32 if nested else 16, 6, nlevels=2 if nested else 1)
    images = (x[0] if nested else x).clamp(-1, 1)
    gam = dref.gammas_f32("DEEPFLOYD", 1000)
    torch.manual_seed(1234)  # same CPU generator draws as Diffusion.get_loss (samplers.py:236-241)
    time = torch.randint(0, 1000, (2,))
    eps = [torch.randn_like(images)]
    scales = [4, 1] if nested else [1]
    if nested:
        eps.append(torch.empty(2, 3, 8, 8).normal_())
    assert np.array_equal(time.numpy(), gold["loss_time"])
    loss, x_t, outs = dref.training_loss(net, P, images, eps, time, lm, mask, gam, scales, dref.V_PREDICTION, dref.DDPM,
                                         shifted=nested, power=1)
    close(x_t[0], gold["loss_xt"], 1e-6)
    close(loss, gold["loss"])
    loss.mean().backward()
    norms = np.array([float(P[k].grad.norm()) for k in names])
    ref = gold["grad_norms"]
    floor = 1e-3 * np.median(ref)
    assert np.max(np.abs(norms - ref) / np.maximum(ref, floor)) < 1e-3
    for k in gold.files:
        if k.startswith("grad__"):
            close(P[k[6:]].grad, gold[k], 2e-4)


@pytest.mark.parametrize("kind", ["unet", "nested"])
def test_reverse_steps_and_sampling_match_reference_golden(kind):
    net, names, gold, nested = tiny(kind)
    P = params_for(kind, names)
    x, t, lm, mask = tc.seeded_inputs(3, 2, 32 if nested else 16, 6, nlevels=2 if nested else 1)
    xs = list(x) if nested else [x]
    scales = [4, 1] if nested else [1]
    gam = dref.gammas_f32("DEEPFLOYD", 1000)
    tabs = [dref.shift_table(gam, s, 1) if nested else gam for s in scales]
    times = torch.full((2,), 499, dtype=torch.long)
    with torch.no_grad():
        o = net.forward(P, xs if nested else xs[0], times, lm, mask, {})
        o = list(o) if nested else [o]
        for i, (xi, p, tab) in enumerate(zip(xs, o, tabs)):
            x0, x_s = dref.reverse_step(xi, p, tab[500], tab[480], dref.V_PREDICTION, True, 1.0, 0.0, True)
            close(x0, gold[f"ddim_x0_{i}"])
            close(x_s, gold[f"ddim_xs_{i}"])
        torch.manual_seed(99)
        for i, (xi, p, tab) in enumerate(zip(xs, o, tabs)):
            _, x_s = dref.reverse_step(xi, p, tab[500], tab[499], dref.V_PREDICTION, True, 1.0, None, True)
            close(x_s, gold[f"ddpm_xs_{i}"])
        # classifier-free guidance, rows [uncond; cond]
        lm2 = torch.cat([torch.zeros_like(lm), lm])
        mask2 = torch.cat([mask, mask])
        o2 = net.forward(P, [torch.cat([a, a]) for a in xs] if nested else torch.cat([xs[0], xs[0]]),
                         torch.cat([times, times]), lm2, mask2, {})
        o2 = list(o2) if nested else [o2]
        for i, (xi, p, tab) in enumerate(zip(xs, o2, tabs)):
            u, c = p.chunk(2)
            _, x_s = dref.reverse_step(xi, u + 3.0 * (c - u), tab[500], tab[480], dref.V_PREDICTION, True, 1.0, 0.0, True)
            close(x_s, gold[f"cfg_xs_{i}"])
        torch.manual_seed(7)
        init = [xs[0]] + ([torch.empty(2, 3, 8, 8).normal_()] if nested else [])
        final = dref.sample_loop(net, P, init, lm, mask, gam, scales, dref.V_PREDICTION, 1000, 4, 0.0, shifted=nested)
        close(final[0], gold["sample4"], 5e-5)


def test_schedule_tables_and_timesteps_bit_exact():
    g = np.load(os.path.join(GOLD, "schedules.npz"))
    for st in ["DEEPFLOYD", "DDPM", "COSINE"]:
        tab = dref.gammas_f32(st, 1000)
        assert np.array_equal(tab.numpy().view(np.uint32), g[f"gammas_{st}"].view(np.uint32)), st
        assert np.array_equal(dref.vdm_weights(tab).numpy().view(np.uint32), g[f"vdm_{st}"].view(np.uint32)), st
    base = dref.gammas_f32("DEEPFLOYD", 1000)
    for p, scales in [(1, [4, 1]), (2, [16, 4, 1])]:
        for s in scales:
            got = dref.shift_table(base, s, p).numpy()
            assert np.array_equal(got.view(np.uint32), g[f"shift_p{p}_s{s}"].view(np.uint32)), (p, s)
    for n in [1, 2, 5, 50, 100, 250, 999, 1000]:
        assert np.array_equal(dref.set_timesteps(1000, n), g[f"timesteps_{n}"])
    # closed-form known answers derived from the reference code (SURVEY.md 8c)
    assert float(base[0]) == 1.0
    assert float(base[1]) == pytest.approx(0.9999586939811707, abs=0)
    assert float(base[500]) == pytest.approx(0.49384358525276184, abs=0)
    ts = dref.set_timesteps(1000, 50)
    assert len(ts) == 51 and list(ts[:4]) == [981, 962, 942, 922] and list(ts[-4:]) == [59, 39, 20, 0]


# (tokens, seed) of the full-width cases; batch 1, parameters and inputs from numpy seeds
SHIPPED = {"cc12m_64x64": (16, 0), "cc12m_256x256": (8, 1), "cc12m_1024x1024": (4, 2)}
SHIPPED_SAMPLE = 2048


def shipped_case(name):
    """Parameters (every tensor of the state_dict seeded, tc.seeded_state_dict) and inputs of one shipped config at
    full width; shapes come from the product's module tree, which test_host pins to the reference's state_dict."""
    import yaml

    from mdm_b200 import config as mc
    from mdm_b200.models import NestedUNet, UNet

    path = os.path.join(os.path.dirname(GOLD), "..", "ml-mdm_b200", "mdm_b200", "configs", name + ".yaml")
    ucfg, _, nested = mc.load_yaml_configs(path)
    with torch.device("meta"):
        m = (NestedUNet if nested else UNet)(3, 3, ucfg)
    tokens, seed = SHIPPED[name]
    P = tc.seeded_state_dict(m.state_dict(), seed)
    res = int(name.split("_")[1].split("x")[0])
    nlev = {64: 1, 256: 2, 1024: 3}[res]
    x, t, lm, mask = tc.seeded_inputs(seed, 1, res, tokens, lm_dim=2048, nlevels=nlev)
    return yaml.safe_load(open(path)), P, x, t, lm, mask, nested


def strip_pretrained(d):
    """Nested config dicts: no pretrained initialisation anywhere."""
    if isinstance(d, dict):
        if "initialize_inner_with_pretrained" in d:
            d["initialize_inner_with_pretrained"] = None
        for v in d.values():
            strip_pretrained(v)
    return d


def check_shipped(name):
    """Oracle forward vs the reference modules' forward on the same parameters and inputs. The reference's outputs
    are stored at fixed sample positions and as means over each image row."""
    y, P, x, t, lm, mask, nested = shipped_case(name)
    gold = np.load(os.path.join(GOLD, f"shipped_{name}.npz"))
    net = unet_ref.OracleNet(ns(strip_pretrained(copy.deepcopy(y["unet_config"]))), 2048)
    with torch.no_grad():
        out = net.forward(P, x, t, lm, mask, {})
    out = list(out) if nested else [out]
    assert len(out) == len([k for k in gold.files if k.startswith("sample")])
    for i, o in enumerate(out):
        assert list(o.shape) == list(gold[f"shape{i}"])
        close(tc.golden_sample(o, SHIPPED_SAMPLE, seed=i), gold[f"sample{i}"], 1e-5)
        close(o.mean(dim=3), gold[f"rowmean{i}"], 1e-5)


def test_oracle_matches_live_reference_on_shipped_64_config():
    """cc12m_64x64 at full width (461 M parameters), B=1, S=16: oracle vs the reference modules."""
    check_shipped("cc12m_64x64")


def test_oracle_matches_live_reference_on_shipped_256_config():
    """cc12m_256x256 at full width (2-level nest, 476.6 M parameters), B=1, S=8: oracle vs the reference's
    NestedUNet — pins the nesting adapters, the inner/outer skip wiring and the 4x resolution ratio at the real
    channel widths (the tiny nested fixture pins them at toy widths)."""
    check_shipped("cc12m_256x256")


def test_oracle_matches_live_reference_on_shipped_1024_config():
    """cc12m_1024x1024 at full width (3-level nest, 481 M parameters), B=1, S=4: oracle vs the reference."""
    check_shipped("cc12m_1024x1024")


MIXED_B = 3
GRAD_SAMPLE = 64  # gradient elements stored per parameter: the whole gradient for 242 of the 461


def test_oracle_mixed_ratio_loss_matches_live_reference():
    """NestedDiffusion.get_loss with mixed_ratio='2:1' (what configs/models/cc12m_256x256.yaml:108 sets): only the
    leading int(2/3 * B) samples run the high-resolution level, predictions are zero-padded, the per-level loss is
    divided by the fraction and masked (diffusion.py:262-274, 378-382; nested_unet.py:180,193-204,209). The oracle
    replays the reference's CPU generator draws; loss, x_t and every gradient (its norm, and GRAD_SAMPLE elements
    at fixed positions) are compared with what the reference computed."""
    B = MIXED_B
    gold = np.load(os.path.join(GOLD, "tiny_nested_mixed.npz"))
    names = open(os.path.join(GOLD, "tiny_nested_params.txt")).read().split()
    P = params_for("nested", names, requires_grad=True)
    x, t, lm, mask = tc.seeded_inputs(3, B, 32, 6, nlevels=2)
    images = x[0].clamp(-1, 1)
    torch.manual_seed(4321)  # the draws of the reference's get_loss
    time = torch.randint(0, 1000, (B,))
    eps = [torch.randn_like(images), None]
    eps[1] = torch.empty(B, 3, 8, 8).normal_()
    assert np.array_equal(time.numpy(), gold["time"])
    ocfg = copy.deepcopy(tc.TINY_NESTED)
    ocfg["initialize_inner_with_pretrained"] = None
    net = unet_ref.OracleNet(ns(ocfg), tc.LM_DIM)
    gam = dref.gammas_f32("DEEPFLOYD", 1000)
    mr = dref.mixed_ratio_fractions("2:1")
    assert int(mr[0] * B) == 2 and mr[1] == 1.0
    oloss, ox_t, _ = dref.training_loss(net, P, images, eps, time, lm, mask, gam, [4, 1], dref.V_PREDICTION, dref.DDPM,
                                        shifted=True, power=1, mixed_ratio=mr)
    close(ox_t[0], gold["x_t"], 1e-6)
    close(oloss.detach(), gold["loss"])
    oloss.mean().backward()
    # Biases in front of a GroupNorm get gradients that are mathematically zero (the reference's are below 4e-8,
    # every other one above 1e-3): their values are rounding noise, which differs between CPUs. Those must stay
    # below 1e-3 of the median gradient norm; every other gradient is compared with the reference's.
    norms = np.array([float(P[k].grad.norm()) for k in names])
    ref = gold["grad_norms"]
    zero = ref < 1e-3 * np.median(ref)
    assert np.all(norms[zero] < 1e-3 * np.median(ref))
    assert np.max(np.abs(norms - ref)[~zero] / ref[~zero]) < 1e-3
    for i, k in enumerate(names):  # close() of the whole gradient, at the stored positions
        if zero[i]:
            continue
        got = tc.golden_sample(P[k].grad, GRAD_SAMPLE, seed=i).double()
        want = torch.from_numpy(gold["grad_sample"][i, :got.numel()]).double()
        assert float((got - want).abs().max()) <= 2e-4 * float(gold["grad_absmax"][i]), k


CLIP_MODES = ["DYNAMIC", "DYNAMIC_IF", "CLIP", "NONE"]


def clip_input():
    g = torch.Generator().manual_seed(3)
    return torch.randn(3, 3, 32, 32, generator=g) * torch.tensor([0.4, 1.3, 9.0]).view(3, 1, 1, 1)


def digest(t):
    return hashlib.sha256(t.contiguous().numpy().tobytes()).hexdigest()


@pytest.mark.parametrize("mode", CLIP_MODES)
def test_oracle_clip_sample_matches_live_reference(mode):
    """Sampler.clip_sample incl. dynamic thresholding (samplers.py:461-508): bit-identical restatement, checked
    against the SHA-256 of the reference's float32 output bytes."""
    want = json.load(open(os.path.join(GOLD, "clip_sample.json")))[mode]
    x = clip_input()
    for scale in (1.0, 4.0):
        out = dref.clip_sample(x, scale, mode if mode != "NONE" else False)
        assert out.dtype == torch.float32 and out.shape == x.shape
        assert digest(out) == want[str(scale)], (mode, scale)
