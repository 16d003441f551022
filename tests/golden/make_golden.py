"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference
(imported through tests/refharness.py) on CPU in fp32.

    ML_MDM_ROOT=<ml-mdm-matryoshka directory> python tests/golden/make_golden.py [fixture ...]

ML_MDM_ROOT is the directory of an apple/ml-mdm checkout that holds the ml_mdm/ package and configs/models/.

The tests do not import the reference, so its outputs on seeded inputs are committed here:
  schedules.npz     gamma tables (float32 bits) for every schedule type / shift used by the configs,
                    vdm loss weights, set_timesteps() for several N
  tiny_unet.npz     tiny UNet: forward, get_loss (loss, model output, per-parameter gradient norms,
                    a few full gradients), one DDIM step, one DDPM step input/output, a 4-step DDIM sample
  tiny_nested.npz   the same for a 2-level NestedUNet (shifted schedule, double loss)
  keys_*.txt        state_dict key order + shapes of the three shipped configs
  shipped_*.npz     forward of each shipped config at full width, B=1 (fixed sample positions + row means)
  tiny_nested_mixed.npz  get_loss with mixed_ratio '2:1': loss, x_t, gradient norms / abs max / samples
  clip_sample.json  SHA-256 of Sampler.clip_sample's output for every threshold mode
  trainer_steps.npz train_batch + ModelEma on a toy pipeline (losses, lrs, final weights, EMA weights)
  checkpoint_*.txt  layout of the file UNet/NestedUNet.save() writes for the tiny configs
  reference_configs.json  the reference's model/pipeline registries, its config dataclasses (field names) and
                    sampler enums (members), and its config objects for cc12m_256x256 as its own loader builds them
Parameters and inputs come from numpy PCG64 seeds (tests/tiny_configs.py), so only outputs are stored.
Outputs too large to commit whole are stored at fixed positions (tiny_configs.golden_sample).
"""
import copy
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, ".."))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
sys.path.insert(0, os.path.join(HERE, "..", "..", "ml-mdm_b200"))

import refharness as rh  # noqa: E402
import tiny_configs as tc  # noqa: E402

torch.set_num_threads(8)
ref = rh.load()
S = ref.samplers


def schedules():
    out = {}
    for st in ["DEEPFLOYD", "DDPM", "COSINE"]:
        cfg = S.SamplerConfig(num_diffusion_steps=1000, schedule_type=S.ScheduleType[st])
        smp = S.Sampler(cfg)
        out[f"gammas_{st}"] = smp.gammas.numpy()
        out[f"vdm_{st}"] = smp.vdm_loss_weights.numpy()
    for power, scales in [(1, [4, 1]), (2, [16, 4, 1])]:
        cfg = S.SamplerConfig(num_diffusion_steps=1000, schedule_type=S.ScheduleType.DEEPFLOYD, schedule_shifted=True,
                              schedule_shifted_power=power)
        smp = S.NestedSampler(cfg)
        for s in scales:
            out[f"shift_p{power}_s{s}"] = smp.get_schedule_shifted(smp.gammas, s).numpy()
    # (rescale_schedule > 1 raises in the reference itself: Sampler.__init__ reads self._config before
    #  assigning it, samplers.py:183-190,259 -- every shipped config uses 1.0)
    smp = S.Sampler(S.SamplerConfig(num_diffusion_steps=1000, schedule_type=S.ScheduleType.DEEPFLOYD))
    for n in [1, 2, 5, 50, 100, 250, 999, 1000]:
        out[f"timesteps_{n}"] = smp.set_timesteps(n)
    np.savez_compressed(os.path.join(HERE, "schedules.npz"), **out)
    print("schedules.npz", len(out))


def model_case(kind):
    nested = kind == "nested"
    ucfg = copy.deepcopy(tc.TINY_NESTED if nested else tc.TINY_UNET)
    dcfg = copy.deepcopy(tc.TINY_NESTED_DIFFUSION if nested else tc.TINY_DIFFUSION)
    model, pipe = rh.build(ucfg, dcfg, "nested_unet" if nested else "unet", tc.LM_DIM)
    sd = tc.seeded_state_dict(model.state_dict(), 7)
    model.load_state_dict(sd)
    res = 32 if nested else 16
    nlev = 2 if nested else 1
    x, t, lm, mask = tc.seeded_inputs(3, 2, res, 6, nlevels=nlev)
    out = {}
    with torch.no_grad():
        o = model(x, t, lm, mask, {})
    for i, oi in enumerate(o if nested else [o]):
        out[f"fwd_out{i}"] = oi.numpy()

    # ---- get_loss with a pinned CPU RNG
    images = (x[0] if nested else x).clamp(-1, 1)
    torch.manual_seed(1234)
    pipe.train()
    loss, time, x_t, pred, tgt, _ = pipe.get_loss({"images": images, "lm_outputs": lm, "lm_mask": mask})
    loss.mean().backward()
    out["loss"] = loss.detach().numpy()
    out["loss_time"] = time.numpy()
    out["loss_xt"] = x_t.detach().numpy()
    out["loss_pred"] = pred.detach().numpy()
    out["loss_tgt"] = tgt.detach().numpy()
    names = [k for k, _ in model.named_parameters()]
    out["grad_norms"] = np.array([float(p.grad.norm()) for _, p in model.named_parameters()], dtype=np.float64)
    out["grad_absmax"] = np.array([float(p.grad.abs().max()) for _, p in model.named_parameters()], dtype=np.float64)
    pick = [n for n in names if n.endswith(("conv_in.weight", "mid_blocks.0.attn.0.kv_cond.weight", "temb_layer2.bias",
                                            "up_blocks.1.resnets.0.conv3.weight", "cond_emb.weight", "in_adapter.bias"))]
    for n in pick:
        out["grad__" + n] = dict(model.named_parameters())[n].grad.numpy()
    model.zero_grad()

    # ---- one reverse step (DDIM eta=0 and DDPM with pinned noise), then a 4-step DDIM sample
    pipe.eval()
    smp = pipe.sampler
    m = pipe.get_model()
    xin = x if nested else x
    with torch.no_grad():
        x0, xs, _ = smp.get_xt_minus_1(m, 500, [xi.clone() for xi in x] if nested else x.clone(), lm, mask, {},
                                       time_step_last=480, ddim_eta=0.0, return_details=True)
        for i, (a, b) in enumerate(zip(x0, xs) if nested else [(x0, xs)]):
            out[f"ddim_x0_{i}"], out[f"ddim_xs_{i}"] = a.numpy(), b.numpy()
        torch.manual_seed(99)
        xs = smp.get_xt_minus_1(m, 500, [xi.clone() for xi in x] if nested else x.clone(), lm, mask, {},
                                time_step_last=499, ddim_eta=None)
        for i, b in enumerate(xs if nested else [xs]):
            out[f"ddpm_xs_{i}"] = b.numpy()
        # CFG step: doubled conditioning rows [uncond; cond]
        lm2 = torch.cat([torch.zeros_like(lm), lm])
        mask2 = torch.cat([mask, mask])
        xs = smp.get_xt_minus_1(m, 500, [xi.clone() for xi in x] if nested else x.clone(), lm2, mask2, {},
                                time_step_last=480, ddim_eta=0.0, guidance_scale=3.0)
        for i, b in enumerate(xs if nested else [xs]):
            out[f"cfg_xs_{i}"] = b.numpy()
        # nested sampling starts from the full-resolution tensor; the low-resolution start is drawn inside
        # with normal_() (samplers.py:669-676) -> pinned by the seed below
        torch.manual_seed(7)
        final = smp.sample(m, x[0].clone() if nested else x.clone(), lm, mask, {}, num_inference_steps=4,
                           ddim_eta=0.0, resample_steps=True)
        out["sample4"] = final.numpy()
    np.savez_compressed(os.path.join(HERE, f"tiny_{kind}.npz"), **out)
    with open(os.path.join(HERE, f"tiny_{kind}_params.txt"), "w") as f:
        f.write("\n".join(names) + "\n")
    print(f"tiny_{kind}.npz", {k: v.shape for k, v in out.items() if k.startswith(("fwd", "loss", "sample"))})


def shipped_keys():
    for y, arch in [("cc12m_64x64", "unet"), ("cc12m_256x256", "nested_unet"), ("cc12m_1024x1024", "nested2_unet")]:
        cfg = rh.load_yaml(y + ".yaml")
        model, _ = rh.build(cfg["unet_config"], cfg["diffusion_config"], arch, 2048)
        with open(os.path.join(HERE, f"keys_{y}.txt"), "w") as f:
            for k, v in model.state_dict().items():
                f.write(f"{k} {'x'.join(str(d) for d in v.shape)}\n")
        print(y, sum(p.numel() for p in model.parameters()))


def shipped_outputs():
    import test_oracle as to

    for name in to.SHIPPED:
        y, P, x, t, lm, mask, nested = to.shipped_case(name)
        arch = {"cc12m_64x64": "unet", "cc12m_256x256": "nested_unet", "cc12m_1024x1024": "nested2_unet"}[name]
        model, _ = rh.build(y["unet_config"], y["diffusion_config"], arch, 2048)
        model.load_state_dict(P)
        with torch.no_grad():
            o = model(x, t, lm, mask, {})
        out = {}
        for i, oi in enumerate(o if nested else [o]):
            out[f"shape{i}"] = np.array(oi.shape)
            out[f"sample{i}"] = tc.golden_sample(oi, to.SHIPPED_SAMPLE, seed=i).numpy()
            out[f"rowmean{i}"] = oi.mean(dim=3).numpy()
        np.savez_compressed(os.path.join(HERE, f"shipped_{name}.npz"), **out)
        print(f"shipped_{name}.npz", {k: v.shape for k, v in out.items()})
        del model, P


def mixed_ratio_loss():
    import test_oracle as to

    B = to.MIXED_B
    dcfg = copy.deepcopy(tc.TINY_NESTED_DIFFUSION)
    dcfg["mixed_ratio"] = "2:1"
    model, pipe = rh.build(copy.deepcopy(tc.TINY_NESTED), dcfg, "nested_unet", tc.LM_DIM)
    model.load_state_dict(tc.seeded_state_dict(model.state_dict(), 7))
    x, t, lm, mask = tc.seeded_inputs(3, B, 32, 6, nlevels=2)
    torch.manual_seed(4321)
    pipe.train()
    loss, time, x_t, pred, tgt, _ = pipe.get_loss({"images": x[0].clamp(-1, 1), "lm_outputs": lm, "lm_mask": mask})
    loss.mean().backward()
    grads = [p.grad for _, p in model.named_parameters()]
    samples = np.zeros((len(grads), to.GRAD_SAMPLE), dtype=np.float32)
    for i, g in enumerate(grads):
        s_ = tc.golden_sample(g, to.GRAD_SAMPLE, seed=i).numpy()
        samples[i, :len(s_)] = s_
    out = {"loss": loss.detach().numpy(), "time": time.numpy(), "x_t": x_t.detach().numpy(),
           "grad_norms": np.array([float(g.norm()) for g in grads]),
           "grad_absmax": np.array([float(g.abs().max()) for g in grads]), "grad_sample": samples}
    np.savez_compressed(os.path.join(HERE, "tiny_nested_mixed.npz"), **out)
    print("tiny_nested_mixed.npz", {k: v.shape for k, v in out.items()})


def clip_sample():
    import json

    import test_oracle as to

    out = {}
    for mode in to.CLIP_MODES:
        cfg = S.SamplerConfig()
        smp = S.Sampler(cfg)
        cfg.threshold_function = getattr(S.ThresholdType, mode)
        out[mode] = {str(scale): to.digest(smp.clip_sample(to.clip_input(), scale)) for scale in (1.0, 4.0)}
    with open(os.path.join(HERE, "clip_sample.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("clip_sample.json", out)


def trainer_steps():
    import warnings

    import test_trainer_host as th
    from ml_mdm import trainer as ref_trainer
    from ml_mdm.models.model_ema import ModelEma

    out = {}
    for weighted in (False, True):
        rec = th.trainer_record(*th._run(ref_trainer.train_batch, ModelEma, weighted))
        out.update({f"weighted{int(weighted)}/{k}": v for k, v in rec.items()})
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")  # torch.cuda.amp.autocast on a CPU-only host warns and disables itself
        rec = th.trainer_record(*th._run_fp16(ref_trainer.train_batch, ModelEma))
    out.update({f"fp16/{k}": v for k, v in rec.items()})
    np.savez_compressed(os.path.join(HERE, "trainer_steps.npz"), **out)
    print("trainer_steps.npz", len(out))


def checkpoint_layouts():
    import tempfile

    import test_trainer_host as th

    for kind, arch in [("unet", "unet"), ("nested", "nested_unet")]:
        model, _ = rh.build(copy.deepcopy(tc.TINY_UNET if kind == "unet" else tc.TINY_NESTED), {}, arch, tc.LM_DIM)
        with tempfile.TemporaryDirectory() as d:
            f = os.path.join(d, "vis_model.pth")
            model.save(f, other_items={"batch_num": 42, "args": {"lr": 1e-4}})
            top, entries = th.checkpoint_layout(torch.load(f, map_location="cpu"))
        with open(os.path.join(HERE, f"checkpoint_{kind}.txt"), "w") as fh:
            fh.write(" ".join(top) + "\n" + "".join(" ".join(e) + "\n" for e in entries))
        print(f"checkpoint_{kind}.txt", len(entries))


def reference_configs():
    import dataclasses
    import enum
    import json

    C = ref.config
    classes, enums = {}, {}

    def enc(v):
        if isinstance(v, enum.Enum):
            enums[type(v).__name__] = {m.name: m.value for m in type(v)}
            return {"enum": type(v).__name__, "member": v.name}
        if dataclasses.is_dataclass(v):
            classes[type(v).__name__] = [f.name for f in dataclasses.fields(v)]
            return {"dataclass": type(v).__name__, "fields": {f.name: enc(getattr(v, f.name)) for f in dataclasses.fields(v)}}
        if isinstance(v, (list, tuple)):
            return [enc(x) for x in v]
        assert v is None or isinstance(v, (bool, int, float, str)), (type(v), v)
        return v

    for t in (S.ScheduleType, S.PredictionType, S.ThresholdType):
        enums[t.__name__] = {m.name: m.value for m in t}
    for cls in [e["config"] for e in C.MODEL_CONFIG_REGISTRY.values()] + list(C.PIPELINE_CONFIG_REGISTRY.values()):
        classes[cls.__name__] = [f.name for f in dataclasses.fields(cls)]
    y = rh.load_yaml("cc12m_256x256.yaml")
    objs = {"unet_config": enc(rh.from_dict(C.MODEL_CONFIG_REGISTRY["nested_unet"]["config"], y["unet_config"])),
            "diffusion_config": enc(rh.from_dict(C.PIPELINE_CONFIG_REGISTRY["nested_unet"], y["diffusion_config"]))}
    out = {"MODEL_CONFIG_REGISTRY": {k: {"model": v["model"], "config": v["config"].__name__}
                                     for k, v in C.MODEL_CONFIG_REGISTRY.items()},
           "PIPELINE_CONFIG_REGISTRY": {k: v.__name__ for k, v in C.PIPELINE_CONFIG_REGISTRY.items()},
           "MODEL_REGISTRY": list(C.MODEL_REGISTRY), "PIPELINE_REGISTRY": list(C.PIPELINE_REGISTRY),
           "classes": classes, "enums": enums, "cc12m_256x256": objs}
    with open(os.path.join(HERE, "reference_configs.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("reference_configs.json", sorted(classes), sorted(enums))


FIXTURES = {"schedules": schedules, "tiny_unet": lambda: model_case("unet"), "tiny_nested": lambda: model_case("nested"),
            "keys": shipped_keys, "shipped": shipped_outputs, "mixed_ratio": mixed_ratio_loss, "clip_sample": clip_sample,
            "trainer": trainer_steps, "checkpoint": checkpoint_layouts, "reference_configs": reference_configs}

if __name__ == "__main__":
    for name in sys.argv[1:] or list(FIXTURES):
        FIXTURES[name]()
