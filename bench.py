#!/usr/bin/env python
"""bench.py -- denoising steps/sec of the Matryoshka denoising path on N x B200.

    python bench.py --gpus 1 --steps 20 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --gpus 1 --steps 3 --warmup 1     # CPU arm (oracle port)

Headline (`value`): BASELINE.json configs[1] -- cc12m_64x64 U-Net training, batch 64 per GPU, random T5 embeddings
with S=128 tokens. One step = Diffusion.get_loss(sample) + loss.mean().backward(): q-sample, full U-Net forward, loss,
full backward with every parameter gradient, plus the one gradient all-reduce when N > 1. The optimizer sweep and the
fp16 weight repack it triggers are NOT in the step (the metric is fwd+bwd); `optimizer_sweep_ms` reports them.

The same line carries, under "configs", the other BASELINE.json configurations measured the same way (fewer steps):
  cc12m_256x256_train     configs[2]: 2-level nest, batch 32 per GPU (weak scaling)
  cc12m_1024x1024_train   configs[3]: 3-level nest, GLOBAL batch 8 split over the N GPUs (8 / N per GPU: strong scaling,
                          1 sample per GPU at N = 8 as BASELINE names it)
  cc12m_256x256_ddim50    configs[4]: DDIM 50-step sampling, batch 16 per GPU, no collective
Prints ONE JSON line. `--only <name>` / `--config/--batch` restrict the run (development aid).
`--dump-outputs DIR` writes what the headline's last timed step computed as DIR/<name>.npy (see dump_outputs), so
that two builds can be compared output for output: weights, inputs and random draws depend only on the arguments.
"""
import argparse
import gc
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "ml-mdm_b200"))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

# Algorithmic work per sample per forward, measured by hooking the reference modules with S=128 (SURVEY.md 8d,
# BASELINE.md section 3): FLOP = 2*MAC of every conv/linear + 4*B*C*T*S per attention; training = 3x.
# By level (outermost first): GFLOP and the activation elements a perfectly fused forward still has to move
# (each conv/linear/attention reads its input once and writes its output once), in M elements.
LEVELS = {
    "cc12m_64x64": [("64-core", 385.4, 261.0)],
    "cc12m_256x256": [("256-outer", 225.1, 281.0), ("64-core", 385.4, 261.0)],
    "cc12m_1024x1024": [("1024-outer", 429.5, 1686.0), ("256-mid", 225.1, 281.0), ("64-core", 385.4, 261.0)],
}
FWD_GFLOP = {k: round(sum(l[1] for l in v), 1) for k, v in LEVELS.items()}  # 385.4 / 610.5 / 1040.0
ATTN_FWD_GFLOP = 19.9  # of which attention (QK^T and PV); runs in the fused attention kernels, not the GEMM engine
PARAMS_M = {"cc12m_64x64": 461.4, "cc12m_256x256": 476.6, "cc12m_1024x1024": 481.0}
RES = {"cc12m_64x64": [64], "cc12m_256x256": [256, 64], "cc12m_1024x1024": [1024, 256, 64]}
TOKENS = 128


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1402.9), d.get("hbm_gbs", 6576.1), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def ideal_ms(cfg_name, batch, passes):
    """Roofline time of `passes` network passes (3 = fwd+bwd, 1 = inference) of `batch` samples: per level
    max(FLOP / measured tensor peak, fp16 activation bytes / measured HBM bandwidth), plus one read of the fp16
    weights per pass. This is SURVEY.md 8(d)'s 'conv+attention roofline'."""
    tf, bw, _ = measured_peaks()
    ms, parts = 0.0, []
    for name, gflop, melem in LEVELS[cfg_name]:
        t_tensor = gflop * 1e9 * batch * passes / (tf * 1e12) * 1e3
        t_hbm = melem * 1e6 * 2 * batch * passes / (bw * 1e9) * 1e3
        ms += max(t_tensor, t_hbm)
        parts.append({"level": name, "tensor_ms": round(t_tensor, 3), "hbm_ms": round(t_hbm, 3),
                      "bound": "tensor" if t_tensor >= t_hbm else "hbm"})
    ms += PARAMS_M[cfg_name] * 1e6 * 2 * passes / (bw * 1e9) * 1e3
    return ms, parts


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc, self.path = None, None
        try:
            self.path = tempfile.mktemp(suffix=".csv")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(index), "-lms", "200"], stdout=open(self.path, "w"),
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for line in open(self.path).read().strip().split("\n"):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_pipeline(cfg_name, device, mixed_ratio=None):
    from mdm_b200 import config as mc
    from mdm_b200.diffusion import Diffusion, NestedDiffusion
    from mdm_b200.models import NestedUNet, UNet

    ucfg, dcfg, nested = mc.load_yaml_configs(os.path.join(ROOT, "ml-mdm_b200", "mdm_b200", "configs", cfg_name + ".yaml"))
    if nested:
        dcfg.mixed_ratio = mixed_ratio
    torch.manual_seed(4321)
    model = (NestedUNet if nested else UNet)(3, 3, ucfg)
    with torch.no_grad():  # the reference zero-initialises ~1/3 of its layers; a trained net has none at zero
        for p in model.parameters():
            if float(p.detach().abs().max()) == 0:
                p.normal_(0, 0.02)
    pipe = (NestedDiffusion if nested else Diffusion)(model, dcfg).to(device)
    return pipe, nested


def synthetic_host_batch(cfg_name, B, seed):
    g = torch.Generator().manual_seed(seed)
    R = RES[cfg_name][0]
    return {
        "images": (torch.rand(B, 3, R, R, generator=g) * 2 - 1).pin_memory(),
        "lm_outputs": torch.randn(B, TOKENS, 2048, generator=g).pin_memory(),
        "lm_mask": torch.ones(B, TOKENS).pin_memory(),
    }


class Ctx:
    def __init__(self):
        import torch.distributed as dist

        self.dist = dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world > 1:
            if os.environ.get("MDM_OVERLAP") is not None and int(os.environ.get("MDM_SM_RESERVE", "0")) > 0:
                os.environ.setdefault("NCCL_MAX_CTAS", os.environ["MDM_SM_RESERVE"])  # the SMs the GEMMs leave free
            dist.init_process_group("nccl", init_method="env://")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, vals):
        if self.world == 1:
            return vals
        t = torch.tensor(vals, device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def free_pipeline(*objs):
    for o in objs:
        del o
    gc.collect()
    torch.cuda.empty_cache()


def timed(ctx, fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ctx.barrier()
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    ctx.barrier()
    return e0.elapsed_time(e1)


DUMP_IMAGE_ELEMS = 1 << 21  # larger image-shaped outputs are dumped at this many fixed positions
DUMP_GRAD_ELEMS = 4096      # gradient elements dumped per parameter
DUMP_MAX_BYTES = 64 << 20


def _fixed_positions(t, n, seed):
    """`t` flattened, at `n` positions drawn from a fixed seed (all of it when it has no more than `n` elements)."""
    flat = t.detach().reshape(-1)
    if flat.numel() <= n:
        return flat
    g = torch.Generator().manual_seed(seed)
    idx = torch.randint(flat.numel(), (n,), generator=g).sort().values
    return flat[idx.to(flat.device)]


def dump_outputs(path, outputs, vm):
    """Writes what one training step returned to its caller: get_loss's (loss, time, x_t, prediction, target[,
    weights]) and the parameter gradients. Image-shaped arrays above DUMP_IMAGE_ELEMS elements are written as
    <name>_sample.npy at fixed positions; gradients as grad_norms.npy (float64, one per parameter) and
    grad_sample.npy (DUMP_GRAD_ELEMS fixed positions of each parameter, zero-padded), in the order of
    grad_names.txt. The gradients are read from the engine's gradient arena, which holds the last backward's
    result until the next backward starts."""
    import numpy as np

    from mdm_b200.models import native

    names = ["loss", "time", "x_t", "pred", "target", "weights"]
    arrays = {}
    for i, (name, t) in enumerate(zip(names, outputs)):
        if t is None:
            continue
        dt = torch.float64 if t.dtype in (torch.int64, torch.float64) else torch.float32
        if t.numel() > DUMP_IMAGE_ELEMS:
            name, t = name + "_sample", _fixed_positions(t, DUMP_IMAGE_ELEMS, i)
        arrays[name] = t.detach().to(dt).cpu().numpy()
    nn_ = vm.native()
    grads = native.arena_views(nn_.active_arena, nn_.params, nn_.offsets)
    arrays["grad_norms"] = torch.stack([g.double().norm() for g in grads]).cpu().numpy()
    sample = torch.zeros(len(grads), DUMP_GRAD_ELEMS, device=grads[0].device)
    for i, g in enumerate(grads):
        s = _fixed_positions(g, DUMP_GRAD_ELEMS, i)
        sample[i, :s.numel()] = s
    arrays["grad_sample"] = sample.cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, total
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)
    with open(os.path.join(path, "grad_names.txt"), "w") as f:
        f.write("\n".join(nn_.param_names) + "\n")


def measure_train(ctx, cfg_name, B, steps, warmup, headline=False, mixed_ratio=None, dump_dir=None):
    """fwd+bwd sample-steps/s of one configuration at ctx.world GPUs; B = per-GPU batch. With `dump_dir`, what the
    last timed step computed is written there (dump_outputs)."""
    from mdm_b200 import _lib, parallel

    pipe, nested = build_pipeline(cfg_name, ctx.dev, mixed_ratio)
    pipe.train()
    vm = pipe.get_model().vision_model
    host = synthetic_host_batch(cfg_name, B, 1234 + ctx.rank)
    resident = {k: v.to(ctx.dev) for k, v in host.items()}
    overlap = (parallel.GradientOverlap(vm, bucket_mb=int(os.environ.get("MDM_BUCKET_MB", "64")),
                                        sm_reserve=int(os.environ.get("MDM_SM_RESERVE", "0")))
               if ctx.world > 1 and os.environ.get("MDM_OVERLAP") is not None else None)

    def step(sample):
        out = pipe.get_loss(sample)
        if overlap is not None:
            overlap.arm()
        out[0].mean().backward()
        if overlap is not None:
            overlap.finish()
        elif ctx.world > 1:
            parallel.allreduce_gradients(vm)
        return out

    def zero():
        vm.zero_grad(set_to_none=True)

    last = []  # the outputs of the latest step, kept only for dump_dir

    def resident_step():
        out = step(resident)
        if dump_dir is not None:
            last[:] = out
        zero()

    for _ in range(max(warmup, 3)):  # also sizes the engine's memory pool
        resident_step()
    clocks = ClockSampler(ctx.local) if (ctx.rank == 0 and headline) else None
    l0 = _lib.launch_count()
    ms = timed(ctx, resident_step, steps)
    launches = _lib.launch_count() - l0
    clk = clocks.stop() if clocks is not None else None
    if dump_dir is not None and ctx.rank == 0:
        dump_outputs(dump_dir, last, vm)
    del last[:]
    # ---- end to end: host (pinned) inputs, H2D inside the timed region, D2H of the loss
    loss_host = torch.empty(B).pin_memory()

    def e2e_step():
        sample = {k: v.to(ctx.dev, non_blocking=True) for k, v in host.items()}
        loss = step(sample)[0]
        loss_host.copy_(loss.detach(), non_blocking=True)
        zero()

    e2e_step()  # untimed: the first host-fed step allocates its device buffers (cudaMalloc in torch's allocator)
    ms_e2e = timed(ctx, e2e_step, steps)
    ms, ms_e2e = ctx.max_over_ranks([ms, ms_e2e])
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    gb = B * ctx.world
    per = ms / steps
    ideal, parts = ideal_ms(cfg_name, B, 3)
    res = {
        "workload": f"{cfg_name} training fwd+bwd, batch {B}/GPU" + (f", mixed_ratio {mixed_ratio}" if mixed_ratio else ""),
        "value": round(gb * steps / (ms * 1e-3), 2), "unit": "sample-steps/s", "ms_per_step": round(per, 3),
        "batch_steps_per_sec": round(steps / (ms * 1e-3), 3), "global_batch": gb, "steps": steps,
        "e2e": {"value": round(gb * steps / (ms_e2e * 1e-3), 2), "unit": "sample-steps/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": B * 4, "ms_per_step": round(ms_e2e / steps, 3)},
        "gpu_launches": int(launches),
        "tflops_per_gpu": round(FWD_GFLOP[cfg_name] * 3 * B / per, 1),
        "roofline": {"bound": "per level: " + ", ".join(f"{p['level']}={p['bound']}" for p in parts),
                     "ideal_ms": round(ideal, 3), "measured_ms": round(per, 3), "frac": round(ideal / per, 4),
                     "levels": parts,
                     "how": "sum over levels of max(FLOP / measured sustained tensor peak, fp16 activation bytes of a "
                            "perfectly fused pass / measured HBM GB/s) x 3 passes + fp16 weight reads, / measured step"},
        "engine_pool_bytes": vm.native().workspace_bytes()[0],
    }
    extra = {"clocks": clk}
    if headline:
        extra["roofline_gemm"] = gemm_roofline(ctx, cfg_name, B, per, resident_step)
        extra["optimizer_sweep_ms"] = sweep_ms(ctx, vm, step, resident)
    if overlap is not None:
        overlap.close()
    free_pipeline(pipe, vm, resident, host)
    return res, extra


def gemm_roofline(ctx, cfg_name, B, step_ms, resident_step):
    """Dominant kernel of the headline: every launch of the tcgen05 GEMM/conv engine is bracketed with CUDA events on
    the launching stream (mdm_profile_gemm) for two extra steps."""
    import ctypes as C

    from mdm_b200 import _lib

    lib = _lib.lib()
    if ctx.rank == 0:
        lib.mdm_profile_gemm(1)
    for _ in range(2):  # every rank runs these steps (they contain the gradient all-reduce)
        resident_step()
    ctx.barrier()
    if ctx.rank != 0:
        return None
    tot, cnt = C.c_double(), C.c_longlong()
    lib.mdm_profile_read(C.byref(tot), C.byref(cnt))
    lib.mdm_profile_gemm(0)
    gemm_ms = tot.value / 2
    peak_tf, _, how = measured_peaks()
    flops = (FWD_GFLOP[cfg_name] - ATTN_FWD_GFLOP) * 3 * B * 1e9
    ach = flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    traffic, note = None, "no ncu capture of this build committed"
    tp = os.path.join(ROOT, "profiles", "traffic_top_kernel.json")
    if os.path.exists(tp):  # written by tests/ncu_hotspots.py from an `ncu --set full` capture; never a literal here
        tj = json.load(open(tp))
        traffic, note = tj.get("dram_bytes_per_launch"), tj.get("note")
    return {"bound": "tensor",
            "kernel": "gemm_tc_persistent_kernel / gemm_tc_kernel (tcgen05 implicit-GEMM 3x3 conv + linear layers; "
                      "the fused attention kernels are timed separately and excluded from these FLOPs)",
            "achieved": round(ach, 1), "peak": peak_tf, "unit": "TFLOP/s", "frac": round(ach / peak_tf, 4),
            "traffic": traffic, "traffic_note": note, "peak_source": how, "launches_per_step": int(cnt.value // 2),
            "kernel_ms_per_step": round(gemm_ms, 3), "share_of_step": round(gemm_ms / step_ms, 3),
            "algorithmic_flops_per_step": flops}


def sweep_ms(ctx, vm, step, resident):
    """The far side of the step (SURVEY 8f rank 1), reported beside the metric, not inside it: the fused clip + Adam +
    EMA + zero-grad sweep alone, and a full training iteration (fwd + bwd + all-reduce + sweep + the fp16 weight repack
    the next forward then does)."""
    from mdm_b200 import optim

    opt = optim.FusedAdam(vm, lr=1e-6)
    step(resident)
    opt.step(max_grad_norm=2.0)  # builds the chunk table (host work, once)
    opt.zero_grad()
    step(resident)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    opt.step(max_grad_norm=2.0)
    e1.record()
    torch.cuda.synchronize()
    opt.zero_grad()
    sweep = e0.elapsed_time(e1)

    def iteration():
        step(resident)
        opt.step(max_grad_norm=2.0)
        opt.zero_grad()

    iteration()
    ms = ctx.max_over_ranks([timed(ctx, iteration, 3)])[0] / 3
    del opt
    return {"sweep": round(sweep, 3), "full_iteration": round(ms, 3)}


def measure_sampling(ctx, cfg_name, B, n_steps, runs):
    """DDIM sampling throughput (BASELINE configs[4]): Diffusion.sample(num_inference_steps=n_steps, ddim_eta=0,
    resample_steps=True, guidance_scale=1) -> n_steps network evaluations of batch B per GPU, no collective."""
    from mdm_b200 import _lib

    pipe, nested = build_pipeline(cfg_name, ctx.dev)
    pipe.eval()
    R = RES[cfg_name][0]
    host = synthetic_host_batch(cfg_name, B, 4321 + ctx.rank)
    resident = {k: host[k].to(ctx.dev) for k in ("lm_outputs", "lm_mask")}
    kw = dict(num_inference_steps=n_steps, ddim_eta=0.0, resample_steps=True, guidance_scale=1.0)

    def run_resident():
        return pipe.sample(B, resident, R, ctx.dev, **kw)

    run_resident()  # warm-up: sizes the pool, builds sampler tables (and CUDA graphs where enabled)
    run_resident()
    l0 = _lib.launch_count()
    ms = timed(ctx, run_resident, runs)
    launches = _lib.launch_count() - l0
    img_host = torch.empty(B, 3, R, R).pin_memory()

    def run_e2e():
        s = {k: host[k].to(ctx.dev, non_blocking=True) for k in ("lm_outputs", "lm_mask")}
        img = pipe.sample(B, s, R, ctx.dev, **kw)
        img_host.copy_(img, non_blocking=True)

    ms_e2e = timed(ctx, run_e2e, runs)  # (run_resident above already sized every buffer this path uses)
    ms, ms_e2e = ctx.max_over_ranks([ms, ms_e2e])
    evals = n_steps * runs
    per = ms / evals
    ideal, parts = ideal_ms(cfg_name, B, 1)
    h2d = sum(host[k].numel() * 4 for k in ("lm_outputs", "lm_mask")) + B * 3 * R * R * 4  # + the CPU-drawn start noise
    res = {
        "workload": f"{cfg_name} DDIM {n_steps}-step sampling, batch {B}/GPU, guidance 1.0",
        "value": round(B * ctx.world * evals / (ms * 1e-3), 2), "unit": "sample-steps/s",
        "ms_per_step": round(per, 3), "denoise_steps_per_sec": round(evals / (ms * 1e-3), 2),
        "images_per_sec": round(B * ctx.world * runs / (ms * 1e-3), 3), "steps": evals,
        "e2e": {"value": round(B * ctx.world * evals / (ms_e2e * 1e-3), 2), "unit": "sample-steps/s",
                "h2d_bytes_per_step": h2d // n_steps, "d2h_bytes_per_step": B * 3 * R * R * 4 // n_steps,
                "ms_per_step": round(ms_e2e / evals, 3),
                "note": "per sampling run: T5 features + start noise up once, final images down once"},
        "gpu_launches": int(launches),
        "tflops_per_gpu": round(FWD_GFLOP[cfg_name] * B / per, 1),
        "roofline": {"bound": "per level: " + ", ".join(f"{p['level']}={p['bound']}" for p in parts),
                     "ideal_ms": round(ideal, 3), "measured_ms": round(per, 3), "frac": round(ideal / per, 4), "levels": parts},
    }
    free_pipeline(pipe, resident, host)
    return res


def run_ours(args):
    ctx = Ctx()
    world = ctx.world
    peak_tf, peak_bw, how = measured_peaks()
    only = args.only
    configs = {}
    if args.config != "cc12m_64x64" or args.batch:  # development: one named training config as the headline
        head, extra = measure_train(ctx, args.config, args.batch or {"cc12m_64x64": 64, "cc12m_256x256": 32,
                                                                       "cc12m_1024x1024": max(1, 8 // world)}[args.config],
                                    args.steps, args.warmup, headline=True, mixed_ratio=args.mixed_ratio,
                                    dump_dir=args.dump_outputs)
        only = "headline"
    else:
        head, extra = measure_train(ctx, "cc12m_64x64", 64, args.steps, args.warmup, headline=True,
                                    dump_dir=args.dump_outputs)
    if only in (None, "cc12m_256x256_train"):
        configs["cc12m_256x256_train"], _ = measure_train(ctx, "cc12m_256x256", 32, max(3, args.steps // 4), 3)
        configs["cc12m_256x256_train"]["baseline_config"] = "BASELINE.json configs[2] (batch 32 per GPU, weak scaling)"
    if only in (None, "cc12m_256x256_train_mixed"):
        configs["cc12m_256x256_train_mixed"], _ = measure_train(ctx, "cc12m_256x256", 32, max(3, args.steps // 4), 3,
                                                                mixed_ratio="2:1")
        configs["cc12m_256x256_train_mixed"]["baseline_config"] = ("configs[2] with the shipped YAML's mixed_ratio '2:1': "
                                                                   "21 of 32 samples run the 256-px level")
    if only in (None, "cc12m_1024x1024_train"):
        b = max(1, 8 // world)
        configs["cc12m_1024x1024_train"], _ = measure_train(ctx, "cc12m_1024x1024", b, max(3, args.steps // 4), 3)
        configs["cc12m_1024x1024_train"]["baseline_config"] = ("BASELINE.json configs[3]: global batch 8 over the N GPUs "
                                                               f"({b}/GPU here; strong scaling, 1/GPU at N=8)")
        configs["cc12m_1024x1024_train"]["scaling"] = "strong"
    if only in (None, "cc12m_256x256_ddim50"):
        configs["cc12m_256x256_ddim50"] = measure_sampling(ctx, "cc12m_256x256", 16, 50, 2)
        configs["cc12m_256x256_ddim50"]["baseline_config"] = "BASELINE.json configs[4] (batch 16 per GPU)"
    if ctx.rank != 0:
        ctx.close()
        return
    cfg_name = head["workload"].split()[0]
    out = {
        "metric": f"denoising steps/sec (fwd+bwd), {cfg_name} U-Net, per-sample steps summed over all GPUs",
        "value": head["value"], "unit": "sample-steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": head["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16 operands, f32 accumulate/residual stream (tcgen05 kind::f16)",
        "data": "synthetic (uniform images, random T5 embeddings S=128, random-init weights incl. the reference's zero-init layers)",
        "config": {"workload": head["workload"] + (" (BASELINE.json configs[1])" if cfg_name == "cc12m_64x64" else ""),
                   "global_batch": head["global_batch"], "tokens": TOKENS, "batch_steps_per_sec": head["batch_steps_per_sec"],
                   "parallelism": f"dp{world}", "l2": "per-step working set (activation stash, GBs) far exceeds the 126 MB L2",
                   "tflops_per_gpu": head["tflops_per_gpu"],
                   "timed_region": "get_loss + backward (+ all-reduce); optimizer sweep and weight repack outside (optimizer_sweep_ms)"},
        "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": extra.get("clocks"),
        "roofline": extra.get("roofline_gemm"), "roofline_step": head["roofline"],
        "optimizer_sweep_ms": extra.get("optimizer_sweep_ms"),
        "engine_pool_bytes": head["engine_pool_bytes"], "peaks": {"tensor_tflops": peak_tf, "hbm_gbs": peak_bw, "source": how},
        "configs": configs,
    }
    if not args.no_cpu_baseline and world == 1:
        out["gpu_eager_baseline"] = gpu_eager_arm("cc12m_64x64", 64 if cfg_name == "cc12m_64x64" else head["global_batch"])
        out["cpu_baseline"] = cpu_arm("cc12m_64x64", steps=5, warmup=1, batch=2)
    print(json.dumps(out), flush=True)
    ctx.close()


def _oracle_setup(cfg_name, device, dtype=torch.float32):
    import types

    import yaml

    from oracle import diffusion_ref as dref
    from oracle import unet_ref
    from mdm_b200 import config as mc
    from mdm_b200.models import NestedUNet, UNet

    y = yaml.safe_load(open(os.path.join(ROOT, "ml-mdm_b200", "mdm_b200", "configs", cfg_name + ".yaml")))

    def ns(d):
        return types.SimpleNamespace(**{k: ns(v) for k, v in d.items()}) if isinstance(d, dict) else d

    ucfg = ns(y["unet_config"])
    c = ucfg
    while c is not None:
        if hasattr(c, "initialize_inner_with_pretrained"):
            c.initialize_inner_with_pretrained = None
        c = getattr(c, "inner_config", None)
    net = unet_ref.OracleNet(ucfg, 2048)
    cfg2, _, nested = mc.load_yaml_configs(os.path.join(ROOT, "ml-mdm_b200", "mdm_b200", "configs", cfg_name + ".yaml"))
    torch.manual_seed(4321)
    shapes = (NestedUNet if nested else UNet)(3, 3, cfg2)  # parameter container only (shapes + init)
    P = {}
    for k, p in shapes.named_parameters():
        v = p.detach().clone()
        if float(v.abs().max()) == 0:
            v.normal_(0, 0.02)
        P[k] = v.to(device, dtype).requires_grad_(True)
    del shapes
    scales = net.nest_ratio + [1] if nested else [1]
    sc = y["diffusion_config"]["sampler_config"]
    gam = dref.gammas_f32(sc.get("schedule_type", "DDPM"), sc.get("num_diffusion_steps", 1000)).to(device)
    return net, P, scales, sc, gam, nested, dref


def _oracle_step_fn(cfg_name, batch, device):
    net, P, scales, sc, gam, nested, dref = _oracle_setup(cfg_name, device)
    R = RES[cfg_name][0]
    g = torch.Generator().manual_seed(1234)
    images = (torch.rand(batch, 3, R, R, generator=g) * 2 - 1).to(device)
    lm = torch.randn(batch, TOKENS, 2048, generator=g).to(device)
    mask = torch.ones(batch, TOKENS, device=device)

    def one():
        time_ = torch.randint(0, 1000, (batch,), generator=g).to(device)
        eps = [torch.randn(batch, 3, R // (scales[0] // s), R // (scales[0] // s), generator=g).to(device) for s in scales]
        loss, _, _ = dref.training_loss(net, P, images, eps, time_, lm, mask, gam, scales, dref.V_PREDICTION, dref.DDPM,
                                        shifted=bool(sc.get("schedule_shifted", False)),
                                        power=sc.get("schedule_shifted_power", 1))
        loss.mean().backward()
        for p in P.values():
            p.grad = None

    return one


def cpu_arm(cfg_name, steps, warmup, batch=2):
    """The reference's CPU path for this workload, timed on this host's cores: the oracle port
    (oracle/unet_ref.py + oracle/diffusion_ref.py; the Python reference itself cannot travel to the GPU box).
    One step = get_loss + backward on a bounded sample of `batch` images; full warm-up steps first, then the MEDIAN
    of `steps` individually timed steps."""
    # oneDNN/MKL stop scaling (and then collapse) beyond ~32 threads on these shapes; measured on the
    # 128-thread GPU host: conv 256->256@64x64 4.0 ms at 32 threads, 18 ms at 64.
    cores = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(cores)
    one = _oracle_step_fn(cfg_name, batch, "cpu")
    for _ in range(max(1, warmup)):
        one()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        one()
        ts.append(time.perf_counter() - t0)
    ts.sort()
    med = ts[len(ts) // 2]
    return {"value": round(batch / med, 4), "unit": "sample-steps/s", "cores": cores, "kind": "port",
            "sample": f"median of {steps} steps of get_loss+backward at batch {batch} after {max(1, warmup)} full warm-up "
                      f"step(s) (fp32, torch CPU oneDNN/MKL ops, {cores} threads)",
            "seconds": round(sum(ts), 2), "step_seconds": [round(t, 3) for t in ts]}


def gpu_eager_arm(cfg_name, batch, steps=3):
    """Same-box PyTorch-eager GPU baseline (SURVEY 8d-ii): the oracle port -- plain functional torch, the reference's
    op sequence -- on the B200 through cuDNN/cuBLAS with TF32 enabled as clis/train_parallel.py:18-19 does. A baseline
    leg only: nothing of it is on the product path."""
    dev = torch.device("cuda", torch.cuda.current_device())
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    try:
        one = _oracle_step_fn(cfg_name, batch, dev)
        one()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            one()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out = {"value": round(batch / (ms * 1e-3), 2), "unit": "sample-steps/s", "ms_per_step": round(ms, 2),
               "impl": "oracle port (functional torch eager, cuDNN/cuBLAS, allow_tf32=True), same box, same workload",
               "workload": f"{cfg_name} training fwd+bwd, batch {batch}", "steps": steps}
    except Exception as e:  # out of memory on a busy box: report, do not fail the bench
        out = {"unavailable": f"{type(e).__name__}: {str(e)[:120]}"}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
    gc.collect()
    torch.cuda.empty_cache()
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg_name = args.config
    steps = max(3, min(args.steps, 5))
    base = cpu_arm(cfg_name, steps=steps, warmup=max(1, min(args.warmup, 1)), batch=2)
    out = {
        "impl": "reference",
        "metric": f"denoising steps/sec (fwd+bwd), {cfg_name} U-Net, per-sample steps summed over all GPUs",
        "value": base["value"], "unit": "sample-steps/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": 1, "ms_per_step": round(1000.0 * 2 / base["value"], 1), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (same generator as the GPU arm)",
        "config": {"workload": f"{cfg_name} training fwd+bwd (BASELINE.json configs[1]), bounded sample of batch 2 per step"},
        "cpu_baseline": base,
        "e2e": {"value": base["value"], "unit": "sample-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cc12m_64x64", choices=sorted(FWD_GFLOP))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: BASELINE config)")
    ap.add_argument("--mixed-ratio", default=None, help="NestedDiffusionConfig.mixed_ratio for --config runs, e.g. 2:1")
    ap.add_argument("--only", default=None, help="headline | one key of the configs object (development aid)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write the headline's last timed step's outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a B200: the mdm_b200 path has no CPU fallback (use --impl reference for the CPU arm)")
        run_ours(args)


if __name__ == "__main__":
    main()
