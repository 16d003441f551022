"""Small configurations of the reference's own config schema, used for parity tests and golden
fixtures (the shipped cc12m_* configs are exercised at full size on the GPU and in bench.py)."""
import copy

import numpy as np
import torch

LM_DIM = 48

_RESNET = dict(num_channels=-1, output_channels=-1, num_groups_norm=32, dropout=0.0,
               use_attention_ffn=True)

TINY_UNET = dict(
    num_resnets_per_resolution=[1, 2],
    attention_levels=[1],
    num_attention_layers=[0, 2],
    conditioning_feature_dim=-1,
    conditioning_feature_proj_dim=64,
    num_lm_head_layers=0,
    masked_cross_attention=0,
    resolution_channels=[32, 64],
    skip_mid_blocks=False,
    skip_cond_emb=False,
    nesting=False,
    micro_conditioning="scale:16",
    temporal_mode=False,
    temporal_spatial_ds=False,
    temporal_positional_encoding=False,
    resnet_config=dict(_RESNET),
)

TINY_DIFFUSION = dict(
    sampler_config=dict(num_diffusion_steps=1000, reproject_signal=False, schedule_type="DEEPFLOYD",
                        prediction_type="V_PREDICTION", loss_target_type="DDPM", beta_start=0.0001,
                        beta_end=0.02, threshold_function="CLIP", rescale_schedule=1.0,
                        schedule_shifted=False),
    model_output_scale=0.0,
    use_vdm_loss_weights=False,
)

# outer level (no attention, no mid blocks) wrapped around TINY_UNET as the inner net
_inner = copy.deepcopy(TINY_UNET)
_inner["nesting"] = True
TINY_NESTED = dict(
    attention_levels=[],
    conditioning_feature_dim=-1,
    conditioning_feature_proj_dim=-1,
    freeze_inner_unet=False,
    initialize_inner_with_pretrained="None",
    inner_config=_inner,
    interp_conditioning=False,
    masked_cross_attention=1,
    micro_conditioning="scale:64",
    nesting=False,
    num_attention_layers=[0, 0, 0],
    num_lm_head_layers=0,
    num_resnets_per_resolution=[2, 1, 1],
    resnet_config=dict(_RESNET, use_attention_ffn=False),
    resolution_channels=[32, 32, 64],
    skip_cond_emb=True,
    skip_inner_unet_input=False,
    skip_mid_blocks=True,
    skip_normalization=True,
    temporal_dim=128,
    temporal_mode=False,
    temporal_positional_encoding=False,
    temporal_spatial_ds=False,
)
# inner net must start at the outer net's last width for in/out adapters (any widths are legal)
TINY_NESTED["inner_config"]["temporal_dim"] = None

TINY_NESTED_DIFFUSION = dict(
    sampler_config=dict(num_diffusion_steps=1000, reproject_signal=False,
                        prediction_type="V_PREDICTION", loss_target_type="DDPM",
                        schedule_type="DEEPFLOYD", rescale_signal=1, schedule_shifted=True),
    model_output_scale=0,
    use_vdm_loss_weights=False,
    use_double_loss=True,
    no_use_residual=True,
)


def seeded_state_dict(ref_state_dict, seed, std=0.05):
    """Deterministic, platform-stable parameters for a model with the given keys/shapes.

    Every tensor (including the reference's zero-initialised ones, SURVEY.md fact 4) is redrawn from
    numpy's PCG64 in sorted-key order: norm weights ~ 1 + N(0, 0.1), biases ~ N(0, 0.05),
    matrices/filters ~ N(0, 1/sqrt(fan_in)) so activations stay O(1).
    """
    rng = np.random.default_rng(seed)
    out = {}
    for k in sorted(ref_state_dict.keys()):
        shape = tuple(ref_state_dict[k].shape)
        if k.endswith(".weight") and len(shape) == 1:
            v = 1.0 + 0.1 * rng.standard_normal(shape)
        elif len(shape) == 1:
            v = std * rng.standard_normal(shape)
        else:
            fan_in = int(np.prod(shape[1:]))
            v = rng.standard_normal(shape) / np.sqrt(fan_in)
        out[k] = torch.from_numpy(v.astype(np.float32))
    return out


def golden_sample(t, n, seed=0):
    """`n` elements of a flattened tensor at fixed, seeded positions (all of it when it has no more than `n`):
    outputs too large to commit whole are stored and compared at these positions."""
    flat = torch.as_tensor(t).detach().reshape(-1)
    if flat.numel() <= n:
        return flat.clone()
    idx = np.sort(np.random.default_rng(seed).choice(flat.numel(), n, replace=False))
    return flat[torch.from_numpy(idx)]


def seeded_inputs(seed, batch, res, tokens, lm_dim=LM_DIM, nlevels=1, ratio=4):
    rng = np.random.default_rng(seed)
    xs = []
    r = res
    for _ in range(nlevels):
        xs.append(torch.from_numpy(rng.standard_normal((batch, 3, r, r)).astype(np.float32)))
        r //= ratio
    times = torch.from_numpy(rng.integers(0, 1000, size=(batch,)).astype(np.int64))
    lm = torch.from_numpy(rng.standard_normal((batch, tokens, lm_dim)).astype(np.float32))
    lens = rng.integers(1, tokens + 1, size=(batch,))
    mask = torch.zeros(batch, tokens)
    for i, n in enumerate(lens):
        mask[i, :n] = 1
    lm = lm * mask.unsqueeze(-1)  # language_models/factory.py:101 zeroes padded tokens
    return (xs if nlevels > 1 else xs[0]), times, lm, mask
