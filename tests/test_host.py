"""CPU-side checks of the product: schedule/index math bit-exact against the reference's golden
tables, parameter trees identical to the reference's state_dict, the C ABI exports everything
include/mdm_b200.h declares, configs load, and compute fails loudly without a GPU."""
import copy
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import tiny_configs as tc
from mdm_b200 import _lib
from mdm_b200 import config as mc
from mdm_b200 import samplers
from mdm_b200.models import NestedUNet, UNet

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
CFG = os.path.join(ROOT, "ml-mdm_b200", "mdm_b200", "configs")


def test_schedule_tables_bit_exact_vs_reference():
    g = np.load(os.path.join(GOLD, "schedules.npz"))
    for st in ["DEEPFLOYD", "DDPM", "COSINE"]:
        s = samplers.Sampler(mc.SamplerConfig(num_diffusion_steps=1000, schedule_type=st))
        assert np.array_equal(s.gammas.numpy().view(np.uint32), g[f"gammas_{st}"].view(np.uint32))
        assert np.array_equal(s.vdm_loss_weights.numpy().view(np.uint32), g[f"vdm_{st}"].view(np.uint32))
    for p, scales in [(1, [4, 1]), (2, [16, 4, 1])]:
        s = samplers.NestedSampler(mc.SamplerConfig(num_diffusion_steps=1000, schedule_type="DEEPFLOYD",
                                                    schedule_shifted=True, schedule_shifted_power=p))
        for sc in scales:
            tab = s.level_table(sc, "cpu")
            assert np.array_equal(tab.numpy().view(np.uint32), g[f"shift_p{p}_s{sc}"].view(np.uint32))
    s = samplers.Sampler(mc.SamplerConfig(num_diffusion_steps=1000, schedule_type="DEEPFLOYD"))
    for n in [1, 2, 5, 50, 100, 250, 999, 1000]:
        ts = s.set_timesteps(n)
        assert ts.dtype == np.int64 and np.array_equal(ts, g[f"timesteps_{n}"])


@pytest.mark.parametrize("name", ["cc12m_64x64", "cc12m_256x256", "cc12m_1024x1024"])
def test_parameter_tree_identical_to_reference(name):
    ucfg, dcfg, nested = mc.load_yaml_configs(os.path.join(CFG, name + ".yaml"))
    with torch.device("meta"):
        m = (NestedUNet if nested else UNet)(3, 3, ucfg)
    want = [l.split() for l in open(os.path.join(GOLD, f"keys_{name}.txt")).read().strip().split("\n")]
    got = [[k, "x".join(str(d) for d in v.shape)] for k, v in m.state_dict().items()]
    assert got == want  # same keys, same order, same shapes (OIHW fp32)


def test_tiny_tree_and_zero_init_layers():
    cfg = mc.unet_config_from_dict(copy.deepcopy(tc.TINY_UNET))
    cfg.conditioning_feature_dim = tc.LM_DIM
    m = UNet(3, 3, cfg)
    names = open(os.path.join(GOLD, "tiny_unet_params.txt")).read().split()
    assert [k for k, _ in m.named_parameters()] == names
    zero = [k for k, p in m.named_parameters() if float(p.abs().max()) == 0]
    assert any(k.endswith("conv_out.weight") for k in zero) and any(k.endswith("conv2.weight") for k in zero)
    assert any(k.endswith("proj_out.weight") for k in zero) and any("ffn.3" in k for k in zero)


def test_c_abi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "mdm_b200.h")).read()
    declared = set(re.findall(r"\b(mdm_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    lib = ctypes.CDLL(_lib.LIB_PATH)
    missing = [s for s in sorted(declared) if not hasattr(lib, s)]
    assert not missing, missing
    assert lib.mdm_version() >= 100


def test_ctypes_mirrors_match_the_compiled_struct_layouts():
    """Every ctypes.Structure that mirrors a struct of include/mdm_b200.h has the size the library was compiled with
    (a field added on one side only would otherwise shift every later field silently)."""
    from mdm_b200 import optim
    from mdm_b200.models import native

    lib = ctypes.CDLL(_lib.LIB_PATH)
    lib.mdm_abi_sizeof.restype = ctypes.c_longlong
    mirrors = [_lib.TmapSpec, _lib.GemmParams, native.LevelCfg, native.NetCfg, native.NetIO, native.NetGradIO,
               optim.OptChunk, optim.AdamCfg]
    for which, cls in enumerate(mirrors):
        assert lib.mdm_abi_sizeof(which) == ctypes.sizeof(cls), (which, cls.__name__)
    assert lib.mdm_abi_sizeof(len(mirrors)) == -1
    # and the field NAMES of the two largest ones, in order, against the header text
    hdr = open(os.path.join(ROOT, "include", "mdm_b200.h")).read()
    for cname, cls in (("mdm_gemm_params", _lib.GemmParams), ("mdm_net_io", native.NetIO)):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (cname, cname), hdr, re.S).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        names = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            for part in decl.split(","):
                names.append(re.sub(r"\[.*\]", "", part.strip().split()[-1].lstrip("*")))
        assert names == [f[0] for f in cls._fields_], (cname, names, [f[0] for f in cls._fields_])


def test_compute_fails_loudly_without_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    cfg = mc.unet_config_from_dict(copy.deepcopy(tc.TINY_UNET))
    cfg.conditioning_feature_dim = tc.LM_DIM
    m = UNet(3, 3, cfg)
    x, t, lm, mask = tc.seeded_inputs(3, 2, 16, 6)
    with pytest.raises(_lib.MdmError):
        m(x, t, lm, mask, {})


def test_plugin_overwrites_reference_registries():
    import types

    from mdm_b200 import plugin
    from mdm_b200.diffusion import Diffusion, NestedDiffusion

    fake = types.SimpleNamespace(
        MODEL_REGISTRY={"unet": object, "nested_unet": object}, PIPELINE_REGISTRY={"unet": object, "nested_unet": object},
        MODEL_CONFIG_REGISTRY={"unet": {"model": "unet", "config": int}, "nested2_unet": {"model": "nested_unet", "config": int}},
        PIPELINE_CONFIG_REGISTRY={"unet": int, "nested_unet": int})
    plugin.register(fake)
    assert fake.MODEL_REGISTRY["unet"] is UNet and fake.MODEL_REGISTRY["nested_unet"] is NestedUNet
    assert fake.PIPELINE_REGISTRY["unet"] is Diffusion and fake.PIPELINE_REGISTRY["nested_unet"] is NestedDiffusion
    plugin.register(fake, parallel_names=True)
    assert fake.MODEL_CONFIG_REGISTRY["nested2_unet_b200"]["model"] == "nested_unet_b200"


def reference_config_module():
    """A stand-in for the reference's ml_mdm.config, rebuilt from tests/golden/reference_configs.json: its model and
    pipeline registries, get_model/get_pipeline (config.py:54-63), its config dataclasses and sampler enums (foreign
    classes, not ours), and its config objects for cc12m_256x256 as the reference's own loader builds them from the
    YAML (including its __post_init__ conversions)."""
    import dataclasses
    import enum
    import json
    import types
    import typing

    d = json.load(open(os.path.join(GOLD, "reference_configs.json")))
    enums = {n: enum.Enum(n, members) for n, members in d["enums"].items()}
    classes = {n: dataclasses.make_dataclass(n, [(f, typing.Any) for f in fields]) for n, fields in d["classes"].items()}

    def dec(v):
        if isinstance(v, dict) and "enum" in v:
            return enums[v["enum"]][v["member"]]
        if isinstance(v, dict) and "dataclass" in v:
            return classes[v["dataclass"]](**{k: dec(x) for k, x in v["fields"].items()})
        if isinstance(v, list):
            return [dec(x) for x in v]
        return v

    m = types.SimpleNamespace(
        MODEL_REGISTRY={k: object for k in d["MODEL_REGISTRY"]}, PIPELINE_REGISTRY={k: object for k in d["PIPELINE_REGISTRY"]},
        MODEL_CONFIG_REGISTRY={k: {"model": v["model"], "config": classes[v["config"]]}
                               for k, v in d["MODEL_CONFIG_REGISTRY"].items()},
        PIPELINE_CONFIG_REGISTRY={k: classes[v] for k, v in d["PIPELINE_CONFIG_REGISTRY"].items()})
    m.get_model = lambda name: m.MODEL_REGISTRY[m.MODEL_CONFIG_REGISTRY[name]["model"]]
    m.get_pipeline = lambda name: m.PIPELINE_REGISTRY[m.MODEL_CONFIG_REGISTRY[name]["model"]]
    return m, {k: dec(v) for k, v in d["cc12m_256x256"].items()}, classes, enums


def test_plugin_on_live_reference_registry():
    """Registration into the reference's registries, and the reference's own config objects (its dataclasses, its
    ScheduleType/PredictionType/ThresholdType members) driving our NestedUNet and NestedDiffusion unchanged."""
    from mdm_b200 import plugin
    from mdm_b200.diffusion import NestedDiffusion

    ref, cfgs, classes, enums = reference_config_module()
    plugin.register(ref)
    assert ref.get_model("nested2_unet") is NestedUNet
    assert ref.get_model("unet") is UNet
    assert ref.get_pipeline("nested_unet") is NestedDiffusion
    ucfg = cfgs["unet_config"]
    assert type(ucfg) is ref.MODEL_CONFIG_REGISTRY["nested_unet"]["config"] is classes["NestedUNetConfig"]
    ucfg.conditioning_feature_dim = 2048
    ucfg.initialize_inner_with_pretrained = None
    with torch.device("meta"):
        m = ref.get_model("nested_unet")(3, 3, ucfg)
    assert m.nest_ratio == [4] and len(m.state_dict()) == 889
    dcfg = cfgs["diffusion_config"]
    assert type(dcfg) is ref.PIPELINE_CONFIG_REGISTRY["nested_unet"]
    assert type(dcfg.sampler_config.schedule_type) is enums["ScheduleType"]  # a foreign enum member
    pipe = ref.get_pipeline("nested_unet")(m, dcfg)
    assert pipe.sampler.gammas.shape == (1001,)
    tab = pipe.sampler.gammas
    want = samplers.Sampler(mc.SamplerConfig(num_diffusion_steps=1000, schedule_type="DEEPFLOYD")).gammas
    assert torch.equal(tab, want)  # DEEPFLOYD, taken from the foreign enum member by name
