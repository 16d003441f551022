"""Import the UNMODIFIED reference (apple/ml-mdm) on CPU so that the golden fixtures under tests/golden/ can be
generated from it. The environment variable ML_MDM_ROOT names the directory of the checkout that holds the ml_mdm/
package and configs/models/ (the ml-mdm-matryoshka tree). The tests themselves never import the reference: they
compare against those fixtures.

The reference's hot path needs five packages that carry no arithmetic and may not be installed
(torchinfo, simple_parsing, dataclass_wizard, mlx/mlx.data, boto3); they are stubbed in sys.modules
before the import (SURVEY.md section 8c).
"""
import dataclasses
import enum
import os
import sys
import types
import typing

REF_ROOT = os.environ.get("ML_MDM_ROOT", "")
CFG_DIR = os.path.join(REF_ROOT, "configs", "models")


def available():
    return os.path.isdir(os.path.join(REF_ROOT, "ml_mdm"))


def _mod(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


_loaded = None


def load():
    """Returns a namespace with the reference modules: unet, nested_unet, diffusion, samplers, config."""
    global _loaded
    if _loaded is not None:
        return _loaded
    if not available():
        raise RuntimeError("reference tree not present: set ML_MDM_ROOT to an apple/ml-mdm checkout")
    if "torchinfo" not in sys.modules:
        _mod("torchinfo", summary=lambda *a, **k: None)
    if "simple_parsing" not in sys.modules:
        class _AP:
            def __init__(self, *a, **k):
                pass

        class _AGM(enum.Enum):
            FLAT = 0
            NESTED = 1
            BOTH = 2

        sp = _mod("simple_parsing", ArgumentParser=_AP)
        w = _mod("simple_parsing.wrappers")
        fw = _mod("simple_parsing.wrappers.field_wrapper", ArgumentGenerationMode=_AGM)
        sp.wrappers = w
        w.field_wrapper = fw
    if "dataclass_wizard" not in sys.modules:
        _mod("dataclass_wizard", YAMLWizard=type("YAMLWizard", (), {}))
    if "mlx" not in sys.modules:
        mlx = _mod("mlx")
        mlx.__path__ = []
        core = _mod("mlx.data.core", CharTrie=object, Tokenizer=object)
        data = _mod("mlx.data", Buffer=object, Stream=object, core=core)
        data.__path__ = []
        mlx.data = data
        mlx.core = _mod("mlx.core", array=type("array", (), {}))
    if "boto3" not in sys.modules:
        b3 = _mod("boto3")
        b3.__path__ = []
        b3.session = _mod("boto3.session")
        _mod("boto3.s3")
        _mod("boto3.s3.transfer", TransferConfig=object)
    if REF_ROOT not in sys.path:
        sys.path.insert(0, REF_ROOT)
    from ml_mdm import config, diffusion, samplers  # noqa: E402
    from ml_mdm.models import nested_unet, unet  # noqa: E402

    _loaded = types.SimpleNamespace(unet=unet, nested_unet=nested_unet, diffusion=diffusion,
                                    samplers=samplers, config=config)
    return _loaded


def from_dict(cls, d):
    """dict (from YAML) -> the reference's config dataclass, recursively (replaces simple_parsing)."""
    ref = load()
    hints = typing.get_type_hints(cls)
    kw = {}
    for f in dataclasses.fields(cls):
        if f.name not in d:
            continue
        v, t = d[f.name], hints[f.name]
        if dataclasses.is_dataclass(t) and isinstance(v, dict):
            v = from_dict(t, v)
        elif isinstance(t, type) and issubclass(t, ref.samplers.Type) and isinstance(v, str):
            v = t.argparse(v)
        kw[f.name] = None if (isinstance(v, str) and v == "None") else v
    return cls(**kw)


def build(unet_cfg: dict, diff_cfg: dict, arch: str, lm_dim: int):
    """Construct (vision_model, pipeline) of the reference from plain dicts."""
    ref = load()
    ucfg = from_dict(ref.config.MODEL_CONFIG_REGISTRY[arch]["config"], unet_cfg)
    ucfg.conditioning_feature_dim = lm_dim  # train_parallel.py:65
    if hasattr(ucfg, "initialize_inner_with_pretrained"):
        ucfg.initialize_inner_with_pretrained = None
    pname = ref.config.MODEL_CONFIG_REGISTRY[arch]["model"]
    dcfg = from_dict(ref.config.PIPELINE_CONFIG_REGISTRY[pname], diff_cfg)
    model = ref.config.get_model(arch)(3, 3, ucfg)
    pipe = ref.config.get_pipeline(arch)(model, dcfg)
    return model, pipe


def load_yaml(name):
    import yaml

    with open(os.path.join(CFG_DIR, name)) as f:
        return yaml.safe_load(f)
