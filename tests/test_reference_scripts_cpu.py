"""Drop-in check against the reference's OWN script code, recorded in tests/golden/reference_scripts.json by running
`measure_throughput/__main__.py` and `main_sampling_fid.py` unmodified with this repo's package (+ the omegaconf/easydict
fallbacks) on the path (oracle/gen_golden.py).  These tests import every name the scripts (and compute_metrics.py, which
main_sampling_fid imports) take from those packages, and replay the scripts' calls: `python -m measure_throughput f=32 d=4
c=... model=...` up to device placement, and main_sampling_fid's checkpoint loading.  The measure_throughput configs and
Experiment fields come from the reference's code; main_sampling_fid's `config_yaml` / `loaded` records are a snapshot of this
package's own load_config / augment_arch_defaults output as that script's load_model() returned it."""
import dataclasses
import importlib.util
import json
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COMPAT = os.path.join(ROOT, "rq-vae-transformer_b200", "compat")


@pytest.fixture(scope="module")
def scripts():
    with open(os.path.join(ROOT, "tests", "golden", "reference_scripts.json")) as f:
        return json.load(f)


@pytest.fixture
def omegaconf_on_path():
    have_real = importlib.util.find_spec("omegaconf") is not None
    if not have_real:
        sys.path.append(COMPAT)
    try:
        yield
    finally:
        if not have_real and COMPAT in sys.path:
            sys.path.remove(COMPAT)
            for k in ("omegaconf", "easydict"):
                sys.modules.pop(k, None)


def _import_surface(entries):
    """every module / name a reference script imports from this repository's packages resolves"""
    for module, name in entries:
        mod = importlib.import_module(module)
        if name is not None:
            assert hasattr(mod, name), "%s.%s" % (module, name)


def test_measure_throughput_module_builds_models_through_our_package(scripts, omegaconf_on_path):
    from omegaconf import OmegaConf
    from rqvae.models import create_model
    from rqvae.utils.config import Config, augment_arch_defaults
    import rqvae
    assert "rq-vae-transformer_b200" in rqvae.__file__
    _import_surface(scripts["imports"]["measure_throughput"])
    rec = scripts["measure_throughput"]
    types = {"int": int, "str": str}
    Experiment = dataclasses.make_dataclass("Experiment", [(n, types[t], dataclasses.field(default=d))
                                                           for n, t, d in rec["experiment_fields"]])
    args = OmegaConf.merge(OmegaConf.structured(Experiment()),
                           OmegaConf.from_cli(["f=32", "d=4", "c=2048", "model=small", "batch_size=7"]))
    assert args.batch_size == 7 and args.model == "small" and args.n_loop == 6

    def build(call):
        vae, _ = create_model(augment_arch_defaults(Config(call["rqvae"])))
        ar, _ = create_model(augment_arch_defaults(Config(call["rqtransformer"])))
        return vae, ar

    small, huge = rec["create_model"]
    assert small["args"] == ["f%d" % args.f, args.model, args.d, args.c]
    vae, ar = build(small)
    assert list(vae.code_shape) == [8, 8, 4] and ar.block_size == torch.Size([8, 8, 4]) and ar.block_size_cond == 1
    assert ar.config.embed_dim == 512 and len(ar.body_transformer.blocks) == 24 and len(ar.head_transformer.blocks) == 4
    assert vae.quantizer.codebooks[0].weight.shape == (2049, 256)
    n_ar = sum(p.numel() for p in ar.parameters()) / 1e6
    assert 80 < n_ar < 110                            # the "small" (~90M) preset, measure_throughput/__main__.py:150-170
    # the huge preset's shape bookkeeping (built on the meta device: no 5.5 GB allocation)
    assert huge["args"] == ["f32", "huge", 4, 16384]
    with torch.device("meta"):
        vae_h, ar_h = build(huge)
    assert ar_h.config.embed_dim == 1536 and len(ar_h.body_transformer.blocks) == 42 and len(ar_h.head_transformer.blocks) == 6


def test_main_sampling_fid_loads_synthetic_checkpoint(tmp_path, scripts, omegaconf_on_path):
    """checkpoint + sibling config.yaml layout (main_sampling_fid.py:146-158) loads through the calls its load_model() makes:
    load_config -> augment_arch_defaults(config.arch) -> create_model(config.arch, ema=False) -> load_state_dict"""
    import yaml
    _import_surface(scripts["imports"]["main_sampling_fid"] + scripts["imports"]["compute_metrics"])
    from tests.helpers import ar_config, vae_config
    from rqvae.models import create_model
    from rqvae.utils.config import augment_arch_defaults, load_config
    for name, cfg in (("ar", ar_config("tiny")), ("vae", vae_config("tiny"))):
        rec = scripts["main_sampling_fid"][name]
        d = tmp_path / name
        d.mkdir()
        model, _ = create_model(cfg)
        torch.save({"state_dict": model.state_dict(), "state_dict_ema": model.state_dict()}, d / "model.pt")
        written = {"arch": cfg.to_dict(), "dataset": {"type": "imagenet"},
                   "sampling": {"temp": 1.0, "top_k": [1024], "top_p": [0.95]}}
        assert written == rec["config_yaml"]
        with open(d / "config.yaml", "w") as f:
            yaml.safe_dump(written, f)
        config = load_config(str(d / "config.yaml"))
        config.arch = augment_arch_defaults(config.arch)
        loaded, _ = create_model(config.arch, ema=False)
        loaded.load_state_dict(torch.load(d / "model.pt", map_location="cpu")["state_dict_ema" if name == "ar" else "state_dict"])
        assert config.to_dict() == rec["loaded"]
        for k, v in model.state_dict().items():
            assert torch.equal(v, loaded.state_dict()[k]), k
        assert config.arch.type in ("rq-transformer", "rq-vae")
