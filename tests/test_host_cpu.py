"""CPU-side host logic: state_dict layout parity with the reference, config layer, C-ABI exports, loud failure
without a GPU.  No kernels are launched here."""
import ctypes
import json
import os
import re

import pytest
import torch

from oracle.zoo import AR_ZOO, VAE_ZOO, vae_ddconfig
from oracle import synth

from rqvae import _native as N
from rqvae.models import create_model
from rqvae.models.rqtransformer import RQTransformer
from rqvae.models.rqvae import RQVAE
from rqvae.utils.config import Config, augment_arch_defaults, merge


def make_ar(name, device="cpu"):
    E, nh, nb, nhl, V, bs, vc, cl = AR_ZOO[name]
    cfg = Config(type="rq-transformer", vocab_size=V, block_size=list(bs), vocab_size_cond=vc, block_size_cond=cl,
                 embed_dim=E, input_embed_dim=256, shared_tok_emb=True, shared_cls_emb=True, input_emb_vqvae=True,
                 head_emb_vqvae=True, cumsum_depth_ctx=True,
                 body=dict(n_layer=nb, block=dict(n_head=nh)), head=dict(n_layer=nhl, block=dict(n_head=nh)))
    cfg = augment_arch_defaults(cfg)
    with torch.device(device):
        model, _ = create_model(cfg)
    return model


def make_vae(name, device="cpu"):
    kw = VAE_ZOO[name]
    cs = kw.get("code_shape", (8, 8, 4))
    cfg = Config(type="rq-vae", hparams=dict(bottleneck_type="rq", embed_dim=256, n_embed=kw["K"],
                                             latent_shape=[cs[0], cs[1], 256], code_shape=list(cs), shared_codebook=True,
                                             decay=0.99, restart_unused_codes=True, loss_type="mse", latent_loss_weight=0.25),
                 ddconfig=vae_ddconfig(**kw))
    cfg = augment_arch_defaults(cfg)
    with torch.device(device):
        model, _ = create_model(cfg)
    return model


@pytest.mark.parametrize("name", list(AR_ZOO))
def test_ar_state_dict_layout_matches_reference(layouts, name):
    m = make_ar(name, "meta")
    mine = {k: list(v.shape) for k, v in m.state_dict().items()}
    assert mine == layouts["ar/" + name]


@pytest.mark.parametrize("name", list(VAE_ZOO))
def test_vae_state_dict_layout_matches_reference(layouts, name):
    m = make_vae(name, "meta")
    mine = {k: list(v.shape) for k, v in m.state_dict().items()}
    assert mine == layouts["vae/" + name]


def test_seeded_default_init_equals_reference():
    """same constructor order => same RNG consumption => torch.manual_seed(0) yields the reference's weights, pinned by the
    per-tensor digests of the reference's own seeded models (tests/golden/seeded_init.json, oracle/gen_golden.py)"""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "seeded_init.json")) as f:
        ref = json.load(f)
    for name, make in (("ar/tiny", make_ar), ("vae/tiny", make_vae)):
        torch.manual_seed(0)
        mine = synth.tensor_digests(make("tiny").state_dict())
        assert mine.keys() == ref[name].keys(), name
        for k, v in ref[name].items():
            assert mine[k] == v, (name, k)


def test_shared_codebook_aliases_one_tensor():
    m = make_vae("tiny")
    cbs = m.quantizer.codebooks
    assert all(cb is cbs[0] for cb in cbs)
    assert m.code_shape == [4, 4, 4] and float(cbs[0].weight[-1].abs().sum()) == 0.0


def test_config_layer():
    c = Config(a=1, b=dict(c=2, d=[1, 2]))
    c2 = c.copy()
    c2.b.c = 5
    c2.b.e = dict(f=1)
    assert c.b.c == 2 and c2.b.c == 5 and c2["b"]["e"].f == 1
    m = merge(c, dict(b=dict(c=7), z=3))
    assert m.b.c == 7 and m.b.d == [1, 2] and m.z == 3 and c.b.c == 2
    assert dict(**c2)["a"] == 1
    ar = make_ar("tiny", "meta")
    assert ar.config.body.block.embed_dim == 128 and ar.config.body.block.resid_pdrop == 0.1
    assert ar.block_size == torch.Size([4, 4, 4]) and ar.block_size_cond == 1 and ar.vocab_size == [512] * 4
    assert ar.get_block_size() == ar.block_size


def test_sample_topk_topp_list_handling():
    ar = make_ar("tiny", "meta")
    assert ar._lists(None, None) == ([512] * 4, [1.0] * 4)
    assert ar._lists(1000, 0.9) == ([512] * 4, [0.9] * 4)
    assert ar._lists([7], [2.0]) == ([7] * 4, [1.0] * 4)
    assert ar._lists([1, 2, 3, 4], [0.1, 0.2, 0.3, 0.4]) == ([1, 2, 3, 4], [0.1, 0.2, 0.3, 0.4])


def test_c_abi_library_exports_every_declared_symbol():
    """every function declared in include/rqb200.h is exported by csrc/librqb200.so"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "rqb200.h")).read()
    declared = set(re.findall(r"\b(rqb200_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    lib = ctypes.CDLL(N.LIB_PATH)
    for sym in declared:
        assert hasattr(lib, sym), sym
    assert set(N.EXPORTS) == declared
    assert N.lib().rqb200_version() >= 100


def test_engine_flag_constants_match_the_header():
    """the binding's AR_* flag values are the header's RQB200_AR_* defines (one bit each, no overlap)"""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, "include", "rqb200.h")).read()
    flags = {n: int(v) for n, v in re.findall(r"#define\s+RQB200_(AR_[A-Z0-9_]+)\s+(\d+)", hdr)}
    assert len(flags) >= 8
    for name, value in flags.items():
        assert value & (value - 1) == 0, name
        assert getattr(N, name) == value, name
    assert len(set(flags.values())) == len(flags)


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_no_cpu_fallback():
    """the product path must fail loudly, never compute on the CPU"""
    ar = make_ar("tiny")
    vae = make_vae("tiny")
    with pytest.raises(N.NativeError):
        ar.sample(torch.zeros(1, 4, 4, 4, dtype=torch.long), model_aux=vae)
    with pytest.raises(N.NativeError):
        vae.decode_code(torch.zeros(1, 4, 4, 4, dtype=torch.long))
    with pytest.raises(N.NativeError):
        vae.quantizer.quantize(torch.zeros(1, 4, 4, 256))
    assert N.lib().rqb200_device_count() == 0

