"""TEST INFRASTRUCTURE ONLY -- deterministic synthetic weights shared by the fixture generator, the tests and
the bench's CPU-baseline leg.

``synth_state_dict(shapes, seed)`` fills a ``{key: shape}`` layout (the reference's ``state_dict`` layout, SURVEY.md
A.3) from one seeded CPU generator, visiting keys in sorted order, so the reference (in the build container), the
oracle and the CUDA engine (on the GPU box, where the reference is absent) all get bit-identical weights from
``(layout, seed)`` alone -- no weight file has to travel.  Distributions follow the reference constructors'
defaults (Linear/Conv: U(+-1/sqrt(fan_in)); Embedding: N(0,1); pos_emb: N(0,0.02), transformers.py:79-81) except
that norm layers get a non-trivial affine (1+0.1 N, 0.1 N) so that the affine path is actually exercised.
"""
import hashlib
import math

import torch


def _fan_in(shape):
    n = 1
    for s in shape[1:]:
        n *= s
    return max(n, 1)


def synth_state_dict(shapes, seed=0):
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for k in sorted(shapes):
        shp = tuple(shapes[k])
        if k.endswith("cluster_size_ema"):
            sd[k] = torch.zeros(shp)
        elif k.endswith("embed_ema"):
            sd[k] = None                                  # filled from the codebook below
        elif k.startswith("pos_emb"):
            sd[k] = torch.randn(shp, generator=g) * 0.02
        elif "codebooks" in k and k.endswith(".weight"):
            w = torch.randn(shp, generator=g)
            w[-1].zero_()                                 # padding row (quantizations.py:28)
            sd[k] = w
        elif k == "cond_emb.weight":
            sd[k] = torch.randn(shp, generator=g)
        elif re_norm(k):
            if k.endswith(".weight"):
                sd[k] = 1.0 + 0.1 * torch.randn(shp, generator=g)
            else:
                sd[k] = 0.1 * torch.randn(shp, generator=g)
        elif k.endswith(".weight"):
            b = 1.0 / math.sqrt(_fan_in(shp))
            sd[k] = (torch.rand(shp, generator=g) * 2 - 1) * b
        elif k.endswith(".bias"):
            wk = k[:-5] + ".weight"
            b = 1.0 / math.sqrt(_fan_in(tuple(shapes[wk]))) if wk in shapes else 0.02
            sd[k] = (torch.rand(shp, generator=g) * 2 - 1) * b
        else:
            sd[k] = torch.randn(shp, generator=g) * 0.02
    # shared codebook: all D entries alias one tensor in the reference (quantizations.py:199-205)
    cb_keys = sorted(k for k in sd if "codebooks" in k and k.endswith(".weight"))
    for k in cb_keys:
        sd[k] = sd[cb_keys[0]]
    for k in sd:
        if k.endswith("embed_ema"):
            sd[k] = sd[cb_keys[0]][:-1].clone()
    return sd


def re_norm(k):
    parts = k.split(".")
    name = parts[-2] if len(parts) >= 2 else ""
    return name.startswith("norm") or name.startswith("ln") or name in ("layer_norm",)


def shapes_of(state_dict):
    return {k: tuple(v.shape) for k, v in state_dict.items()}


def tensor_digests(state_dict):
    """{key: [shape, sha256 of the raw bytes]} -- pins a state dict bit for bit without storing its values"""
    return {k: [list(v.shape), hashlib.sha256(v.detach().contiguous().cpu().numpy().tobytes()).hexdigest()]
            for k, v in state_dict.items()}


def randn_seeded(shape, seed, scale=1.0):
    return torch.randn(shape, generator=torch.Generator().manual_seed(seed)) * scale


def randint_seeded(lo, hi, shape, seed):
    return torch.randint(lo, hi, shape, generator=torch.Generator().manual_seed(seed))


def exp_noise(seed, step, B, V):
    """per-token Exp(1) noise [B,V] from its own seeded generator (stream-independent of model/init RNG)."""
    g = torch.Generator().manual_seed(seed * 100003 + step)
    return torch.empty(B, V).exponential_(1, generator=g)
