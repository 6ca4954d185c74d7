"""TEST INFRASTRUCTURE ONLY -- writes tests/golden/*.pt from the UNMODIFIED reference classes.

Run in the build container (needs /root/reference):   python oracle/gen_golden.py
Every fixture stores only seeds/configs + the reference's outputs; inputs and weights are regenerated from
``oracle/synth.py`` (bit-identical everywhere), so the fixtures stay small enough to commit.

The sampling fixtures inject the per-token Exp(1) noise by monkey-patching ``torch.multinomial`` to
``argmax(probs / q)`` (identity verified in ``check_multinomial_identity`` below and in SURVEY.md finding 7).
"""
import json
import os
import sys
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)

from oracle import ref_loader as R          # noqa: E402
from oracle import synth                    # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")

from oracle.zoo import AR2_FILES, AR_ZOO, VAE_ZOO      # noqa: E402


def ar_cfg(name):
    E, nh, nb, nhl, V, bs, vc, cl = AR_ZOO[name]
    return R.transformer_cfg(E, nh, nb, nhl, V, block_size=bs, vocab_cond=vc, cond_len=cl)


def build_ar(ns, name, seed=0):
    model = ns.RQTransformer(ar_cfg(name)).eval()
    sd = synth.synth_state_dict(synth.shapes_of(model.state_dict()), seed)
    model.load_state_dict(sd)
    return model, sd


def build_vae(ns, name, seed=0):
    kw = R.vae_kwargs(**VAE_ZOO[name])
    model = ns.RQVAE(**kw).eval()
    sd = synth.synth_state_dict(synth.shapes_of(model.state_dict()), seed)
    model.load_state_dict(sd)
    return model, sd, kw


class NoiseInjector:
    """patches torch.multinomial -> argmax(probs / q_step) with q from synth.exp_noise(seed, step, B, V)."""

    def __init__(self, seed):
        self.seed, self.step = seed, 0

    def __enter__(self):
        self._orig = torch.multinomial

        def fake(probs, num_samples=1, **kw):
            q = synth.exp_noise(self.seed, self.step, probs.shape[0], probs.shape[1])
            self.step += 1
            return torch.argmax(probs / q, dim=-1, keepdim=True)

        torch.multinomial = fake
        return self

    def __exit__(self, *a):
        torch.multinomial = self._orig


def check_multinomial_identity():
    for seed in range(8):
        probs = torch.softmax(synth.randn_seeded((4, 2048), seed, 2.0), -1)
        torch.manual_seed(seed)
        a = torch.multinomial(probs, 1).view(-1)
        torch.manual_seed(seed)
        q = torch.empty_like(probs).exponential_(1)
        assert torch.equal(a, torch.argmax(probs / q, -1)), "multinomial identity broken"


def gen_rq(ns, out):
    import importlib
    quant_mod = ns.modules["rqvae.models.rqvae.quantizations"]
    cases = []
    for (B, K, seeds) in ((2, 2048, (0, 1, 2, 3)), (64, 16384, (0, 1)), (3, 512, (7,))):
        for s in seeds:
            bott = quant_mod.RQBottleneck(latent_shape=[8, 8, 256], code_shape=[8, 8, 4], n_embed=K, shared_codebook=True).eval()
            cb = synth.randn_seeded((K, 256), 1000 + s)
            with torch.no_grad():
                bott.codebooks[0].weight[:-1].copy_(cb)
            x = synth.randn_seeded((B, 8, 8, 256), 2000 + s, 0.2)
            quants, codes = bott.quantize(x)
            emb = bott.embed_code(codes)
            cases.append(dict(B=B, K=K, seed=s, codes=codes.to(torch.int32),
                              agg_sum=[float(q.double().sum()) for q in quants],
                              agg_last_sub=quants[-1][:, ::4, ::4, ::16].clone(),
                              embed_sub=emb[:, ::4, ::4, ::16].clone()))
    # adversarial: exact ties (duplicate codewords) -> first index must win; x equal to a codeword
    K = 64
    bott = quant_mod.RQBottleneck(latent_shape=[8, 8, 256], code_shape=[8, 8, 4], n_embed=K, shared_codebook=True).eval()
    cb = synth.randn_seeded((K, 256), 4242)
    cb[40] = cb[5]
    cb[63] = cb[5]
    with torch.no_grad():
        bott.codebooks[0].weight[:-1].copy_(cb)
    x = synth.randn_seeded((1, 8, 8, 256), 4243, 0.2)
    x[0, 0, 0] = cb[5]
    x[0, 0, 1] = cb[40] * 1.0
    quants, codes = bott.quantize(x)
    out["rq_ties"] = dict(codes=codes.to(torch.int32), agg_sum=[float(q.double().sum()) for q in quants])
    out["rq"] = cases


def gen_sampler(ns, out):
    cases = []
    i = 0
    for V in (2048, 16384):
        for B in (1, 5):
            for k in (1, 250, 1024, None):
                for p in (None, 0.92, 0.95, 0.3):
                    for T in (1.0, 0.9):
                        i += 1
                        if (i % 3) and not (k == 1024 and p in (None, 0.95) and T == 1.0):
                            continue          # thin the grid but keep the BASELINE settings
                        seed = 3000 + i
                        logits = synth.randn_seeded((B, V), seed, 2.5)
                        with NoiseInjector(seed):
                            idx = ns.sample_from_logits(logits.clone(), temperature=T, top_k=k,
                                                        top_p=(1.0 if p is None else p))
                        cases.append(dict(V=V, B=B, k=k, p=p, T=T, seed=seed, idx=idx.to(torch.int32)))
    # ties at the top-k boundary + peaked rows
    seed = 3999
    logits = synth.randn_seeded((4, 2048), seed, 1.0)
    logits[:, 100:140] = 1.25                     # 40-way tie
    logits[1, 7] = 30.0                           # one-hot-ish row
    with NoiseInjector(seed):
        idx = ns.sample_from_logits(logits.clone(), temperature=1.0, top_k=20, top_p=0.9)
    cases.append(dict(V=2048, B=4, k=20, p=0.9, T=1.0, seed=seed, idx=idx.to(torch.int32), ties=True))
    out["sampler"] = cases


def gen_ar2(ns, out):
    """second batch of AR fixtures (tests/golden/ar2.pt, ar3.pt): the text-conditioned BASELINE shapes (configs 4 / 5) -- 32-token
    prefix prefill, the synthetic 16x16x4 grid, the 3.9B widths.  Same protocol as gen_ar."""
    plan = [
        ("cc3m654m", 2, [dict(top_k=1), dict(top_k=1024, top_p=0.95)], [0, 1, 4, 255]),
        ("cc3m654m_16", 2, [dict(top_k=1024, top_p=0.95)], [0, 5, 1023]),
        ("t2i3900m", 2, [dict(top_k=1024, top_p=0.95)], [0, 1, 7, 255]),
    ]
    out["ar"] = _gen_ar_plan(ns, plan, keep_logits_of=lambda si: True)


def save_ar2(res):
    """writes AR2_FILES; logits that two runs of a model share bit for bit (the runs have not diverged yet: step 0) are stored
    once, as one tensor referenced from both runs"""
    for g in res.values():
        kept = []
        for run in g["runs"]:
            for step, lg in (run["logits"] or {}).items():
                same = next((t for t in kept if torch.equal(t, lg)), None)
                if same is None:
                    kept.append(lg)
                else:
                    run["logits"][step] = same
    for fixture, names in AR2_FILES.items():
        torch.save({"ar": {n: res[n] for n in names}}, os.path.join(GOLD, fixture + ".pt"))


def gen_ar(ns, out):
    plan = [
        # name, B, vae codebook K(=V), settings list, logits steps to keep
        ("tiny", 3, [dict(top_k=1), dict(top_k=100, top_p=0.9), dict()], list(range(0, 64, 5))),
        ("tiny_txt", 2, [dict(top_k=1), dict(top_k=64, top_p=0.95)], list(range(0, 36, 4))),
        ("ffhq355m", 2, [dict(top_k=1), dict(top_k=1024)], [0, 1, 2, 3, 4, 5, 100, 255]),
        ("in1400m", 2, [dict(top_k=1), dict(top_k=1024)], [0, 3, 4, 255]),
    ]
    out["ar"] = _gen_ar_plan(ns, plan, keep_logits_of=lambda si: si == 0)


def _gen_ar_plan(ns, plan, keep_logits_of):
    res = {}
    for name, B, settings, keep in plan:
        t0 = time.time()
        model, sd = build_ar(ns, name, seed=11)
        E, nh, nb, nhl, V, bs, vc, cl = AR_ZOO[name]
        cb = synth.randn_seeded((V, 256), 12)

        class Aux:          # the only thing sample() needs from the RQ-VAE (transformers.py:109-111)
            def get_code_emb_with_depth(self, code):
                parts = [torch.nn.functional.embedding(c, cb) for c in torch.chunk(code, code.shape[-1], dim=-1)]
                return torch.cat(parts, dim=-2), None

        cond = synth.randint_seeded(0, max(vc, 1), (B, cl), 13) if vc > 1 else None
        runs = []
        for si, st in enumerate(settings):
            kept = {}
            orig_cf = model.cached_forward
            counter = [0]

            def spy(*a, **kw):
                lg = orig_cf(*a, **kw)
                if counter[0] in keep:
                    kept[counter[0]] = lg.clone()
                counter[0] += 1
                return lg

            model.cached_forward = spy
            with NoiseInjector(500 + si) as inj:
                codes = model.sample(torch.zeros(B, *bs, dtype=torch.long), model_aux=Aux(), cond=cond, **st)
            model.cached_forward = orig_cf
            runs.append(dict(setting=st, noise_seed=500 + si, codes=codes.to(torch.int32),
                             logits={k: v for k, v in kept.items()} if keep_logits_of(si) else None))
        # start_loc resume (image completion): keep the first rows of run 0, resample from (h0, w0)
        h0, w0 = bs[0] // 2, 1
        part = runs[0]["codes"].long().clone()
        with NoiseInjector(900):
            codes2 = model.sample(part, model_aux=Aux(), cond=cond, start_loc=(h0, w0), top_k=settings[-1].get("top_k"))
        res[name] = dict(B=B, weight_seed=11, codebook_seed=12, cond_seed=13, runs=runs,
                         resume=dict(start_loc=(h0, w0), noise_seed=900, codes=codes2.to(torch.int32),
                                     top_k=settings[-1].get("top_k")))
        print("  ar %-10s %.1fs" % (name, time.time() - t0), flush=True)
        del model
    return res


def gen_vae(ns, out):
    res = {}
    for name in ("tiny", "tiny_attn_mid", "ffhq", "imagenet"):
        t0 = time.time()
        model, sd, kw = build_vae(ns, name, seed=21)
        K = kw["n_embed"]
        cs = kw["code_shape"]
        R_ = kw["ddconfig"]["resolution"]
        B = 2
        codes = synth.randint_seeded(0, K, (B, *cs), 22)
        x = synth.randn_seeded((B, 3, R_, R_), 23)
        with torch.no_grad():
            pix = model.decode_code(codes)
            z_e = model.encode(x)
            out_full, _, codes_fwd = model(x)
        st = 8 if R_ >= 256 else 1
        res[name] = dict(weight_seed=21, codes_seed=22, x_seed=23, stride=st,
                         pixels_sub=pix[:, :, ::st, ::st].clone(), pixels_l2=float(pix.double().pow(2).sum().sqrt()),
                         pixels_mean=float(pix.double().mean()),
                         z_e=z_e.clone(), codes_fwd=codes_fwd.to(torch.int32),
                         recon_sub=out_full[:, :, ::st, ::st].clone(), recon_l2=float(out_full.double().pow(2).sum().sqrt()))
        print("  vae %-14s %.1fs" % (name, time.time() - t0), flush=True)
        del model
    out["vae"] = res


def gen_layouts(ns):
    lay = {}
    for name in AR_ZOO:
        if AR_ZOO[name][0] >= 1024:
            with torch.device("meta"):
                m = ns.RQTransformer(ar_cfg(name))
        else:
            m = ns.RQTransformer(ar_cfg(name))
        lay["ar/" + name] = {k: list(v.shape) for k, v in m.state_dict().items()}
    for name in VAE_ZOO:
        m = ns.RQVAE(**R.vae_kwargs(**VAE_ZOO[name]))
        lay["vae/" + name] = {k: list(v.shape) for k, v in m.state_dict().items()}
    with open(os.path.join(GOLD, "state_dict_layouts.json"), "w") as f:
        json.dump(lay, f)


def gen_seeded_init(ns):
    """the reference's default initialisation after torch.manual_seed(0) (tests/test_host_cpu.py)"""
    E, nh, nb, nhl, V, bs, vc, cl = AR_ZOO["tiny"]
    torch.manual_seed(0)
    ar = ns.RQTransformer(R.transformer_cfg(E, nh, nb, nhl, V, block_size=bs, vocab_cond=vc, cond_len=cl))
    torch.manual_seed(0)
    vae = ns.RQVAE(**R.vae_kwargs(**VAE_ZOO["tiny"]))
    with open(os.path.join(GOLD, "seeded_init.json"), "w") as f:
        json.dump({"ar/tiny": synth.tensor_digests(ar.state_dict()), "vae/tiny": synth.tensor_digests(vae.state_dict())}, f)


SCRIPTS = {"measure_throughput": os.path.join("measure_throughput", "__main__.py"),
           "main_sampling_fid": "main_sampling_fid.py",
           "compute_metrics": "compute_metrics.py"}          # imported by main_sampling_fid


def script_imports(path):
    """[[module, name or None], ...]: what a script imports from the modules this repository provides (``rqvae`` and the
    ``compat`` omegaconf / easydict stand-ins), read from its source with ast"""
    import ast
    with open(path) as f:
        tree = ast.parse(f.read())
    ours = ("rqvae", "omegaconf", "easydict")
    found = []
    for node in ast.walk(tree):
        if isinstance(node, ast.Import):
            found += [[a.name, None] for a in node.names if a.name.split(".")[0] in ours]
        elif isinstance(node, ast.ImportFrom) and node.level == 0 and node.module.split(".")[0] in ours:
            found += [[node.module, a.name] for a in node.names]
    return found


def gen_scripts(ns):
    """what the reference's own scripts take from this repository's ``rqvae`` package (tests/test_reference_scripts_cpu.py):
    every name they import from it; measure_throughput's Experiment fields and the arch configs it passes to
    augment_arch_defaults for `f=32 d=4 c=2048 model=small` and `f=32 d=4 c=16384 model=huge`; and the configs
    main_sampling_fid.load_model() reads back from a checkpoint directory written with the tiny test configs (that function
    calls this package's load_config / augment_arch_defaults, so those are a snapshot of this package's output)."""
    import dataclasses
    import importlib.util
    import tempfile
    import yaml
    pkg = os.path.join(ROOT, "rq-vae-transformer_b200")
    added = [pkg, os.path.join(pkg, "compat"), R.REFERENCE_ROOT]     # ours shadows the reference's `rqvae`
    sys.path.insert(0, added[0])
    sys.path.extend(added[1:])
    out = {"imports": {k: script_imports(os.path.join(R.REFERENCE_ROOT, rel)) for k, rel in SCRIPTS.items()}}
    try:
        def load(name, rel):
            spec = importlib.util.spec_from_file_location(name, os.path.join(R.REFERENCE_ROOT, rel))
            mod = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mod)
            return mod

        mt = load("ref_measure_throughput", SCRIPTS["measure_throughput"])
        out["measure_throughput"] = {"experiment_fields": [[f.name, f.type if isinstance(f.type, str) else f.type.__name__, f.default]
                                                           for f in dataclasses.fields(mt.Experiment)],
                                     "create_model": []}
        augment = mt.augment_arch_defaults
        for args in (("f32", "small", 4, 2048), ("f32", "huge", 4, 16384)):
            seen = []
            mt.augment_arch_defaults = lambda c: (seen.append(c.to_dict()), augment(c))[1]
            with torch.device("meta"):
                mt.create_model(*args)
            mt.augment_arch_defaults = augment
            out["measure_throughput"]["create_model"].append({"args": list(args), "rqvae": seen[0], "rqtransformer": seen[1]})

        msf = load("ref_main_sampling_fid", SCRIPTS["main_sampling_fid"])
        from tests.helpers import ar_config, vae_config
        from rqvae.models import create_model
        out["main_sampling_fid"] = {}
        with tempfile.TemporaryDirectory() as tmp:
            for name, cfg in (("ar", ar_config("tiny")), ("vae", vae_config("tiny"))):
                os.makedirs(os.path.join(tmp, name))
                model, _ = create_model(cfg)
                torch.save({"state_dict": model.state_dict(), "state_dict_ema": model.state_dict()}, os.path.join(tmp, name, "model.pt"))
                written = {"arch": cfg.to_dict(), "dataset": {"type": "imagenet"},
                           "sampling": {"temp": 1.0, "top_k": [1024], "top_p": [0.95]}}
                with open(os.path.join(tmp, name, "config.yaml"), "w") as f:
                    yaml.safe_dump(written, f)
                _, config = msf.load_model(os.path.join(tmp, name, "model.pt"), ema=(name == "ar"))
                out["main_sampling_fid"][name] = {"config_yaml": written, "loaded": config.to_dict()}
    finally:
        for p in added:
            sys.path.remove(p)
    with open(os.path.join(GOLD, "reference_scripts.json"), "w") as f:
        json.dump(out, f, indent=1)


def main():
    torch.set_grad_enabled(False)
    os.makedirs(GOLD, exist_ok=True)
    ns = R.load_reference()
    check_multinomial_identity()
    which = sys.argv[1:] or ["rq", "sampler", "ar", "vae", "ar2", "layouts", "init", "scripts"]
    for part, fn in (("rq", gen_rq), ("sampler", gen_sampler), ("ar", gen_ar), ("vae", gen_vae), ("ar2", gen_ar2)):
        if part in which:
            out = {}
            t0 = time.time()
            fn(ns, out)
            if part == "ar2":
                save_ar2(out["ar"])
            else:
                torch.save(out, os.path.join(GOLD, part + ".pt"))
            print("%s done in %.1fs" % (part, time.time() - t0), flush=True)
    if "layouts" in which:
        gen_layouts(ns)
    if "init" in which:
        gen_seeded_init(ns)
    if "scripts" in which:
        gen_scripts(ns)
    meta = dict(torch=torch.__version__, threads=torch.get_num_threads(), reference="kakaobrain/rq-vae-transformer@341395e")
    with open(os.path.join(GOLD, "META.json"), "w") as f:
        json.dump(meta, f)


if __name__ == "__main__":
    main()
