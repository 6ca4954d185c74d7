"""Fast tier (fp16 -- the reference's autocast class -- or bf16 operands on tcgen05, PDL chain, CUDA graphs) of the AR step
against (a) the logits the unmodified reference stored in tests/golden/ar.pt and (b) the fp32 exact tier, which is itself
pinned bit-exactly to the reference fixtures (tests/test_gpu_parity.py).  Protocol (SURVEY.md 8c / Appendix E):
teacher-forced step parity -- logits within a 16-bit error bound, indices identical except where the fp32 decision margin is
inside that bound --, the free-running first-divergence statistic against the reference's own trajectories, and
self-consistency of the free-running loop (graph == no graph, run-to-run determinism, resume, chunked noise)."""
import os

import pytest
import torch

from oracle import synth
from oracle.zoo import AR_ZOO, ar_fixture
from tests.helpers import CodebookAux, build_ar, noise_tensor

pytestmark = pytest.mark.gpu
torch.set_grad_enabled(False)
DEV = "cuda"


def _case(name, golden, layouts):
    g = golden(ar_fixture(name))["ar"][name]
    E, nh, nb_, nhl, V, bs, vc, cl = AR_ZOO[name]
    model, sd = build_ar(name, layouts, g["weight_seed"])
    cb = synth.randn_seeded((V, 256), g["codebook_seed"]).to(DEV)
    cond = synth.randint_seeded(0, max(vc, 1), (g["B"], cl), g["cond_seed"]).to(DEV) if vc > 1 else None
    return g, model, CodebookAux(cb), cond, bs, V


def _with_env(model, env, fn):
    for k, v in env.items():
        os.environ[k] = v
    model._invalidate_native()
    try:
        return fn()
    finally:
        for k in env:
            del os.environ[k]
        model._invalidate_native()


def fast_tier_parity_stats(model, aux, cond, g, bs, V):
    """the numbers the bench line's `parity` record carries: teacher-forced on the reference's last (seeded top-k) trajectory"""
    codes = g["runs"][-1]["codes"].long().to(DEV)
    tf = dict(noise=False, return_logits=True, force_codes=codes)
    model.precision = "exact"
    _, lg32 = model._native_sample(codes, aux, cond, (0, 0), 1.0, None, None, False, **tf)
    model.precision = "fast"
    out, lg16 = model._native_sample(codes, aux, cond, (0, 0), 1.0, None, None, True, **tf)
    assert torch.equal(out, codes)
    err = (lg16 - lg32).abs()
    top2 = lg32.topk(2, dim=-1).values
    margin = top2[..., 0] - top2[..., 1]
    differ = lg16.argmax(-1) != lg32.argmax(-1)
    outside = differ & (margin > 2 * err.amax(-1))
    return dict(std=float(lg32.std()), rms=float(err.pow(2).mean().sqrt()), max=float(err.max()), flips=int(differ.sum()),
                flips_outside_margin=int(outside.sum()), n=differ.numel(), lg16=lg16, lg32=lg32)


@pytest.mark.parametrize("name", ["tiny", "tiny_txt", "ffhq355m", "in1400m", "cc3m654m", "t2i3900m"])
@pytest.mark.parametrize("fmt", ["fp16", "bf16"])
def test_fast_tier_teacher_forced_step_parity(golden, layouts, name, fmt):
    g, model, aux, cond, bs, V = _case(name, golden, layouts)
    r = _with_env(model, {"RQB200_FAST_DTYPE": fmt}, lambda: fast_tier_parity_stats(model, aux, cond, g, bs, V))
    print("%s %s: logits std %.3f, fast-tier error rms %.5f max %.5f; %d / %d greedy indices differ, %d outside the margin bound"
          % (name, fmt, r["std"], r["rms"], r["max"], r["flips"], r["n"], r["flips_outside_margin"]))
    # fp16 has three more mantissa bits than bf16: its bound is 4x tighter
    k = 1.0 if fmt == "bf16" else 0.25
    assert r["rms"] < 0.02 * k * r["std"] and r["max"] < 0.15 * k * r["std"]
    assert r["flips_outside_margin"] == 0, "index flip outside the arithmetic error bound"
    # ... and against the logits the REFERENCE itself stored for this trajectory (golden fixture), not only our exact tier
    run = g["runs"][-1]
    if run["logits"]:
        for step, lg in run["logits"].items():
            e = (r["lg16"][step].cpu() - lg).abs()
            assert float(e.max()) < 0.15 * k * r["std"] + 2e-4, (step, float(e.max()))


@pytest.mark.parametrize("name", ["ffhq355m", "in1400m"])
def test_fast_tier_free_running_first_divergence_vs_reference(golden, layouts, name):
    """SURVEY Appendix E statistic: free-running fp16 sampling against the reference's own fp32 trajectories under the same
    injected noise -- a 16-bit tier cannot pass a bit-exact free-running gate (the reference itself does not: bf16-vs-fp32 of the
    SAME code diverges at step 48-120 greedy); what is recorded is the first divergent step per sample.  Gate: no divergence
    before step 8 for seeded top-k (wide Exp(1) margins), and every sample's prefix up to its divergence is identical."""
    g, model, aux, cond, bs, V = _case(name, golden, layouts)
    model.precision = "fast"
    B = g["B"]
    n_tok = bs[0] * bs[1] * bs[2]
    for run in g["runs"]:
        st = run["setting"]
        noise = noise_tensor(run["noise_seed"], n_tok, B, V)
        codes = model._native_sample(torch.zeros(B, *bs, dtype=torch.long, device=DEV), aux, cond, (0, 0), 1.0, st.get("top_k"),
                                     st.get("top_p"), True, noise=noise).cpu().reshape(B, -1)
        ref = run["codes"].long().reshape(B, -1)
        first = [int((codes[b] != ref[b]).nonzero()[0]) if bool((codes[b] != ref[b]).any()) else n_tok for b in range(B)]
        print("%s %s: first divergent step per sample %s of %d" % (name, st, first, n_tok))
        if st.get("top_k", 0) and st.get("top_k") > 1:
            assert min(first) >= 8, first


def test_fast_tier_free_running_consistency(golden, layouts):
    g, model, aux, cond, bs, V = _case("tiny", golden, layouts)
    model.precision = "fast"
    B = g["B"]
    n_tok = bs[0] * bs[1] * bs[2]
    noise = noise_tensor(77, n_tok, B, V)
    part = torch.zeros(B, *bs, dtype=torch.long, device=DEV)
    a = model._native_sample(part, aux, cond, (0, 0), 1.0, 100, 0.95, True, noise=noise)
    b = model._native_sample(part, aux, cond, (0, 0), 1.0, 100, 0.95, True, noise=noise)
    assert torch.equal(a, b), "fast tier is not run-to-run deterministic"
    assert int(a.min()) >= 0 and int(a.max()) < V
    # free-running == teacher-forced replay of its own trajectory
    _, lg = model._native_sample(a, aux, cond, (0, 0), 1.0, 100, 0.95, True, noise=False, return_logits=True, force_codes=a)
    from rqvae.models import _bind as nb
    for step in (0, 1, 5, n_tok - 1):
        idx = nb.sample_logits(lg[step], 1.0, 100, 0.95, q=noise[step])
        assert torch.equal(idx, a.reshape(B, -1)[:, step])
    # resume from the middle reproduces the tail when fed the same noise tail
    h0, w0 = bs[0] // 2, 1
    skip = (h0 * bs[1] + w0) * bs[2]
    c = _with_env(model, {"RQB200_SEQ_PREFILL": "1"},
                  lambda: model._native_sample(a, aux, cond, (h0, w0), 1.0, 100, 0.95, True, noise=noise[skip:].contiguous()))
    assert torch.equal(c, a)
    # the default (batched, one M = B*T pass) prefill sums in a different order: same prefix by construction, and on this toy the
    # same tail unless a sampled token sat on a rounding-level tie
    cb = model._native_sample(a, aux, cond, (h0, w0), 1.0, 100, 0.95, True, noise=noise[skip:].contiguous())
    assert torch.equal(cb.flatten(1)[:, :skip], a.flatten(1)[:, :skip])
    print("resume with batched prefill: %d of %d tail codes differ from the sequential-prefill trajectory"
          % (int((cb != a).sum()), cb.numel() - B * skip))
    # CUDA graphs, PDL, ring depth and L2 prefetch are pure scheduling: same codes without / with them
    for var in ("RQB200_NO_GRAPH", "RQB200_NO_PDL", "RQB200_GEMM_SHALLOW", "RQB200_GEMM_L2PF", "RQB200_TRACE"):
        d = _with_env(model, {var: "1"}, lambda: model._native_sample(part, aux, cond, (0, 0), 1.0, 100, 0.95, True, noise=noise))
        assert torch.equal(a, d), var
    # noise drawn span by span (bounded buffer, KV state resumed between spans) == one call with the whole noise tensor
    torch.manual_seed(4321)
    full = torch.empty(n_tok, B, V, device=DEV)
    for t in range(n_tok):
        full[t].exponential_(1)
    want = model._native_sample(part, aux, cond, (0, 0), 1.0, 100, 0.95, True, noise=full)
    for budget in (1, 3 * 4 * B * V * 4, 1 << 40):            # one position per span, three, everything
        model.noise_budget_bytes = budget
        torch.manual_seed(4321)
        got = model._native_sample(part, aux, cond, (0, 0), 1.0, 100, 0.95, True)
        assert torch.equal(got, want), budget
    model.precision = "exact"                                 # the exact tier resumes between spans the same way
    want32 = model._native_sample(part, aux, cond, (0, 0), 1.0, 100, 0.95, False, noise=full)
    model.noise_budget_bytes = 2 * 4 * B * V * 4
    torch.manual_seed(4321)
    assert torch.equal(model._native_sample(part, aux, cond, (0, 0), 1.0, 100, 0.95, False), want32)
    model.noise_budget_bytes = 256 << 20


def test_fast_tier_text_conditioned_prefill(golden, layouts):
    """cond_len = 4 prefill + resume on the fast tier equals its own teacher-forced replay"""
    g, model, aux, cond, bs, V = _case("tiny_txt", golden, layouts)
    model.precision = "fast"
    B = g["B"]
    n_tok = bs[0] * bs[1] * bs[2]
    noise = noise_tensor(78, n_tok, B, V)
    part = torch.zeros(B, *bs, dtype=torch.long, device=DEV)
    a = model._native_sample(part, aux, cond, (0, 0), 1.0, 64, None, True, noise=noise)
    model.precision = "exact"
    _, lg32 = model._native_sample(a, aux, cond, (0, 0), 1.0, None, None, False, noise=False, return_logits=True, force_codes=a)
    model.precision = "fast"
    _, lg16 = model._native_sample(a, aux, cond, (0, 0), 1.0, None, None, True, noise=False, return_logits=True, force_codes=a)
    assert float((lg16 - lg32).abs().max()) < 0.15 * 0.25 * float(lg32.std())
    # batched prefill (one M = B*T pass) against the token-by-token prefill (its oracle): same logits up to summation order
    _, lgseq = _with_env(model, {"RQB200_SEQ_PREFILL": "1"}, lambda: model._native_sample(
        a, aux, cond, (0, 0), 1.0, None, None, True, noise=False, return_logits=True, force_codes=a))
    d = float((lg16 - lgseq).abs().max())
    print("batched vs sequential prefill (cond_len 4): max logit difference %.2e" % d)
    assert d < 0.02 * float(lg32.std())
    # start_loc resume: prefix = 4 cond tokens + the code tokens of 5 positions, batched vs sequential
    h0, w0 = 1, 2
    skip = (h0 * bs[1] + w0) * bs[2]
    rb = model._native_sample(a, aux, cond, (h0, w0), 1.0, 64, None, True, noise=noise[skip:].contiguous(), return_logits=True)
    rs = _with_env(model, {"RQB200_SEQ_PREFILL": "1"}, lambda: model._native_sample(
        a, aux, cond, (h0, w0), 1.0, 64, None, True, noise=noise[skip:].contiguous(), return_logits=True))
    assert torch.equal(rs[0], a), "sequential-prefill resume must reproduce the trajectory bit for bit"
    d = float((rb[1][0] - rs[1][0]).abs().max())
    print("resume at (%d,%d): batched vs sequential prefill, first-step max logit difference %.2e" % (h0, w0, d))
    assert d < 0.02 * float(lg32.std())
    assert torch.equal(rb[0].flatten(1)[:, :skip], a.flatten(1)[:, :skip])


def test_16x16_grid_with_text_prefix_exact_tier_vs_oracle():
    """BASELINE configs 4/5 ask for 16x16x4 grids (synthetic: the reference ships 8x8x4 only, SURVEY finding 8): body sequence
    32 + 256 tokens, 1024 sampled tokens.  Small width so the CPU oracle finishes in seconds; exact tier must match it."""
    from oracle import rq_oracle as O
    from rqvae.models import create_model
    from rqvae.utils.config import Config, augment_arch_defaults
    E, nh, nb_, nhl, V, bs, vc, cl = 128, 2, 1, 1, 512, (16, 16, 4), 32, 32
    cfg = augment_arch_defaults(Config(type="rq-transformer", vocab_size=V, block_size=list(bs), vocab_size_cond=vc, block_size_cond=cl,
                                       embed_dim=E, input_embed_dim=256, shared_tok_emb=True, shared_cls_emb=True, input_emb_vqvae=True,
                                       head_emb_vqvae=True, cumsum_depth_ctx=True, body=dict(n_layer=nb_, block=dict(n_head=nh)),
                                       head=dict(n_layer=nhl, block=dict(n_head=nh))))
    torch.manual_seed(5)
    model, _ = create_model(cfg)
    model = model.to(DEV).eval()
    sd = {k: v.detach().cpu() for k, v in model.state_dict().items()}
    cb = synth.randn_seeded((V, 256), 41)
    B = 2
    cond = synth.randint_seeded(0, vc, (B, cl), 42)
    n_tok = bs[0] * bs[1] * bs[2]
    ref = O.ar_sample(sd, O.ArConfig(E, nh, nb_, nhl, V, bs, vc, cl), torch.zeros(B, *bs, dtype=torch.long), cb, cond=cond, top_k=50,
                      top_p=0.9, noise=lambda s, b, v: synth.exp_noise(43, s, b, v))
    model.precision = "exact"
    got = model._native_sample(torch.zeros(B, *bs, dtype=torch.long, device=DEV), CodebookAux(cb.to(DEV)), cond.to(DEV), (0, 0), 1.0, 50,
                               0.9, False, noise=noise_tensor(43, n_tok, B, V))
    fd = (got.cpu() != ref).flatten(1).any(0).nonzero()
    assert len(fd) == 0, "first divergent token %d of %d" % (int(fd[0]), n_tok)
    model.precision = "fast"
    fast = model._native_sample(torch.zeros(B, *bs, dtype=torch.long, device=DEV), CodebookAux(cb.to(DEV)), cond.to(DEV), (0, 0), 1.0, 50,
                                0.9, True, noise=noise_tensor(43, n_tok, B, V))
    assert fast.shape == ref.shape and int(fast.min()) >= 0 and int(fast.max()) < V
    # fp16 tier: the first tokens (no accumulated feedback yet) agree with the fp32 trajectory
    assert torch.equal(fast.cpu().flatten(1)[:, :8], ref.flatten(1)[:, :8])


def test_fast_tier_large_batch_is_chunked(golden, layouts):
    """B > 256 (the reference's throughput runs use up to 500): chunks of <= 256 rows, each row independent of its chunk"""
    g, model, aux, cond, bs, V = _case("tiny", golden, layouts)
    model.precision = "fast"
    B = 300
    n_tok = bs[0] * bs[1] * bs[2]
    noise = torch.empty(n_tok, B, V, device=DEV).exponential_(1, generator=torch.Generator(DEV).manual_seed(3))
    cond = torch.randint(0, 10, (B, 1), device=DEV)
    part = torch.zeros(B, *bs, dtype=torch.long, device=DEV)
    full = model._native_sample(part, aux, cond, (0, 0), 1.0, 64, None, True, noise=noise)
    sub = model._native_sample(part[140:160], aux, cond[140:160], (0, 0), 1.0, 64, None, True, noise=noise[:, 140:160].contiguous())
    assert torch.equal(full[140:160], sub)


@pytest.mark.parametrize("name", ["tiny", "tiny_txt", "cc3m654m"])
def test_fast_tier_batched_forward(golden, layouts, name):
    """RQTransformer.forward on the fast tier = a handful of large-M GEMM passes (body over B*(cond_len+H*W-1) rows, head over
    B*H*W*D rows).  Against (a) the same tier's sequential teacher-forced replay, (b) the CPU oracle's forward (small shapes) incl.
    the cond_classifier logits of a text-conditioned model (reference transformers.py:153-156,185-186)."""
    from oracle import rq_oracle as O
    g, model, aux, cond, bs, V = _case(name, golden, layouts)
    E, nh, nb_, nhl, V_, bs_, vc, cl = AR_ZOO[name]
    codes = g["runs"][-1]["codes"].long().to(DEV)
    B = codes.shape[0]
    model.precision = "fast"
    out = model(codes, model_aux=aux, cond=cond, amp=True)
    cond_logits = None
    if isinstance(out, tuple):
        out, cond_logits = out
    assert out.shape == (B, *bs, V)
    _, seq = model._native_sample(codes, aux, cond, (0, 0), 1.0, None, None, True, noise=False, return_logits=True, force_codes=codes)
    seq = seq.reshape(*bs, B, V).permute(3, 0, 1, 2, 4)
    std = float(seq.std())
    d = float((out - seq).abs().max())
    print("%s: batched forward vs sequential replay (fp16 tier): max logit difference %.2e (std %.3f)" % (name, d, std))
    assert d < 0.02 * std
    if E <= 128:
        sd = {k: v.cpu() for k, v in model.state_dict().items()}
        ref = O.ar_forward(sd, O.ArConfig(E, nh, nb_, nhl, V_, bs_, vc, cl), codes.cpu(), aux.quantizer._shared_table().cpu(),
                           None if cond is None else cond.cpu())
        assert float((out.cpu() - ref).abs().max()) < 0.04 * std
    if cl > 1:
        assert cond_logits is not None and cond_logits.shape == (B, cl - 1, vc)
        sd = {k: v.cpu() for k, v in model.state_dict().items()}
        _, cref = O.ar_forward(sd, O.ArConfig(E, nh, nb_, nhl, V_, bs_, vc, cl), codes.cpu(), aux.quantizer._shared_table().cpu(),
                               cond.cpu(), with_cond_logits=True)
        e = float((cond_logits.cpu() - cref).abs().max())
        print("%s: cond_logits vs oracle: max error %.2e (std %.3f)" % (name, e, float(cref.std())))
        assert e < 0.04 * float(cref.std())


@pytest.mark.parametrize("name", ["tiny", "in1400m"])
def test_fast_tier_batched_forward_bf16(golden, layouts, name):
    """the batched passes in the bf16 operand format (the bf16 instantiations of the mma.sync attention / pair GEMM / LayerNorm
    kernels): batched forward == the same tier's sequential teacher-forced replay up to summation order"""
    g, model, aux, cond, bs, V = _case(name, golden, layouts)
    codes = g["runs"][-1]["codes"].long().to(DEV)
    B = codes.shape[0]
    model.precision = "fast"

    def run():
        out = model(codes, model_aux=aux, cond=cond, amp=True)
        out = out[0] if isinstance(out, tuple) else out
        _, seq = model._native_sample(codes, aux, cond, (0, 0), 1.0, None, None, True, noise=False, return_logits=True, force_codes=codes)
        return out, seq.reshape(*bs, B, V).permute(3, 0, 1, 2, 4)

    out, seq = _with_env(model, {"RQB200_FAST_DTYPE": "bf16"}, run)
    std = float(seq.std())
    d = float((out - seq).abs().max())
    print("%s: bf16 batched forward vs sequential replay: max logit difference %.2e (std %.3f)" % (name, d, std))
    assert d < 0.15 * std           # (bf16: 8-bit mantissa; the fp16 gate is 0.02)
