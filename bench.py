#!/usr/bin/env python
"""bench.py -- 256x256 images/sec of the RQ-Transformer sampling path (BASELINE.json metric).

One step = one pass of the hot path over one batch of synthetic input:
    codes  = RQTransformer.sample(zeros[B,H,W,D], model_aux=RQVAE, cond=labels / text tokens, top_k=1024[, top_p])   (P3 + sampler)
    pixels = RQVAE.decode_code(codes)                                                                             (P2)
Default workload (N=1 and every N): ImageNet-256 class-conditional 1.4B RQ-Transformer (E=1536, 24 heads, 42+6 layers,
V=K=16384, 8x8x4 codes) + the ImageNet RQ-VAE decoder, random-init weights, synthetic labels, per-GPU batch fixed
(weak scaling): each rank samples its own shard of images with seed 1234+rank (main_sampling_fid.py:166-167); the
only exchange is one all_gather of the finished [B,8,8,4] int64 code maps before the decoder (north star).
`--model` selects the other BASELINE configs (2: ffhq355m, 4: cc3m654m / cc3m654m_16, 5: t2i3900m / t2i3900m_16).

Arithmetic: the fast tier -- fp16 weights / activations / KV on tcgen05 with fp32 accumulation, the reference's own GPU
sampling class (fp16 autocast, main_sampling_fid.py:216); `--dtype bf16` selects bf16, `--precision exact` the fp32 tier.

Prints ONE JSON line (rank 0).  `value`: images/sec with inputs resident in HBM; `e2e`: same through the public API with
pinned HOST inputs (labels + empty code map) copied H2D and the finished pixels copied D2H inside the timed region;
`exact_tier`: the same step on the fp32 tier (the tier whose free-running codes are bit-exact vs the reference); `parity`:
the fast tier's teacher-forced / free-running statistics against the reference-generated trajectories of this model
(tests/golden/ar.pt) measured in this run; `strong`: the fixed-total-batch point (global batch 64 split over N GPUs).
`--impl reference` times the CPU oracle port of the reference's own PyTorch path on the host cores (rank 0 only).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "rq-vae-transformer_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

# dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed `ncu --set full` capture (profiles/), or None
TRAFFIC_NCU = {"gemm_tc_fc2": 19736320}   # profiles/ncu_ar_chain_r2_raw.csv, fc2 launch: 19.74 MB read + 0 B written (partials stay in L2)

MODELS = {
    # name: (E, heads, n_body, n_head_layers, V, block, vocab_cond, cond_len, vae attn_res, vae ch_mult, top_p, default B, text)
    "in1400m": (1536, 24, 42, 6, 16384, (8, 8, 4), 1000, 1, (8,), (1, 1, 2, 2, 4, 4), None, 64,
                "imagenet256 class-cond 1.4B RQ-Transformer 8x8x4 K=16384 top-k=1024 + RQ-VAE decode"),
    "ffhq355m": (1024, 16, 24, 4, 2048, (8, 8, 4), 1, 1, (16,), (1, 1, 2, 2, 4, 4), None, 16,
                 "FFHQ 355M RQ-Transformer unconditional 8x8x4 K=2048 top-k=1024 + RQ-VAE decode"),
    "cc3m654m": (1280, 20, 26, 4, 16384, (8, 8, 4), 16384, 32, (8,), (1, 1, 2, 2, 4, 4), 0.95, 32,
                 "CC-3M 654M text-to-image 8x8x4 (the reference's grid), 32-token prefix, top-(k,p)=(1024,0.95) + RQ-VAE decode"),
    "cc3m654m_16": (1280, 20, 26, 4, 16384, (16, 16, 4), 16384, 32, (16,), (1, 1, 2, 2, 4), 0.95, 32,
                    "CC-3M 654M text-to-image 16x16x4 (synthetic grid, f16 RQ-VAE), 32-token prefix, top-(k,p)=(1024,0.95) + decode"),
    "t2i3900m": (2560, 40, 42, 6, 16384, (8, 8, 4), 16384, 32, (8,), (1, 1, 2, 2, 4, 4), 0.95, 16,
                 "3.9B text-to-image (3800M widths + 32-token prefix) 8x8x4, top-(k,p)=(1024,0.95) + RQ-VAE decode"),
    "t2i3900m_16": (2560, 40, 42, 6, 16384, (16, 16, 4), 16384, 32, (16,), (1, 1, 2, 2, 4), 0.95, 16,
                    "3.9B text-to-image 16x16x4 (synthetic grid, f16 RQ-VAE), top-(k,p)=(1024,0.95) + decode"),
    "tiny": (128, 2, 2, 2, 512, (8, 8, 4), 10, 1, (8,), (1, 1, 2, 2, 4, 4), None, 8, "tiny"),
}


def metric_text(name):
    if name == "in1400m":
        return "256x256 images/sec (ImageNet 1.4B RQ-Transformer, 8x8x4 codes, K=16384, top-k 1024, sample+decode)"
    return "256x256 images/sec (%s, sample+decode)" % name


def build_models(name, device, precision, tiny_vae=False):
    from rqvae.models import create_model
    from rqvae.utils.config import Config, augment_arch_defaults
    E, nh, nb, nhl, V, bs, vc, cl, attn, ch_mult = MODELS[name][:10]
    ar_cfg = augment_arch_defaults(Config(
        type="rq-transformer", vocab_size=V, block_size=list(bs), vocab_size_cond=vc, block_size_cond=cl, embed_dim=E,
        input_embed_dim=256, shared_tok_emb=True, shared_cls_emb=True, input_emb_vqvae=True, head_emb_vqvae=True,
        cumsum_depth_ctx=True, body=dict(n_layer=nb, block=dict(n_head=nh)), head=dict(n_layer=nhl, block=dict(n_head=nh))))
    dd = dict(double_z=False, z_channels=256, resolution=256, in_channels=3, out_ch=3, ch=128, ch_mult=list(ch_mult),
              num_res_blocks=2, attn_resolutions=list(attn), dropout=0.0)
    if tiny_vae:
        dd.update(ch=32)
    vae_cfg = augment_arch_defaults(Config(
        type="rq-vae", hparams=dict(bottleneck_type="rq", embed_dim=256, n_embed=V, latent_shape=[bs[0], bs[1], 256],
                                    code_shape=list(bs), shared_codebook=True, decay=0.99, restart_unused_codes=True,
                                    loss_type="mse", latent_loss_weight=0.25), ddconfig=dd))
    torch.manual_seed(0)            # identical weights on every rank (replaces the reference's ~780 per-tensor broadcasts)
    with torch.device(device):
        ar, _ = create_model(ar_cfg)
        vae, _ = create_model(vae_cfg)
    ar.eval()
    vae.eval()
    ar.precision = precision
    vae.precision = precision
    return ar, vae, dd


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        self.stop_flag = True
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def ar_bytes_per_position(name, B, wbytes):
    """ALGORITHMIC HBM bytes per spatial position (SURVEY.md 8d): every body weight once, every head + classifier
    weight D times (KV reads excluded: <= 3 % at these batch sizes)."""
    E, nh, nb, nhl, V, bs = MODELS[name][:6]
    D = bs[2]
    per_block = 12 * E * E
    body, head, cls = nb * per_block, nhl * per_block, E * V
    return wbytes * (body + D * (head + cls))


def gemm_kernel_roofline(ar, B, hbm_peak, peak_src):
    """The step's dominant kernel (ncu launch list, profiles/): gemm_tc_kernel<64,8> at the split-K shapes.  Timed live: a
    CUDA graph of one launch per body layer on that layer's own fc2 weight (42 x 18.9 MB = 0.8 GB >> L2, i.e. cold
    weights, exactly as in the step), replayed; CUDA events on the launching stream.  Algorithmic bytes = weights +
    activations in + the [B,E] fp32 result; the split-K partials are L2-resident scratch (ncu: 0 B written to DRAM)."""
    from rqvae import _native as N
    L = N.lib()
    blocks = ar.body_transformer.blocks
    E = ar.config.embed_dim
    dt = N.fast_dtype()
    Ws = [b.mlp[2].weight.detach().to(dt).contiguous() for b in blocks]       # [E, 4E]
    X = torch.randn(B, 4 * E, device=Ws[0].device).to(dt)
    splits = max(1, min(148 // (E // 128), 4 * E // 64))
    part = torch.empty(splits, B, E, device=Ws[0].device)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        def launch_all():
            for W in Ws:
                N.check(L.rqb200_dbg_gemm_tc(N.ptr(W), N.ptr(X), None, None, None, 0, 0, N.ptr(part), E, 4 * E, B, splits,
                                             0 if dt == torch.float16 else 1, N.stream_ptr()), "dbg_gemm_tc")
        launch_all()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=stream):
            launch_all()
        for _ in range(3):
            g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for _ in range(reps):
            g.replay()
        e1.record()
        torch.cuda.synchronize()
    us = e0.elapsed_time(e1) * 1e3 / (reps * len(Ws))
    alg = E * 4 * E * 2 + B * 4 * E * 2 + B * E * 4                      # weights + activations in + result out
    ach = alg / 1e9 / (us * 1e-6)
    return {"bound": "hbm", "kernel": "gemm_tc_kernel<64,8> fc2 (N_out=%d, K=%d, B=%d, split-K %d, %d CTAs)" % (E, 4 * E, B, splits, E // 128 * splits),
            "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "us_per_launch": us,
            "algorithmic_bytes_per_launch": alg, "traffic": None, "peak_source": peak_src,
            "how": "CUDA graph of %d back-to-back launches on distinct (cold) layer weights, CUDA events, %d replays" % (len(Ws), reps)}


def cpu_reference_leg(name, steps, warmup, budget_s, B):
    """The reference's own CPU PyTorch path, restated in oracle/rq_oracle.py (kind = 'port': the reference's classes do not travel
    to the GPU box), all host threads, at the STATED per-GPU batch.  One full batch of the 1.4B model takes ~90 s of host time, so
    a step is a bounded sample of the workload: the first `n_pos` of the H*W spatial positions of `sample` (D tokens each, KV
    cache growing as in the real loop) + `n_dec` of the B per-image decodes (the reference decodes image by image,
    main_sampling_fid.py:223); images/s = B / (H*W * t_position + B * t_decode)."""
    from oracle import rq_oracle as O
    E, nh, nb, nhl, V, bs, vc, cl = MODELS[name][:8]
    top_p = MODELS[name][10]
    # all physical cores this process may run on (torchrun exports OMP_NUM_THREADS=1; 2 hardware threads per core on the GPU hosts:
    # one torch thread per logical CPU measured 30x slower here)
    try:
        logical = len(os.sched_getaffinity(0))
    except AttributeError:
        logical = os.cpu_count() or 1
    torch.set_num_threads(max(1, logical // 2 if logical >= 16 else logical))
    cores = torch.get_num_threads()
    torch.manual_seed(0)
    ar, vae, dd = build_models(name, "cpu", "exact")
    sd = {k: v.detach() for k, v in ar.state_dict().items()}
    vsd = {k: v.detach() for k, v in vae.state_dict().items()}
    cfg = O.ArConfig(E, nh, nb, nhl, V, bs, vc, cl)
    table = O.codebook_of(vsd)
    torch.set_grad_enabled(False)
    HW, D = bs[0] * bs[1], bs[2]

    def ar_positions(n_pos):
        cond = torch.randint(0, max(vc, 1), (B, cl))
        state = O.new_state(cfg)
        xs = torch.zeros(B, *bs, dtype=torch.long)
        t0 = time.perf_counter()
        for idx in range(n_pos):
            h, w = idx // bs[1], idx % bs[1]
            for d in range(D):
                lg = O.ar_cached_forward(sd, cfg, state, xs[:, :h + 1], table, cond, (h, w, d))
                xs[:, h, w, d] = O.sample_from_logits(lg, 1.0, min(1024, V), top_p)
        return (time.perf_counter() - t0) / n_pos, xs

    def decodes(xs, n_dec):
        t0 = time.perf_counter()
        for i in range(n_dec):
            O.vae_decode_code(vsd, dd, xs[i:i + 1])
        return (time.perf_counter() - t0) / n_dec

    # calibrate on one position / one decode, then size the per-step sample to the budget
    t_pos, xs = ar_positions(1)
    t_dec = decodes(xs, 1)
    per_step = max(budget_s / max(steps + warmup, 1) - 0.0, 0.5)
    n_pos = int(max(1, min(HW, (0.75 * per_step) // max(t_pos, 1e-3))))
    n_dec = int(max(1, min(B, (0.25 * per_step) // max(t_dec, 1e-3))))
    tp, td = [], []
    for i in range(steps + warmup):
        a, xs = ar_positions(n_pos)
        b = decodes(xs, n_dec)
        if i >= warmup:
            tp.append(a)
            td.append(b)
    t_pos, t_dec = sum(tp) / len(tp), sum(td) / len(td)
    t_batch = HW * t_pos + B * t_dec
    return {"value": B / t_batch, "B": B, "cores": cores, "ms_per_step": 1000 * t_batch,
            "ar_ms_per_token": 1000 * t_pos / D,
            "sample": "per step: the first %d of %d spatial positions of sample() at B=%d (%.2f s / position) + %d of %d per-image "
                      "decodes (%.2f s / image), %d steps after %d warm-up; images/s = B / (%d * t_position + B * t_decode)"
                      % (n_pos, HW, B, t_pos, n_dec, B, t_dec, len(tp), warmup, HW)}


def parity_record(name, dev):
    """Fast tier vs the reference, measured in THIS run on this model shape: the reference-generated trajectories and logits of
    tests/golden/ar.pt (written by oracle/gen_golden.py from the unmodified reference; weights / noise regenerated from seeds).
    teacher_forced: fast-tier logits vs the fp32 exact tier (itself bit-exact vs the reference, tests/test_gpu_parity.py) and vs
    the logits the reference stored; greedy index flips and how many of them fall OUTSIDE the fp32 decision margin (must be 0).
    free_running: first divergent AR step per sample against the reference's trajectory (SURVEY Appendix E)."""
    import json as _json
    from oracle import synth
    from tests.helpers import CodebookAux, build_ar, noise_tensor
    gold = os.path.join(ROOT, "tests", "golden")
    g, fixture = None, None
    for fixture in ("ar.pt", "ar2.pt", "ar3.pt"):
        g = torch.load(os.path.join(gold, fixture), weights_only=False)["ar"].get(name)
        if g is not None:
            break
    if g is None:
        return {"unavailable": "no reference fixture for " + name}
    with open(os.path.join(gold, "state_dict_layouts.json")) as f:
        layouts = _json.load(f)
    E, nh, nb, nhl, V, bs, vc, cl = MODELS[name][:8]
    model, _ = build_ar(name, layouts, g["weight_seed"], dev)
    aux = CodebookAux(synth.randn_seeded((V, 256), g["codebook_seed"]).to(dev))
    B = g["B"]
    cond = synth.randint_seeded(0, max(vc, 1), (B, cl), g["cond_seed"]).to(dev) if vc > 1 else None
    ref_run = next((r for r in g["runs"] if r["logits"]), g["runs"][-1])      # a trajectory the reference stored logits for
    codes = ref_run["codes"].long().to(dev)
    tf = dict(noise=False, return_logits=True, force_codes=codes)
    model.precision = "exact"
    _, lg32 = model._native_sample(codes, aux, cond, (0, 0), 1.0, None, None, False, **tf)
    model.precision = "fast"
    _, lg16 = model._native_sample(codes, aux, cond, (0, 0), 1.0, None, None, True, **tf)
    err = (lg16 - lg32).abs()
    top2 = lg32.topk(2, dim=-1).values
    differ = lg16.argmax(-1) != lg32.argmax(-1)
    outside = differ & ((top2[..., 0] - top2[..., 1]) > 2 * err.amax(-1))
    std = float(lg32.std())
    ref_err = None
    if ref_run["logits"]:
        ref_err = max(float((lg16[s].cpu() - lg).abs().max()) for s, lg in ref_run["logits"].items())
    n_tok = bs[0] * bs[1] * bs[2]
    free = []
    for run in g["runs"]:
        st = run["setting"]
        noise = noise_tensor(run["noise_seed"], n_tok, B, V, dev)
        got = model._native_sample(torch.zeros(B, *bs, dtype=torch.long, device=dev), aux, cond, (0, 0), 1.0, st.get("top_k"),
                                   st.get("top_p"), True, noise=noise).cpu().reshape(B, -1)
        ref = run["codes"].long().reshape(B, -1)
        first = [int((got[b] != ref[b]).nonzero()[0]) if bool((got[b] != ref[b]).any()) else n_tok for b in range(B)]
        free.append({"setting": {k: v for k, v in st.items()}, "first_divergent_step": first, "n_steps": n_tok})
    del model
    torch.cuda.empty_cache()
    return {"reference_fixture": "tests/golden/%s[%s] (B=%d, unmodified reference, fp32)" % (fixture, name, B),
            "teacher_forced": {"trajectory": {k: v for k, v in ref_run["setting"].items()}, "logit_std": std, "err_rms_over_std": float(err.pow(2).mean().sqrt()) / std,
                               "err_max_over_std": float(err.max()) / std, "max_err_vs_reference_logits": ref_err,
                               "greedy_flips": int(differ.sum()), "greedy_flips_outside_margin": int(outside.sum()),
                               "steps": int(differ.numel())},
            "free_running": free}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, codes, pix, rank, world):
    """What a caller of the timed path receives -- the [B,H,W,D] code maps and the [B,3,R,R] pixels in [0,1] -- as float32
    .npy files, so that two builds can be compared output for output on identical seeded inputs.  All ranks together stay
    within DUMP_BYTES: when the pixels do not fit, a fixed seeded subset of the images is written, with their batch indices
    in pixels_index.npy."""
    import numpy as np
    sfx = "_rank%d" % rank if world > 1 else ""
    codes = codes.float().cpu().numpy()
    pix = pix.float().cpu().numpy()
    per_image = pix[0].nbytes
    keep = max(1, min(len(pix), (DUMP_BYTES // max(world, 1) - codes.nbytes - 8 * len(pix)) // per_image))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "codes%s.npy" % sfx), codes)
    if keep < len(pix):
        idx = np.sort(np.random.default_rng(0).choice(len(pix), keep, replace=False))
        pix = pix[idx]
        np.save(os.path.join(out_dir, "pixels_index%s.npy" % sfx), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "pixels%s.npy" % sfx), pix)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="in1400m", choices=list(MODELS))
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (weak scaling); 0 = the config's batch")
    ap.add_argument("--precision", default="fast", choices=["fast", "exact"])
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"], help="16-bit operand format of the fast tier")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the exact_tier and strong records")
    ap.add_argument("--cpu-budget", type=float, default=25.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the codes and pixels of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; --impl reference times a bounded sample of the CPU path")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    name = args.model
    E, nh, nb, nhl, V, bs, vc, cl, attn, ch_mult, top_p, defB, text = MODELS[name]
    H, W, D = bs
    B = args.batch or defB
    os.environ["RQB200_FAST_DTYPE"] = args.dtype
    config = {"workload": text, "per_gpu_batch": B, "global_batch": B * max(world, 1), "grid": "%dx%dx%d" % bs,
              "parallelism": "dp%d (independent images, one all_gather of code maps)" % max(world, 1),
              "l2": "inputs larger than L2: %.2f GB of weights streamed per spatial position" % (ar_bytes_per_position(name, B, 2) / 1e9)}

    if args.impl == "reference":
        if rank != 0:
            return 0
        r = cpu_reference_leg(name, args.steps, args.warmup, budget_s=150.0, B=B)
        line = {"impl": "reference", "metric": metric_text(name) + " [CPU arm: oracle port of the reference's PyTorch path]",
                "value": r["value"], "unit": "images/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "ar_ms_per_token": r["ar_ms_per_token"],
                "cpu_baseline": {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]},
                "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback (use --impl reference for the CPU baseline)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from rqvae import _native as N
    from rqvae.utils.utils import set_seed
    torch.set_grad_enabled(False)
    ar, vae, dd = build_models(name, dev, args.precision)
    set_seed(1234 + rank)
    amp = args.precision == "fast"
    kw = dict(top_k=min(1024, V), top_p=top_p, amp=amp)

    def make_io(b):
        lab = torch.randint(0, max(vc, 1), (b, cl)).pin_memory()
        emp = torch.zeros(b, H, W, D, dtype=torch.long).pin_memory()
        return {"B": b, "lab_h": lab, "emp_h": emp, "lab_d": lab.to(dev), "emp_d": emp.to(dev),
                "pix_h": torch.empty(b, 3, dd["resolution"], dd["resolution"]).pin_memory(),
                "gathered": [torch.empty(b, H, W, D, dtype=torch.long, device=dev) for _ in range(world)] if world > 1 else None}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(io, e2e, steps, model=ar):
        ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
        barrier()
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for i in range(steps):
            ev[i][0].record()
            if e2e:
                cond = io["lab_h"].to(dev, non_blocking=True)
                part = io["emp_h"].to(dev, non_blocking=True)
            else:
                cond, part = io["lab_d"], io["emp_d"]
            codes = model.sample(part, model_aux=vae, cond=cond, **kw)
            ev[i][1].record()
            if world > 1:
                dist.all_gather(io["gathered"], codes)   # the single collective: finished code maps (2 KB / image)
                codes = io["gathered"][rank]             # every rank decodes its own shard
            pix = vae.decode_code(codes)
            pix = (pix * 0.5 + 0.5).clamp_(0, 1)
            if e2e:
                io["pix_h"].copy_(pix, non_blocking=True)
            ev[i][2].record()
            io["last"] = (codes, pix)
        t1.record()
        barrier()
        total = t0.elapsed_time(t1)
        ar_ms = sum(e[0].elapsed_time(e[1]) for e in ev)
        dec_ms = sum(e[1].elapsed_time(e[2]) for e in ev)
        tt = torch.tensor([total, ar_ms, dec_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return [float(x) for x in tt]

    io = make_io(B)
    timed(io, False, args.warmup)
    launches0 = N.launch_count["total"]
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    total, ar_ms, dec_ms = timed(io, False, args.steps)
    clock_summary = clocks.summary() if rank == 0 else None
    launches = N.launch_count["total"] - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, *io["last"], rank, world)
    timed(io, True, 1)
    e_total, e_ar, e_dec = timed(io, True, args.steps)

    n_img = B * max(world, 1) * args.steps
    value = n_img / (total / 1e3)
    e2e_value = n_img / (e_total / 1e3)
    ar_ms_token = ar_ms / args.steps / (H * W * D)
    # P3 roofline: algorithmic bytes per spatial position / measured time per position (weights stream from HBM every
    # position: 3.94 GB >> 126 MB L2)
    wbytes = 2 if amp else 4
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
    pos_ms = ar_ms / args.steps / (H * W)
    ach = ar_bytes_per_position(name, B, wbytes) / 1e9 / (pos_ms / 1e3)
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
    roofline_step = {"bound": "hbm", "kernel": "AR spatial position (body stack + D x (head stack + classifier + sampler))",
                     "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak, "traffic": None,
                     "algorithmic_bytes_per_position": ar_bytes_per_position(name, B, wbytes), "ms_per_position": pos_ms,
                     "peak_source": peak_src}
    roofline = roofline_step
    if rank == 0 and amp:
        try:
            roofline = gemm_kernel_roofline(ar, B, hbm_peak, peak_src)
            roofline["traffic"] = TRAFFIC_NCU.get("gemm_tc_fc2") if name == "in1400m" and B == 64 else None
        except Exception as ex:
            roofline = dict(roofline_step, note="kernel-level measurement failed: %s" % str(ex)[:120])
    line = {"metric": metric_text(name), "value": value, "unit": "images/s", "n_gpus": max(world, 1), "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": (args.dtype if amp else "f32"), "data": "synthetic", "config": config,
            "ar_ms_per_token": ar_ms_token, "ar_ms_per_step": ar_ms / args.steps, "decode_ms_per_step": dec_ms / args.steps,
            "clocks": clock_summary, "gpu_launches": launches,
            "e2e": {"value": e2e_value, "unit": "images/s",
                    "h2d_bytes_per_step": io["lab_h"].numel() * 8 + io["emp_h"].numel() * 8,
                    "d2h_bytes_per_step": io["pix_h"].numel() * 4},
            "roofline": roofline, "roofline_ar_step": roofline_step}

    if not args.no_extras:
        # strong scaling point of BASELINE config 3: a fixed global batch (the config's batch) split over the N GPUs
        gb = defB
        if world > 1 and gb % world == 0:
            ios = make_io(gb // world)
            timed(ios, False, 2)
            s_total, s_ar, s_dec = timed(ios, False, max(2, args.steps // 2))
            line["strong"] = {"global_batch": gb, "per_gpu_batch": gb // world, "value": gb * max(2, args.steps // 2) / (s_total / 1e3),
                              "unit": "images/s", "ms_per_step": s_total / max(2, args.steps // 2),
                              "note": "weight-streaming bound: every GPU streams all weights for fewer rows (SURVEY finding 5)"}
        elif world == 1:
            line["strong"] = {"global_batch": gb, "per_gpu_batch": B, "value": value if B == gb else None, "unit": "images/s",
                              "note": "N=1: identical to `value` when --batch equals the config's global batch"}
        # the fp32 exact tier (bit-exact free-running codes vs the reference) on the same step
        if amp:
            try:
                ar.precision = "exact"
                vae.precision = "exact"
                kw["amp"] = False
                timed(io, False, 1)
                x_total, x_ar, x_dec = timed(io, False, 2)
                line["exact_tier"] = {"value": B * max(world, 1) * 2 / (x_total / 1e3), "unit": "images/s", "dtype": "f32",
                                      "ar_ms_per_token": x_ar / 2 / (H * W * D), "ar_ms_per_step": x_ar / 2,
                                      "decode_ms_per_step": x_dec / 2,
                                      "parity": "free-running codes bit-exact vs the reference (tests/test_gpu_parity.py)"}
            except Exception as ex:
                line["exact_tier"] = {"error": str(ex)[:200]}
            finally:
                ar.precision = "fast"
                vae.precision = "fast"
                kw["amp"] = True
                ar._invalidate_native()
                vae._invalidate_native()
                torch.cuda.empty_cache()
    if rank == 0:
        if amp and not args.no_parity:
            try:
                line["parity"] = parity_record(name, dev)
            except Exception as ex:
                line["parity"] = {"error": str(ex)[:200]}
        if not args.no_cpu_baseline and world == 1:
            try:
                r = cpu_reference_leg(name, 1, 0, budget_s=args.cpu_budget, B=B)
                line["cpu_baseline"] = {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port",
                                        "sample": r["sample"], "ar_ms_per_token": r["ar_ms_per_token"]}
            except Exception as ex:   # the baseline is reported, never required
                line["cpu_baseline"] = {"value": None, "error": str(ex)[:200]}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
