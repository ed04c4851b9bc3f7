#!/usr/bin/env python
"""bench.py — Taylor-score UNet fwd+bwd passes/sec (BASELINE.json metric) on N B200s.

A "step" = one pass of ddpm_prune.py:97-102 (add_noise -> UNet fwd -> mse -> full bwd, gradients accumulated) over one synthetic
Gaussian batch.  Workloads (--config):
  c1 (default)  CIFAR-10 DDPM UNet (tools/ddpm_cifar10_config.json, seed-0 random init), batch 128 x 3x32x32 — BASELINE configs[1]
                ("DDPM CIFAR-10 32x32 ... 1xB200"; batch from scripts/prune_ddpm_cifar10.sh).
  c3            google/ddpm-ema-bedroom-256 architecture (seed-0 random init), batch 4 x 3x256x256, ratio 0.05 — BASELINE configs[2]
                (README.md:140-148), the configuration the north star shards over 8 GPUs.
Multi-GPU: timesteps are sharded across ranks (weak scaling: every rank runs K steps on its own timesteps) and the flat gradient arena
is all-reduced ONCE at the end, inside the timed region.  Secondary leg (`finetune`): the pruned-UNet finetune step of
ddpm_train.py:437-469 on the ratio-0.3 network (imgs/s; fp32-grade and, separately, the bf16 tier of BASELINE configs[3]).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c1|c3] [--batch B] [--no-graph]
                  [--dump-outputs DIR]
Under torchrun the usual RANK/LOCAL_RANK/WORLD_SIZE/MASTER_* env is used; rank 0 prints ONE JSON line.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "taylor_score_unet_fwd_bwd_passes_per_sec"
UNIT = "passes/s"

# conv_flop: algorithmic FLOPs of the 4-D-weight convolutions per image per pass (fprop + dgrad + wgrad = 6 x MACs), SURVEY.md §8(d)
CONFIGS = {
    "c1": dict(model="CIFAR10_DDPM_CONFIG", hw=32, batch=128, conv_flop=34.27e9, ratio=0.3,
               name="C1 CIFAR-10 DDPM UNet2DModel (35.7M params, seed-0 init)",
               cpu_sample=(128, 32)),                # the reference arm runs the SAME batch (one full pass ~ seconds on the host cores)
    "c3": dict(model="LSUN256_DDPM_CONFIG", hw=256, batch=4, conv_flop=1.4806e12, ratio=0.05,
               name="C3 LSUN-256 DDPM UNet2DModel (113.7M params, google/ddpm-ema-bedroom-256 architecture, seed-0 init)",
               cpu_sample=(1, 128)),                 # a full B=4 256x256 CPU pass takes minutes: bounded sample = 1 image at 128x128 (1/16 of the conv work)
    # BASELINE configs[4]: the class-conditional ImageNet latent-diffusion UNet (ldm_exp/prune_ldm.py: 6 latents of 3x64x64 per step, one
    # context token per latent).  conv_flop here = GEMM-class work of the conv + linear launches, 6 x 99.8 G MACs (SURVEY.md §2.5 / §8d;
    # the 4.5 G MACs of the attention cores are not in the timed conv-tagged launches)
    "c5": dict(model="ldm:CIN256_V2_CONFIG", hw=64, batch=6, conv_flop=598.8e9, ratio=0.3,
               name="C5 LDM ImageNet-256 UNetModel cin256-v2 (400.9M params, seed-0 init, zero-initialised convolutions re-drawn)",
               cpu_sample=(1, 64)),
}


def make_model(cfg_key):
    """(model, scorer kwargs builder): the DDPM UNet2DModel configs, or the LDM UNetModel with its sqrt-linear schedule and a context."""
    import diff_pruning_b200 as dp
    name = CONFIGS[cfg_key]["model"]
    torch.manual_seed(0)
    if name.startswith("ldm:"):
        from diff_pruning_b200 import ldm
        cfg = getattr(ldm, name[4:])
        m = ldm.UNetModel(**cfg)
        g = torch.Generator().manual_seed(5)
        for p in m.parameters():          # a freshly constructed LDM UNet outputs exactly 0 (zero_module convolutions): re-draw them
            if p.dim() > 1 and float(p.detach().abs().sum()) == 0:
                p.data.copy_(torch.randn(p.shape, generator=g) * 0.02)

        def extra(B, dev):
            ctx = torch.randn(B, 1, cfg["context_dim"], generator=torch.Generator().manual_seed(9)).to(dev)
            return {"alphas_cumprod": ldm.ldm_alphas_cumprod(), "context": ctx}
        return m, cfg, extra
    cfg = getattr(dp, name)
    return dp.UNet2DModel(**cfg), cfg, (lambda B, dev: {})


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops_sustained", 1400.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1400.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle sampling DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        self.index = index

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(",") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for nm, v in zip(names, r[2:6]):
                if "Active" in v and "Not" not in v:
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# gradient entries --dump-outputs writes: 32 MB of float32, which with the loss keeps a dump well under 64 MB
DUMP_GRAD_SAMPLES = 1 << 23


def dump_outputs(out_dir, model, loss):
    """What a caller of the timed Taylor path holds after its last step: that step's loss (loss.npy) and the gradients accumulated in
    Parameter.grad.  Those are 143 MB for C1 and more for C3 / C5, so grad_sample.npy holds a fixed sample of them: positions drawn
    from a seeded generator in the concatenation of every .grad in named_parameters() order, sorted, so two builds are compared at the
    same entries."""
    os.makedirs(out_dir, exist_ok=True)
    flat = torch.cat([p.grad.reshape(-1) for _, p in model.named_parameters()])
    if flat.numel() > DUMP_GRAD_SAMPLES:
        idx = torch.randint(flat.numel(), (DUMP_GRAD_SAMPLES,), generator=torch.Generator().manual_seed(0)).sort().values
        flat = flat[idx.to(flat.device)]
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "grad_sample.npy"), flat.float().cpu().numpy())


def synth_batch(B, hw=32, seed_off=0):
    g1, g2 = torch.Generator().manual_seed(1 + seed_off), torch.Generator().manual_seed(2 + seed_off)
    return torch.randn(B, 3, hw, hw, generator=g1), torch.randn(B, 3, hw, hw, generator=g2)


# ------------------------------------------------------------------------------------------------------------------------
# baselines: the oracle port (torch ATen ops = the reference's own backend) on the host cores, and the same modules torch-eager
# on the GPU (cuDNN, TF32 on/off) — SURVEY.md §8(d): "time torch-eager on the same B200 as the real bar to beat"
# ------------------------------------------------------------------------------------------------------------------------
def _oracle_setup(cfg_key, sample_B, sample_hw, device="cpu"):
    model, mcfg, extra = make_model(cfg_key)
    sd = {k: v.detach().clone().to(device).requires_grad_(True) for k, v in model.state_dict().items()}
    del model
    clean, noise = synth_batch(sample_B, sample_hw)
    clean, noise = clean.to(device), noise.to(device)
    if CONFIGS[cfg_key]["model"].startswith("ldm:"):
        from oracle import ldm_oracle as lorc
        ac = lorc.alphas_cumprod().to(device)
        ctx = extra(sample_B, device)["context"]

        def one_pass(k):
            t = torch.full((sample_B,), int(k), dtype=torch.long, device=device)
            return lorc.taylor_pass(sd, mcfg, ac, clean, noise, t, ctx)
        return one_pass
    from oracle import unet_oracle as orc
    ac = orc.alphas_cumprod().to(device)

    def one_pass(k):
        t = torch.full((sample_B,), int(k), dtype=torch.long, device=device)
        return orc.taylor_pass(sd, mcfg, ac, clean, noise, t)
    return one_pass


def best_cpu_threads(one_pass):
    """Give the CPU arm its best thread count: torch's intra-op pool over-subscribes badly on 100+ core hosts for these convs
    (measured 79 s/pass at 128 threads vs ~1.5 s at 8-32, C1 batch 16), so try a few and keep the fastest."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64) if c <= ncpu}) or [ncpu]
    best, best_t = cands[0], None
    for c in cands:
        torch.set_num_threads(c)
        one_pass(0)                       # warm-up at this thread count (oneDNN primitive creation)
        t0 = time.time(); one_pass(1); dt = time.time() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
        if dt > 1.25 * best_t:            # past the knee (larger pools only get worse): stop
            break
    torch.set_num_threads(best)
    return best, best_t


def _sample_plan(cfg_key, B, budget_s, n_steps):
    """(sample_B, sample_hw, work fraction of one full step): the full batch when n_steps of it fit the budget, else the bounded sample
    the config names."""
    c = CONFIGS[cfg_key]
    sB, shw = c["cpu_sample"]
    sB = min(sB, B)
    return sB, shw, (sB * shw * shw) / float(B * c["hw"] * c["hw"])


def cpu_oracle_passes(cfg_key, B, min_seconds, max_passes):
    """cpu_baseline: the CPU restatement of the reference path (oracle port) timed on the host cores, bounded sample."""
    c = CONFIGS[cfg_key]
    sB, shw = (16, 32) if cfg_key == "c1" else c["cpu_sample"]        # ~10-30 s of CPU work inside the default GPU run
    frac = (sB * shw * shw) / float(B * c["hw"] * c["hw"])
    one_pass = _oracle_setup(cfg_key, sB, shw)
    threads, _ = best_cpu_threads(one_pass)
    one_pass(0)
    times, t_all, k = [], time.time(), 1
    while len(times) < max_passes and (time.time() - t_all < min_seconds or len(times) < 2):
        t0 = time.time(); one_pass(k); times.append(time.time() - t0); k += 1
    med = statistics.median(times)
    return {"value": frac / med, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{threads} of {os.cpu_count()} host threads (fastest of a short sweep); {len(times)} timed + 1 warm-up oracle passes at batch {sB} x "
                      f"{shw}x{shw} (median {med:.2f} s, best {min(times):.2f}) = {frac:.4g} of the conv work of one batch-{B} {c['hw']}x{c['hw']} pass, scaled by "
                      f"that fraction; loadavg {os.getloadavg()[0]:.1f}"}


def gpu_eager_passes(cfg_key, B, dev, n=5):
    """The reference's modules as torch-eager ops on THIS GPU (cuDNN / cuBLAS / ATen), same batch and resolution: the bar SURVEY.md
    §0.1 sets.  torch's default is cudnn.allow_tf32=True (convolutions in single-pass TF32) and matmul.allow_tf32=False; the fp32 row
    switches cuDNN's TF32 off as well, which is the precision class the fp32-grade tier of this repo delivers."""
    c = CONFIGS[cfg_key]
    out = {}
    prev = torch.backends.cudnn.allow_tf32
    try:
        one_pass = _oracle_setup(cfg_key, B, c["hw"], device=dev)
        for name, tf32 in (("cudnn_tf32", True), ("fp32", False)):
            torch.backends.cudnn.allow_tf32 = tf32
            for k in range(3):
                one_pass(k)
            torch.cuda.synchronize(dev)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for k in range(n):
                one_pass(3 + k)
            e1.record()
            torch.cuda.synchronize(dev)
            ms = e0.elapsed_time(e1) / n
            out[name] = {"passes_per_s": 1e3 / ms, "ms_per_pass": ms}
    except Exception as e:                      # an OOM of the eager graph must not cost the bench line
        out["error"] = f"{type(e).__name__}: {str(e)[:160]}"
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    out["what"] = (f"oracle port (torch functional ops = the reference's ATen/cuDNN path) on the same B200, batch {B} x {c['hw']}x{c['hw']}, "
                   f"CUDA events over {n} passes after 3 warm-ups; cudnn_tf32 = torch default (conv in TF32), fp32 = cudnn.allow_tf32 False")
    torch.cuda.empty_cache()
    return out


def measure_tf32_peak(dev):
    """One cuBLAS TF32 GEMM (8192^3, torch.matmul with allow_tf32), same recipe as MEASURED_PEAKS.json's bf16 figure: burst = best of 10,
    sustained = back to back for ~2 s.  Context for the gpu_eager rows: cuDNN's default convolution runs single-pass TF32."""
    prev = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        n = 8192
        a = torch.randn(n, n, device=dev); b = torch.randn(n, n, device=dev)
        for _ in range(3):
            a @ b
        torch.cuda.synchronize(dev)
        best = 1e9
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); a @ b; e1.record(); torch.cuda.synchronize(dev)
            best = min(best, e0.elapsed_time(e1))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = max(10, int(2000.0 / best))
        e0.record()
        for _ in range(reps):
            a @ b
        e1.record(); torch.cuda.synchronize(dev)
        fl = 2.0 * n ** 3
        return {"tf32_tflops": fl / (best * 1e-3) / 1e12, "tf32_tflops_sustained": fl * reps / (e0.elapsed_time(e1) * 1e-3) / 1e12,
                "how": f"torch.matmul fp32 {n}^3 with allow_tf32 (cuBLAS), best of 10 / {reps} back to back"}
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path (torch ATen ops through the oracle port — the reference
    is an un-packaged Python script tree that cannot travel to the GPU box) on the host cores, same config, metric and unit."""
    if rank != 0:
        return
    c = CONFIGS[args.config]
    B = args.batch
    sB, shw, frac = _sample_plan(args.config, B, 300.0, args.steps + args.warmup)
    one_pass = _oracle_setup(args.config, sB, shw)
    threads, t_pass = best_cpu_threads(one_pass)
    same = (sB == B and shw == c["hw"])
    if same and t_pass * (args.steps + args.warmup) > 420.0:
        # the full-batch step does not fit "a few minutes" on this host: fall back to a bounded sub-batch of 16 images
        sB, frac, same = 16, 16.0 / B, False
        one_pass = _oracle_setup(args.config, sB, shw)
        one_pass(0)
    for w in range(args.warmup):
        one_pass(w)
    t0 = time.time()
    for k in range(args.steps):
        one_pass(k)
    dt = time.time() - t0
    value = frac * args.steps / dt
    sample = (f"each step = one oracle (torch CPU fp32, ATen/oneDNN = the reference's backend) Taylor pass at batch {sB} x {shw}x{shw} on {threads} of "
              f"{os.cpu_count()} host threads (fastest of a short sweep)" +
              ("" if same else f" = {frac:.4g} of the conv work of one batch-{B} {c['hw']}x{c['hw']} pass; value scaled by that fraction"))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{c['name']} Taylor pass, batch {B} x 3x{c['hw']}x{c['hw']}", "same_config": same,
                   "cpu_sample_batch": sB, "cpu_sample_hw": shw},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


# ------------------------------------------------------------------------------------------------------------------------
# ours
# ------------------------------------------------------------------------------------------------------------------------
def timed_conv_launches(plan, prologue=None, midlogue=None):
    """Runs one eager pass of `plan` step by step with CUDA events around every launch tagged conv (fprop / dgrad / wgrad / split-K
    reduce): (summed seconds, launch count, ms by tag, ms by (tag, layer shape))."""
    s_int = torch.cuda.current_stream().cuda_stream
    s = torch.cuda.current_stream()
    pairs, others = [], []

    def run_list(steps):
        for i, f in enumerate(steps):
            if i % 64 == 0:
                # keep the GPU busy with a spin kernel (~3 ms) while the host enqueues the next launches: a CUDA-event pair around a
                # short kernel otherwise measures the host's launch latency (ctypes call + tensor-map encodes, ~20 us), not the kernel
                torch.cuda._sleep(6_000_000)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s); f(s_int); e1.record(s)
            (pairs if getattr(f, "what", "").startswith("conv") else others).append((e0, e1, getattr(f, "what", "") or "untagged", getattr(f, "info", "")))
    if prologue:
        prologue(s_int)
    run_list(plan.fwd)
    if midlogue:
        midlogue(s_int)
    saved = plan.grad_arena.clone()
    plan.gradof(plan.silu_temb).t.zero_()
    run_list(plan.bwd_steps)
    torch.cuda.synchronize()
    plan.grad_arena.copy_(saved)
    by_tag, by_layer = {}, {}
    for a, b, tag, info in pairs:
        ms = a.elapsed_time(b)
        by_tag[tag] = by_tag.get(tag, 0.0) + ms
        if info:
            key = f"{tag.replace('conv ', '')} {info}"
            cnt, tot = by_layer.get(key, (0, 0.0))
            by_layer[key] = (cnt + 1, tot + ms)
    total = sum(a.elapsed_time(b) for a, b, _, _ in pairs) * 1e-3
    other = {}
    for a, b, tag, _ in others:         # everything that is not a convolution launch, by tag (same eager, L2-warm conditions)
        other[tag] = other.get(tag, 0.0) + a.elapsed_time(b)
    timed_conv_launches.last_other_ms = {k: round(v, 3) for k, v in sorted(other.items(), key=lambda kv: -kv[1])}
    ranked = sorted(by_layer.items(), key=lambda kv: -kv[1][1])
    dump = os.environ.get("DPB200_LAYERS_OUT")           # developer knob: append the full per-layer table of every timed plan to a file
    if dump:
        with open(dump, "a") as f:
            f.write(json.dumps({"compute": getattr(plan, "compute", "fp32"), "B": plan.B, "H": plan.H, "total_ms": round(total * 1e3, 3),
                                "layers": {k: {"n": n, "ms": round(t, 4)} for k, (n, t) in ranked}}) + "\n")
    return total, len(pairs), {k: round(v, 3) for k, v in sorted(by_tag.items())}, {k: {"n": n, "ms": round(t, 3)} for k, (n, t) in ranked[:12]}


def pruned_model(cfg_key, dev, ratio=0.3):
    """The network the finetune leg trains: the config's UNet pruned at `ratio` by this package's own Taylor path (three accumulated
    scoring passes on the device, then pruning.taylor_prune — ddpm_prune.py:79-116).  Widths depend on the ratio only; for C1 this is the
    reference's 19.85 M-parameter architecture."""
    import diff_pruning_b200 as dp
    from diff_pruning_b200 import pruning
    from diff_pruning_b200.scoring import TaylorScorer
    c = CONFIGS[cfg_key]
    torch.manual_seed(0)
    m = dp.UNet2DModel(**getattr(dp, c["model"])).eval().to(dev)
    clean, noise = synth_batch(min(4, c["batch"]), c["hw"])
    m.zero_grad()
    sc = TaylorScorer(m, clean.to(dev), noise.to(dev), use_graph=False)
    for t in (0, 500, 999):
        sc.step(t)
    torch.cuda.synchronize(dev)
    del sc
    pruning.taylor_prune(m, ratio, "taylor", ignored_layers=[m.conv_out])
    m.zero_grad(set_to_none=True)
    if hasattr(m, "_dpb200_plans"):
        m._dpb200_plans.clear()
    torch.cuda.empty_cache()
    return m


def finetune_bench(args, rank, world, dev, barrier, compute="fp32"):
    """Secondary metric of BASELINE.json: finetune imgs/sec on the ratio-0.3 pruned network — ddpm_train.py:437-469 (antithetic
    timesteps, add_noise, fwd, loss, bwd, clip 1.0, Adam 2e-4, EMA 0.9999, dropout 0.1), config batch per GPU, gradient all-reduce
    (mean) per step when N > 1.  compute = "fp32" (fp32-grade 3 x fp16 split tier) or "bf16" (single-pass tier, ddpm_train.py --mixed_precision bf16)."""
    import torch.distributed as dist
    from diff_pruning_b200.scoring import FinetuneStepper
    c = CONFIGS[args.config]
    m = pruned_model(args.config, dev, 0.3)
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.1                      # scripts/finetune_ddpm_cifar10.sh --dropout 0.1 (utils.set_dropout)
    m.train()
    B, hw = args.batch, c["hw"]
    kw = {"compute": compute} if compute != "fp32" else {}
    st = FinetuneStepper(m, lr=2e-4, ema_decay=0.9999, max_grad_norm=1.0, use_graph=not args.no_graph, **kw)
    g = torch.Generator().manual_seed(7 + rank)
    clean, noise = torch.randn(B, 3, hw, hw, generator=g).to(dev), torch.randn(B, 3, hw, hw, generator=g).to(dev)
    t = torch.randint(0, 1000, (B // 2 + 1,), generator=g)
    t = torch.cat([t, 1000 - t - 1])[:B].to(dev)
    K = args.steps
    for _ in range(3):
        st.step(clean, noise, t)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        st.step(clean, noise, t)
    e1.record()
    barrier()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms[0])
    nparams = sum(p.numel() for p in m.parameters())
    res = {"metric": "finetune_imgs_per_sec", "value": world * B * K / (ms * 1e-3), "unit": "imgs/s", "ms_per_step": ms / K, "steps": K,
           "dtype": compute,
           "config": f"{args.config.upper()} pruned at ratio 0.3 by taylor_prune ({nparams / 1e6:.3f} M params), batch {B}/GPU, dropout 0.1, Adam+clip+EMA, "
                     f"{world} GPU(s)", "loss": float(st.loss.item())}
    if rank == 0:
        _, tf_sus, _, which = peaks()
        conv_s, n_conv, by_tag, by_layer = timed_conv_launches(st.plan)
        flops = 6.0 * st.plan.conv_macs
        res["roofline"] = {"bound": "tensor", "achieved": flops / conv_s / 1e12, "peak": tf_sus, "unit": "TFLOP/s",
                           "frac": flops / conv_s / 1e12 / tf_sus, "conv_ms": round(conv_s * 1e3, 3), "breakdown_ms": by_tag, "top_layers_ms": by_layer,
                           "conv_gflop_per_image": 6.0 * st.plan.conv_macs / B / 1e9,
                           "note": f"6 x conv MACs of the pruned network (from the launch plan) / summed conv-launch time of one step; peak = bf16_tflops_sustained ({which})"}
    del st
    if hasattr(m, "_dpb200_plans"):
        m._dpb200_plans.clear()
    del m
    torch.cuda.empty_cache()
    return res


def secondary_scoring_leg(cfg_key, args, rank, world, dev, barrier):
    """The Taylor-scoring metric on ANOTHER BASELINE configuration inside the default run (the driver only launches `bench.py --gpus N`):
    c3 = LSUN-256 architecture, batch 4 per GPU, timesteps sharded over the ranks, one gradient all-reduce at the end."""
    import torch.distributed as dist
    import diff_pruning_b200 as dp
    from diff_pruning_b200 import _lib as L
    from diff_pruning_b200.scoring import TaylorScorer
    lib = L.load()
    c = CONFIGS[cfg_key]
    B, hw = c["batch"], c["hw"]
    model, _, extra = make_model(cfg_key)
    model = model.eval().to(dev)
    clean, noise = synth_batch(B, hw, seed_off=100 * rank)
    model.zero_grad()
    sc = TaylorScorer(model, clean.to(dev), noise.to(dev), use_graph=not args.no_graph, **extra(B, dev))
    K, Wm = args.steps, 3
    ts = [(rank + k * world) % 1000 for k in range(Wm + K)]
    for k in range(Wm):
        sc.step(ts[k])
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(K):
        sc.step(ts[Wm + k])
    if world > 1:
        dist.all_reduce(sc.plan.grad_arena, op=dist.ReduceOp.SUM)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    res = {"metric": METRIC, "value": world * K / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / K, "steps": K, "warmup": Wm, "dtype": "f32",
           "config": {"workload": f"{c['name']} Taylor pass, batch {B} x 3x{hw}x{hw} per GPU, timesteps sharded over {world} GPU(s), one grad all-reduce at the end"}}
    if rank == 0:
        p = sc.plan

        def pro(s_int):
            p.t_dev.fill_(3)
            L.check(lib.dp_add_noise(sc.clean.data_ptr(), sc.noise.data_ptr(), p.t_dev.data_ptr(), sc.acp.data_ptr(),
                                     p.x_in.ptr, sc.B, sc.C, sc.H, sc.W, 1, p.x_in.ld, s_int))

        def mid(s_int):
            gy = p.gradof(p.y_out)
            L.check(lib.dp_mse_loss_grad(p.y_out.ptr, sc.noise_nhwc.data_ptr(), gy.ptr, sc.n, sc.loss_scale, sc.grad_scale,
                                         sc.partial.data_ptr(), sc.loss.data_ptr(), s_int))
        conv_s, n_conv, by_tag, by_layer = timed_conv_launches(p, pro, mid)
        _, tf_sus, _, which = peaks()
        ach = B * c["conv_flop"] / conv_s / 1e12
        res["roofline"] = {"bound": "tensor", "achieved": ach, "peak": tf_sus, "unit": "TFLOP/s", "frac": ach / tf_sus,
                           "conv_ms": round(conv_s * 1e3, 3), "breakdown_ms": by_tag, "top_layers_ms": by_layer,
                           "note": f"{B} x {c['conv_flop'] / 1e12:.4f} TFLOP algorithmic conv work per pass (SURVEY.md §8d) / summed conv-launch time; peak = bf16_tflops_sustained ({which}); fp32-grade 3 x fp16 split tier"}
    del sc
    if hasattr(model, "_dpb200_plans"):
        model._dpb200_plans.clear()
    del model
    torch.cuda.empty_cache()
    return res


def run_ours(args, rank, world, local_rank):
    import torch.distributed as dist
    import diff_pruning_b200 as dp
    from diff_pruning_b200 import _lib as L
    from diff_pruning_b200.scoring import TaylorScorer
    import __graft_entry__ as ge
    if rank == 0:
        ge.build()
    if world > 1:
        dist.barrier()
    lib = L.load()
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    c = CONFIGS[args.config]
    B, hw = args.batch, c["hw"]
    model, _, extra = make_model(args.config)
    model = model.eval().to(dev)
    clean, noise = synth_batch(B, hw, seed_off=100 * rank)
    clean_pin, noise_pin = clean.pin_memory(), noise.pin_memory()
    model.zero_grad()
    sc = TaylorScorer(model, clean.to(dev), noise.to(dev), use_graph=not (args.no_graph or args.profile_pass), **extra(B, dev))
    if args.profile_pass:   # for ncu: `--profile-from-start off`; exactly one eager pass inside the profiler range
        for k in range(2):
            sc.step(k)
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.start()
        sc.step(5)
        torch.cuda.synchronize(dev)
        torch.cuda.profiler.stop()
        return
    # timesteps: rank r takes t = r, r+W, r+2W, ... (SURVEY.md §8(e))
    ts = [(rank + k * world) % 1000 for k in range(args.warmup + args.steps)]
    for k in range(args.warmup):
        sc.step(ts[k])
    torch.cuda.synchronize(dev)
    launches_per_pass = None
    if not args.no_graph:
        # the graph replays exactly the launches recorded by one eager body
        c0 = lib.dp_launch_count(); saved = sc.plan.grad_arena.clone(); sc._body(); sc.plan.grad_arena.copy_(saved)
        launches_per_pass = lib.dp_launch_count() - c0
        torch.cuda.synchronize(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    # ---------------- device-resident timing
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    c_before = lib.dp_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        sc.step(ts[args.warmup + k])
    if world > 1:
        dist.all_reduce(sc.plan.grad_arena, op=dist.ReduceOp.SUM)   # the one collective of the scoring path
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, model, sc.loss)
    eager_launches = lib.dp_launch_count() - c_before
    gpu_launches = eager_launches if args.no_graph else launches_per_pass * args.steps
    # ---------------- end-to-end through host buffers (H2D batch each step, D2H loss each step)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for k in range(args.steps):
        sc.step_from_host(clean_pin, noise_pin, ts[args.warmup + k])
    if world > 1:
        dist.all_reduce(sc.plan.grad_arena, op=dist.ReduceOp.SUM)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms, ms_e2e = float(t[0]), float(t[1])
    # ---------------- roofline of the dominant kernel family (conv implicit GEMM), live CUDA events
    if rank == 0:
        p = sc.plan

        def pro(s_int):
            p.t_dev.fill_(3)
            L.check(lib.dp_add_noise(sc.clean.data_ptr(), sc.noise.data_ptr(), p.t_dev.data_ptr(), sc.acp.data_ptr(),
                                     p.x_in.ptr, sc.B, sc.C, sc.H, sc.W, 1, p.x_in.ld, s_int))

        def mid(s_int):
            gy = p.gradof(p.y_out)
            L.check(lib.dp_mse_loss_grad(p.y_out.ptr, sc.noise_nhwc.data_ptr(), gy.ptr, sc.n, sc.loss_scale, sc.grad_scale,
                                         sc.partial.data_ptr(), sc.loss.data_ptr(), s_int))
        conv_s, n_conv, conv_by_tag, conv_by_layer = timed_conv_launches(p, pro, mid)
        other_ms = timed_conv_launches.last_other_ms
    else:
        conv_s, n_conv, conv_by_tag, conv_by_layer = 1.0, 0, {}, {}
    sampling = None
    if c["model"].startswith("ldm:") and rank == 0:
        # the other half of prune_ldm.py's step (prune_ldm.py:111-118): class-conditional DDIM-20 sampling with classifier-free guidance =
        # 2 x 20 UNet forwards per batch of latents; forward-only launch plan, CUDA-graph replay
        from diff_pruning_b200.engine import frozen_weights, get_plan
        kw = extra(B, dev)
        with torch.no_grad(), frozen_weights(model):
            fplan = get_plan(model, B, hw, hw, dev, need_grad=False)
            fplan.ensure_packed(force=True)
            fplan.load_context(kw["context"])
            fplan.load_input_nchw(clean.to(dev), torch.full((B,), 500, device=dev, dtype=torch.long))
            fplan.run_forward(); torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                fplan.run_forward()
            for _ in range(3):
                g.replay()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s0.record()
            for _ in range(20):
                g.replay()
            s1.record(); torch.cuda.synchronize(dev)
            fms = s0.elapsed_time(s1) / 20
        sampling = {"unet_forward_ms": fms, "latents_per_forward": B, "ddim20_cfg_batches_per_s": 1e3 / (40 * fms),
                    "note": "forward-only UNet step (no-grad plan, CUDA graph); a DDIM-20 sample with classifier-free guidance costs 40 of them (prune_ldm.py:111-118)"}
        del fplan, g
    plan_B, plan_macs, plan_bytes = sc.plan.B, sc.plan.conv_macs, sc.plan.bytes_allocated()
    plan_lin_macs = getattr(sc.plan, "lin_macs", 0)
    del sc
    if hasattr(model, "_dpb200_plans"):
        model._dpb200_plans.clear()
    del model
    torch.cuda.empty_cache()
    finetune_leg = finetune_bf16 = None
    if not args.no_finetune and not c["model"].startswith("ldm:"):      # the reference's LDM path is prune_ldm.py only (no finetune script in scope)
        finetune_leg = finetune_bench(args, rank, world, dev, barrier)
        from diff_pruning_b200 import engine as _eng
        if getattr(_eng, "BF16_TIER", False):
            finetune_bf16 = finetune_bench(args, rank, world, dev, barrier, compute="bf16")
    config3 = None
    if args.config == "c1" and not args.no_c3:
        config3 = secondary_scoring_leg("c3", args, rank, world, dev, barrier)
    if rank != 0:
        return
    hbm, tf_sus, tf_burst, which = peaks()
    flops = plan_B * c["conv_flop"]
    achieved = flops / conv_s / 1e12
    tc = bool(lib.dp_tc_available())
    tf32 = measure_tf32_peak(dev)
    traffic = None
    tp = os.path.join(ROOT, "profiles", "r02_conv_traffic.json" if os.path.exists(os.path.join(ROOT, "profiles", "r02_conv_traffic.json"))
                      else "r01_conv_traffic.json")
    if os.path.exists(tp) and B == 128 and args.config == "c1":   # dram__bytes_read+write summed over the conv launches of one pass (committed ncu capture)
        tj = json.load(open(tp))
        traffic = tj["dram_read_bytes"] + tj["dram_write_bytes"]
    tier_ceiling = tf_sus / 3.0      # 3 kind::f16 tensor instructions per product (fp16 runs at the bf16 rate MEASURED_PEAKS.json holds)
    roofline = {"bound": "tensor", "achieved": achieved, "peak": tf_sus, "unit": "TFLOP/s", "frac": achieved / tf_sus,
                "traffic": traffic, "breakdown_ms": conv_by_tag, "top_layers_ms": conv_by_layer,
                "other_launches_ms": other_ms, "tf32_peak_measured": tf32, "tier_ceiling_tflops": tier_ceiling, "frac_of_tier_ceiling": achieved / tier_ceiling,
                "plan_conv_gflop_per_image": 6.0 * plan_macs / plan_B / 1e9, "plan_linear_gflop_per_image": 6.0 * plan_lin_macs / plan_B / 1e9,
                "kernel": "conv implicit GEMM (fprop+dgrad+wgrad launches of one pass: %d)" % n_conv,
                "note": (f"algorithmic conv FLOPs/pass = {B} x {c['conv_flop'] / 1e9:.2f} GFLOP (SURVEY.md §8d) / summed conv-launch device time "
                         f"{conv_s * 1e3:.2f} ms of a {ms / args.steps:.2f} ms step; peak = bf16_tflops_sustained ({which}); "
                         "fp32-grade tier: " + ("tcgen05 kind::f16 on a 3-product fp16 hi/lo split of power-of-two-scaled operands (22 bits per operand, fp32 accumulation: "
                                                 "tier ceiling = peak / 3; tf32_peak_measured = cuBLAS TF32, the rate torch-eager's cuDNN default runs at)" if tc
                                                 else "CUDA-core FFMA (SIMT) — tensor path not active") +
                         "; traffic = DRAM bytes of all conv launches of one pass (committed ncu capture, C1 only)")}
    value = world * args.steps / (ms * 1e-3)
    e2e = world * args.steps / (ms_e2e * 1e-3)
    cpu = cpu_oracle_passes(args.config, B, min_seconds=12.0, max_passes=8) if args.gpus == 1 and not args.no_cpu else None
    eager = gpu_eager_passes(args.config, B, dev) if args.gpus == 1 and not args.no_cpu else None
    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{c['name']} Taylor pass, batch {B} x 3x{hw}x{hw} per GPU, "
                               f"timesteps sharded over {world} GPU(s), one grad all-reduce at the end",
                   "l2": f"per-pass working set (activations+grads, {plan_bytes / 2**30:.1f} GiB) >> 126 MB L2: inputs larger than L2, no explicit flush",
                   "cuda_graph": not args.no_graph, "imgs_per_s": value * B},
        "clocks": clocks, "gpu_launches": int(gpu_launches),
        "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(2 * clean.numel() * 4 + 8 * B), "d2h_bytes_per_step": 4,
                "ms_per_step": ms_e2e / args.steps},
        "roofline": roofline,
    }
    if cpu is not None:
        out["cpu_baseline"] = cpu
    if eager is not None:
        out["gpu_eager_baseline"] = eager
    if finetune_leg is not None:
        out["finetune"] = finetune_leg
    if finetune_bf16 is not None:
        out["finetune_bf16"] = finetune_bf16
    if config3 is not None:
        out["config3"] = config3
    if sampling is not None:
        out["sampling"] = sampling
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default=os.environ.get("DPB200_BENCH_CONFIG", "c1"), choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline and gpu_eager_baseline legs (profiling runs)")
    ap.add_argument("--profile-pass", action="store_true", help="run one eager pass inside cudaProfilerStart/Stop (ncu)")
    ap.add_argument("--no-finetune", action="store_true", help="skip the secondary finetune imgs/s legs")
    ap.add_argument("--no-c3", action="store_true", help="skip the secondary BASELINE-config-3 (LSUN-256) scoring leg of the default run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the last step's loss and a fixed sample of the accumulated gradients as DIR/*.npy "
                         "(float32); the inputs depend on the arguments only, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the device path computed: use it with --impl ours")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.batch is None:
        args.batch = CONFIGS[args.config]["batch"]
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 1)
    rank, world, local_rank = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    run_ours(args, rank, world, local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
