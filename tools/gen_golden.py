#!/usr/bin/env python
"""Generate tests/golden/* by importing the UNMODIFIED reference (read-only /root/reference).

Run in the build container only (the reference does not exist on the GPU box):
    python tools/gen_golden.py [--skip-cfg1]
Outputs (all small, committed):
    tests/golden/tiny_unet.pt      TINY config: inputs, output, loss, all grads after 1 pass (B=2)
    tests/golden/blocks.pt         one ResnetBlock2D (with shortcut) and one Attention: in/out/grads
    tests/golden/cifar_fwd.pt      C1 seed-0: state-dict fingerprints, eps_hat for B=2 at t in {0,500,999},
                                   KAT losses at B=16 t in {0,50,99}, grad fingerprints after one pass
    tests/golden/cifar_cfg1.pt     BASELINE config 1 (B=16, t=0..99, ratio 0.3): per importance variant, the
                                   interactive group sequence (structure, importance vector, pruned indices),
                                   post-prune shapes / param+MAC counts / pruned-model eps
    tests/golden/cifar_cfg1_s3.pt  same with 3 timesteps (fast CPU check of the oracle)
    tests/golden/finetune_tiny.pt  2 finetune steps on TINY (Adam + clip + EMA), dropout 0
    tests/golden/ddim_tiny.pt      DDIMPipeline samples (uniform/eta 0/10 steps, quad/eta 0.5/7 steps) on TINY
    tests/golden/ddpm_prune_magnitude_tiny.json  what ddpm_prune.py, run unmodified on the compat names, printed and saved
"""
import argparse
import hashlib
import json
import os
import sys
import time

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
import ref_shim  # noqa: E402

diffusers, tp = ref_shim.install()
from diffusers import DDPMScheduler, UNet2DModel  # noqa: E402
from diffusers.models.attention_processor import Attention, AttnProcessor  # noqa: E402
from diffusers.models.resnet import Downsample2D, ResnetBlock2D, Upsample2D  # noqa: E402
from torch_pruning.pruner import function as tpf  # noqa: E402

import diff_pruning_b200 as dp  # noqa: E402  (configs only)

OUT = os.path.join(ROOT, "tests", "golden")
os.makedirs(OUT, exist_ok=True)


def legacy_attn(model):
    for m in model.modules():
        if isinstance(m, Attention):
            m.set_processor(AttnProcessor())


def fp(t):
    t = t.detach().double()
    return [float(t.sum()), float(t.abs().sum()), float((t * t).sum())]


def build(cfg, seed=0):
    torch.manual_seed(seed)
    m = UNet2DModel(**cfg).eval()
    legacy_attn(m)  # identical math to 2_0 pre-pruning, and the only one that survives pruning
    return m


def inputs(b, hw, c=3):
    g1, g2 = torch.Generator().manual_seed(1), torch.Generator().manual_seed(2)
    return torch.randn(b, c, hw, hw, generator=g1), torch.randn(b, c, hw, hw, generator=g2)


def gen_tiny():
    cfg = dict(dp.TINY_TEST_CONFIG)
    m = build(cfg)
    sched = DDPMScheduler(num_train_timesteps=1000)
    clean, noise = inputs(2, 16)
    t = torch.tensor([7, 7]).long()
    m.zero_grad()
    losses = []
    for tt in (7, 400):  # two accumulated passes (no zero_grad in between)
        t = (tt * torch.ones(2)).long()
        out = m(sched.add_noise(clean, noise, t), t).sample
        loss = torch.nn.functional.mse_loss(out, noise)
        loss.backward()
        losses.append(loss.item())
    with torch.no_grad():
        t2 = torch.tensor([3, 950]).long()  # per-sample timesteps (finetune style)
        out2 = m(sched.add_noise(clean, noise, t2), t2).sample
    torch.save({"cfg": cfg, "seed": 0, "losses": losses, "out_last": out.detach(), "t2": t2, "out_t2": out2,
                "grads": {k: p.grad.clone() for k, p in m.named_parameters()}},
               os.path.join(OUT, "tiny_unet.pt"))
    print("tiny", losses)


def gen_blocks():
    torch.manual_seed(3)
    rb = ResnetBlock2D(in_channels=32, out_channels=64, temb_channels=128, groups=8, eps=1e-6)
    x = torch.randn(2, 32, 8, 8, requires_grad=True)
    temb = torch.randn(2, 128, requires_grad=True)
    y = rb(x, temb)
    gy = torch.randn_like(y)
    y.backward(gy)
    res = {"sd": {k: v.clone() for k, v in rb.state_dict().items()}, "x": x.detach(), "temb": temb.detach(),
           "y": y.detach(), "gy": gy, "gx": x.grad.clone(), "gtemb": temb.grad.clone(),
           "grads": {k: p.grad.clone() for k, p in rb.named_parameters()}}
    torch.manual_seed(4)
    at = Attention(64, heads=1, dim_head=64, rescale_output_factor=1.0, eps=1e-6, norm_num_groups=8,
                   residual_connection=True, bias=True, upcast_softmax=True, _from_deprecated_attn_block=True)
    at.set_processor(AttnProcessor())
    xa = torch.randn(2, 64, 4, 4, requires_grad=True)
    ya = at(xa)
    gya = torch.randn_like(ya)
    ya.backward(gya)
    att = {"sd": {k: v.clone() for k, v in at.state_dict().items()}, "x": xa.detach(), "y": ya.detach(), "gy": gya,
           "gx": xa.grad.clone(), "grads": {k: p.grad.clone() for k, p in at.named_parameters()}, "scale": at.scale}
    torch.save({"resnet": res, "attn": att}, os.path.join(OUT, "blocks.pt"))
    print("blocks ok")


def cifar_cfg():
    cfg = json.load(open(os.path.join(ref_shim.REF, "tools", "ddpm_cifar10_config.json")))
    return {k: v for k, v in cfg.items() if not k.startswith("_")}


def gen_cifar_fwd():
    m = build(cifar_cfg())
    sched = DDPMScheduler(num_train_timesteps=1000)
    sd = m.state_dict()
    res = {"sd_fp": {k: fp(v) for k, v in sd.items()},
           "sd_sha": hashlib.sha256(b"".join(v.numpy().tobytes() for v in sd.values())).hexdigest(),
           "n_params": sum(p.numel() for p in m.parameters())}
    clean16, noise16 = inputs(16, 32)
    kat = {}
    with torch.no_grad():
        for tt in (0, 50, 99):
            t = (tt * torch.ones(16)).long()
            out = m(sched.add_noise(clean16, noise16, t), t).sample
            kat[tt] = torch.nn.functional.mse_loss(out, noise16).item()
    res["kat_losses_b16"] = kat
    clean, noise = clean16[:2].clone(), noise16[:2].clone()
    eps = {}
    with torch.no_grad():
        for tt in (0, 500, 999):
            t = (tt * torch.ones(2)).long()
            eps[tt] = m(sched.add_noise(clean, noise, t), t).sample.clone()
    res["eps_b2"] = eps
    m.zero_grad()
    t = (500 * torch.ones(2)).long()
    out = m(sched.add_noise(clean, noise, t), t).sample
    loss = torch.nn.functional.mse_loss(out, noise)
    loss.backward()
    res["loss_b2_t500"] = loss.item()
    res["grad_fp_b2_t500"] = {k: fp(p.grad) for k, p in m.named_parameters()}
    res["grad_samples_b2_t500"] = {k: p.grad.flatten()[:64].clone() for k, p in m.named_parameters()}
    torch.save(res, os.path.join(OUT, "cifar_fwd.pt"))
    print("cifar_fwd", kat, res["loss_b2_t500"])


KIND = {tpf.prune_conv_out_channels: "out", tpf.prune_linear_out_channels: "out",
        tpf.prune_conv_in_channels: "in", tpf.prune_linear_in_channels: "in",
        tpf.prune_groupnorm_out_channels: "gn"}


def describe_group(group, names):
    items = []
    for dep, idxs in group:
        layer = dep.target.module
        kind = KIND.get(dep.handler)
        if layer not in names or kind is None:
            continue  # non-parametric nodes (concat/split/elementwise) carry no score
        if kind == "gn" and not layer.affine:
            continue
        items.append((names[layer], kind, [int(i) for i in idxs]))
    return items


def compress(idxs):
    idxs = [int(i) for i in idxs]
    if idxs and idxs == list(range(idxs[0], idxs[0] + len(idxs))):
        return ("range", idxs[0], len(idxs))
    return idxs


def describe_group_c(group, names):
    return [(n, k, compress(i)) for n, k, i in describe_group(group, names)]


class VariantTaylor:
    """reference importance.py:375-434 with :393/:407 switched per variant (SURVEY.md §8(c)); :416 for GroupNorm."""

    def __init__(self, variant):
        self.variant = variant

    @torch.no_grad()
    def __call__(self, group, ch_groups=1):
        imps = []
        for dep, idxs in group:
            idxs.sort()
            layer, fn = dep.target.module, dep.handler
            if fn in (tpf.prune_conv_out_channels, tpf.prune_linear_out_channels):
                w, dw = layer.weight.data[idxs].flatten(1), layer.weight.grad.data[idxs].flatten(1)
            elif fn in (tpf.prune_conv_in_channels, tpf.prune_linear_in_channels):
                w = layer.weight.data.transpose(0, 1).flatten(1)[idxs]
                dw = layer.weight.grad.data.transpose(0, 1).flatten(1)[idxs]
            elif fn == tpf.prune_groupnorm_out_channels:
                if layer.affine:
                    imps.append((layer.weight.data[idxs] * layer.weight.grad.data[idxs]).abs())
                continue
            else:
                continue
            p = w * dw
            imps.append({"vendored": p.abs().pow(2).sum(1), "taylor": p.sum(1).abs(), "diff": p.abs().sum(1)}[self.variant])
        if not imps:
            return None
        size = len(imps[0])
        return torch.stack([i for i in imps if len(i) == size], 0).sum(0)


def gen_cfg1(n_steps=100, ratio=0.3, B=16, out_name="cifar_cfg1.pt", cfg=None, hw=32, timesteps=None, eps_stride=None):
    import copy
    os.chdir("/tmp")  # prune_local writes ./run/pruning_logs
    m0 = build(cifar_cfg() if cfg is None else cfg)
    sched = DDPMScheduler(num_train_timesteps=1000)
    clean, noise = inputs(B, hw)
    example = {"sample": torch.randn(1, 3, hw, hw), "timestep": torch.ones((1,)).long()}
    m0.zero_grad()
    m0.eval()
    losses, eps_sub = [], []
    t0 = time.time()
    timesteps = list(range(n_steps)) if timesteps is None else list(timesteps)
    cache = os.path.join("/tmp", out_name + ".passes")          # scratch cache of the (slow) passes while iterating on this script
    if os.path.exists(cache):
        c = torch.load(cache, weights_only=False)
        losses, eps_sub = c["losses"], c["eps_sub"]
        for k_, p_ in m0.named_parameters():
            p_.grad = c["grads"][k_]
        timesteps_run = []
    else:
        timesteps_run = timesteps
    for k in timesteps_run:
        t = (k * torch.ones(B)).long()
        out = m0(sched.add_noise(clean, noise, t), t).sample
        loss = torch.nn.functional.mse_loss(out, noise)
        loss.backward()
        losses.append(loss.item())
        if eps_stride:   # strided sample of eps_hat (the full tensor would be MBs per timestep)
            eps_sub.append(out.detach()[:, :, ::eps_stride, ::eps_stride].clone())
        if k % 10 == 0 or hw > 32:
            print(f"  {out_name} pass t={k} loss {losses[-1]:.7f} ({time.time() - t0:.0f}s)", flush=True)
    if hw > 32 and not os.path.exists(cache):
        torch.save({"losses": losses, "eps_sub": eps_sub, "grads": {k_: p_.grad for k_, p_ in m0.named_parameters()}}, cache)
    grad_fp = {k: fp(p.grad) for k, p in m0.named_parameters()}
    res = {"n_steps": len(timesteps), "timesteps": timesteps, "ratio": ratio, "B": B, "hw": hw, "losses": losses, "grad_fp": grad_fp,
           "variants": {}}
    if eps_stride:
        res["eps_stride"], res["eps_sub"] = eps_stride, eps_sub
    for variant in ("vendored", "taylor", "diff"):
        m = copy.deepcopy(m0)
        for (k, p), (_, q) in zip(m.named_parameters(), m0.named_parameters()):
            p.grad = q.grad.clone()
        legacy_attn(m)
        names = {mod: n for n, mod in m.named_modules()}
        # the pinned behaviour: the vendored TaylorImportance class for "vendored" (unmodified reference code),
        # the same class body with the product/abs placement switched for the two pip forms.
        imp = tp.importance.TaylorImportance() if variant == "vendored" else VariantTaylor(variant)
        pruner = tp.pruner.MagnitudePruner(m, example, importance=imp, iterative_steps=1, channel_groups={},
                                           ch_sparsity=ratio, ignored_layers=[m.conv_out])
        base_macs, base_params = tp.utils.count_ops_and_params(m, example)
        checker = VariantTaylor(variant)
        groups = []
        # Scores are evaluated INTERACTIVELY: later groups see layers already sliced by earlier groups
        # (ddpm_prune.py:108-109 + metapruner.py:205-254), so record each group right before it is pruned.
        for g in pruner.step(interactive=True):
            module, fn = g[0][0].target.module, g[0][0].handler
            cur = pruner.DG.get_out_channels(module)
            full = pruner.DG.get_pruning_group(module, fn, list(range(cur)))
            ch_groups = pruner.get_channel_groups(full)
            sc = checker(full, ch_groups=ch_groups)
            sc_ref = imp(full, ch_groups=ch_groups)
            assert torch.equal(sc, sc_ref), names[module]
            sel = [int(i) for i in g[0][1]]
            full_items = describe_group(full, names)
            pr_items = describe_group(g, names)
            # index mapping is positional: pruned idxs of every item == its full idxs at the selected positions
            # (same traversal => same item order; a layer may appear twice when both halves of a concat are in the group)
            # (a GroupNorm-coupled group whose per-GN-group quota n_pruned // 32 is 0 — every such group at ratio 0.05 — is yielded
            #  with an EMPTY selection and prunes nothing: metapruner.py:237-246)
            assert len(full_items) == len(pr_items) or not sel
            for (n, k, i), (n2, k2, fi) in zip(pr_items if sel else [], full_items):
                # a layer fed by BOTH halves of a concat owned by this group appears once with the two index lists
                # merged (len = parts * channels); such items are skipped by the importance (:422-426) but pruned.
                parts = len(fi) // cur
                assert (n, k) == (n2, k2) and len(fi) == parts * cur, (n, k)
                assert sorted(i) == sorted(fi[q * cur + j] for q in range(parts) for j in sel), (n, k)
            n_pruned = cur - int(pruner.layer_init_out_ch[module] * (1 - pruner.get_target_sparsity(module)))
            groups.append({"root": names[module], "root_kind": KIND[fn], "ch_groups": int(ch_groups), "channels": int(cur),
                           "n_pruned": int(n_pruned), "items": [(n, k, compress(i)) for n, k, i in full_items],
                           "imp": sc.clone(), "idxs": sel})
            g.prune()
        for mod in m.modules():
            if isinstance(mod, (Upsample2D, Downsample2D)):
                mod.channels = mod.conv.in_channels
        macs, params = tp.utils.count_ops_and_params(m, example)
        shapes = {k: list(v.shape) for k, v in m.state_dict().items()}
        with torch.no_grad():  # pruned-model forward (legacy attention, stale scale)
            t = (10 * torch.ones(2)).long()
            out = m(sched.add_noise(clean[:2], noise[:2], t), t).sample
        res["variants"][variant] = {"groups": groups, "base": [base_macs, base_params], "pruned": [macs, params],
                                    "pruned_shapes": shapes,
                                    "pruned_eps_b2_t10": (out[:, :, ::eps_stride, ::eps_stride] if eps_stride else out).clone()}
        print("cfg1", variant, base_params, params, macs, len(groups), sum(len(g["idxs"]) for g in groups), flush=True)
    torch.save(res, os.path.join(OUT, out_name))


def gen_cfg1_s3():
    gen_cfg1(n_steps=3, out_name="cifar_cfg1_s3.pt")


def gen_cfg3_s3():
    """BASELINE config 3 (google/ddpm-ema-bedroom-256 architecture, README.md:140-148: --batch_size 4 --pruning_ratio 0.05) with 3 of
    the 1000 timesteps (t = 0, 500, 999): losses, a strided sample of eps_hat, gradient fingerprints and the interactive prune
    sequence (scores + selected channels) for all three importance variants.  ~2 CPU-minutes for the passes."""
    gen_cfg1(ratio=0.05, B=4, out_name="lsun_cfg3_s3.pt", cfg=dict(dp.LSUN256_DDPM_CONFIG), hw=256, timesteps=(0, 500, 999),
             eps_stride=4)


def gen_finetune():
    cfg = dict(dp.TINY_TEST_CONFIG)
    m = build(cfg).train()
    sched = DDPMScheduler(num_train_timesteps=1000)
    opt = torch.optim.Adam(m.parameters(), lr=2e-4, betas=(0.9, 0.999), weight_decay=0.0, eps=1e-8)
    from diffusers.training_utils import EMAModel
    ema = EMAModel(m.parameters(), decay=0.9999, use_ema_warmup=True, inv_gamma=1.0, power=0.75,
                   model_cls=UNet2DModel, model_config=m.config)
    g = torch.Generator().manual_seed(5)
    rec = {"cfg": cfg, "steps": []}
    for step in range(2):
        clean = torch.randn(4, 3, 16, 16, generator=g)
        noise = torch.randn(4, 3, 16, 16, generator=g)
        t = torch.randint(0, 1000, (4 // 2 + 1,), generator=g)
        t = torch.cat([t, 1000 - t - 1], dim=0)[:4]
        noisy = sched.add_noise(clean, noise, t)
        opt.zero_grad()
        out = m(noisy, t).sample
        loss = (noise - out).square().sum(dim=(1, 2, 3)).mean(dim=0)
        loss.backward()
        gn = torch.nn.utils.clip_grad_norm_(m.parameters(), 1.0)
        opt.step()
        ema.step(m.parameters())
        rec["steps"].append({"clean": clean, "noise": noise, "t": t, "loss": loss.item(), "grad_norm": gn.item()})
    rec["params"] = {k: p.detach().clone() for k, p in m.named_parameters()}
    rec["ema"] = {k: s.clone() for (k, _), s in zip(m.named_parameters(), ema.shadow_params)}
    torch.save(rec, os.path.join(OUT, "finetune_tiny.pt"))
    print("finetune", [s["loss"] for s in rec["steps"]], [s["grad_norm"] for s in rec["steps"]])


def gen_ddim():
    """DDIMPipeline (pipeline_ddim.py:45-122) + the reference's modified DDIMScheduler on the TINY UNet, CPU generator."""
    from diffusers import DDIMPipeline
    cfg = dict(dp.TINY_TEST_CONFIG)
    m = build(cfg)
    res = {"cfg": cfg}
    for name, skip, eta, steps in (("uniform_eta0", "uniform", 0.0, 10), ("quad_eta05", "quad", 0.5, 7)):
        pipe = DDIMPipeline(unet=m, scheduler=DDPMScheduler(num_train_timesteps=1000))
        pipe.scheduler.skip_type = skip
        pipe.set_progress_bar_config(disable=True)
        g = torch.Generator().manual_seed(0)
        out = pipe(batch_size=2, generator=g, eta=eta, num_inference_steps=steps, output_type="numpy").images
        res[name] = {"skip_type": skip, "eta": eta, "steps": steps, "images": torch.from_numpy(out),
                     "timesteps": pipe.scheduler.timesteps.clone()}
    torch.save(res, os.path.join(OUT, "ddim_tiny.pt"))
    print("ddim", {k: float(v["images"].mean()) for k, v in res.items() if k != "cfg"})


def gen_ckpt():
    """`DDPMPipeline.save_pretrained` of the reference's vendored diffusers (pipeline_utils.py:485-560, modeling_utils.py:250-330,
    configuration_utils.py:138-170) on the TINY UNet: keeps the three JSON files (the weights are the seeded tiny UNet, whose
    state-dict keys/shapes are pinned elsewhere) as tests/golden/ckpt_tiny_ref/, plus a digest of the state-dict it wrote."""
    import hashlib
    import shutil
    import tempfile
    from diffusers import DDPMPipeline
    m = build(dict(dp.TINY_TEST_CONFIG))
    pipe = DDPMPipeline(unet=m, scheduler=DDPMScheduler(num_train_timesteps=1000))
    tmp = tempfile.mkdtemp()
    pipe.save_pretrained(tmp)
    dst = os.path.join(OUT, "ckpt_tiny_ref")
    for rel in ("model_index.json", "unet/config.json", "scheduler/scheduler_config.json"):
        os.makedirs(os.path.dirname(os.path.join(dst, rel)), exist_ok=True)
        shutil.copy(os.path.join(tmp, rel), os.path.join(dst, rel))
    sd = torch.load(os.path.join(tmp, "unet", "diffusion_pytorch_model.bin"), map_location="cpu")
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode()); h.update(v.contiguous().numpy().tobytes())
    json.dump({"files": sorted(os.listdir(os.path.join(tmp, "unet"))), "n_tensors": len(sd), "state_dict_sha256": h.hexdigest()},
              open(os.path.join(dst, "weights_digest.json"), "w"), indent=1)
    shutil.rmtree(tmp)
    print("ckpt", len(sd), h.hexdigest()[:16])


def gen_lr():
    """diffusers.optimization.get_scheduler (optimization.py:282-340) sampled at a few optimiser steps: multipliers of the base lr."""
    from diffusers.optimization import get_scheduler
    out = {}
    for name in ("constant", "constant_with_warmup", "linear", "cosine"):
        for warm, total in ((0, 100), (5, 100), (500, 10000)):
            steps = sorted({0, 1, 2, warm - 1, warm, warm + 1, total // 2, total - 1, total, total + 3} - {-1})
            prm = torch.nn.Parameter(torch.zeros(1))
            opt = torch.optim.SGD([prm], lr=1.0)
            sch = get_scheduler(name, opt, num_warmup_steps=warm, num_training_steps=total)
            vals, k = {}, 0
            for s in range(max(steps) + 1):
                if s in steps:
                    vals[str(s)] = sch.get_last_lr()[0]
                opt.step(); sch.step()
            out[f"{name}|{warm}|{total}"] = vals
    json.dump(out, open(os.path.join(OUT, "lr_schedules.json"), "w"), indent=1)
    print("lr", len(out))


def gen_lsun_struct(ratio=0.05):
    """The six-level LSUN-256 architecture (google/ddpm-ema-bedroom-256: BASELINE config 3, ratio 0.05) at reduced widths
    (32, 32, 64, 64, 128, 128), `--pruner magnitude` (ddpm_prune.py:70-71: tp.importance.MagnitudeImportance()) through the
    interactive prune sequence: pins the structural group derivation, ch_groups, the per-group magnitude scores and the selected
    channel indices for the second headline architecture.  No gradients needed."""
    cfg = dict(dp.LSUN256_DDPM_CONFIG, block_out_channels=(32, 32, 64, 64, 128, 128))
    m = build(cfg)
    example = {"sample": torch.randn(1, 3, 64, 64), "timestep": torch.ones((1,)).long()}
    names = {mod: n for n, mod in m.named_modules()}
    imp = tp.importance.MagnitudeImportance()
    pruner = tp.pruner.MagnitudePruner(m, example, importance=imp, iterative_steps=1, channel_groups={}, ch_sparsity=ratio,
                                       ignored_layers=[m.conv_out])
    base_macs, base_params = tp.utils.count_ops_and_params(m, example)
    groups = []
    for g in pruner.step(interactive=True):
        module, fn = g[0][0].target.module, g[0][0].handler
        cur = pruner.DG.get_out_channels(module)
        full = pruner.DG.get_pruning_group(module, fn, list(range(cur)))
        ch_groups = pruner.get_channel_groups(full)
        sc = imp(full, ch_groups=ch_groups)
        groups.append({"root": names[module], "root_kind": KIND[fn], "ch_groups": int(ch_groups), "channels": int(cur),
                       "items": [(n, k, compress(i)) for n, k, i in describe_group(full, names)],
                       "imp": sc.clone(), "idxs": [int(i) for i in g[0][1]]})
        g.prune()
    for mod in m.modules():
        if isinstance(mod, (Upsample2D, Downsample2D)):
            mod.channels = mod.conv.in_channels
    macs, params = tp.utils.count_ops_and_params(m, example)
    res = {"cfg": cfg, "ratio": ratio, "groups": groups, "base": [base_macs, base_params], "pruned": [macs, params],
           "pruned_shapes": {k: list(v.shape) for k, v in m.state_dict().items()}}
    torch.save(res, os.path.join(OUT, "lsun_struct_magnitude.pt"))
    print("lsun_struct", len(groups), base_params, params, base_macs, macs)


def gen_exp_importance():
    """The ddpm_exp importance criteria (ddpm_exp/torch_pruning/importance.py:438-548 FullTaylor order 1/2, :553-670 AbsTaylor,
    :672-781 Fisher) evaluated by the UNMODIFIED vendored classes on every pruning group of the TINY UNet after two accumulated passes."""
    os.chdir("/tmp")
    cfg = dict(dp.TINY_TEST_CONFIG)
    m = build(cfg)
    sched = DDPMScheduler(num_train_timesteps=1000)
    clean, noise = inputs(2, 16)
    m.zero_grad()
    for tt in (7, 400):
        t = (tt * torch.ones(2)).long()
        torch.nn.functional.mse_loss(m(sched.add_noise(clean, noise, t), t).sample, noise).backward()
    example = {"sample": torch.randn(1, 3, 16, 16), "timestep": torch.ones((1,)).long()}
    pruner = tp.pruner.MagnitudePruner(m, example, importance=tp.importance.MagnitudeImportance(), iterative_steps=1, channel_groups={},
                                       ch_sparsity=0.3, ignored_layers=[m.conv_out])
    names = {mod: n for n, mod in m.named_modules()}
    crits = {"full1": tp.importance.FullTaylorImportance(order=1), "full2": tp.importance.FullTaylorImportance(order=2),
             "abs": tp.importance.AbsTaylorImportance(), "fisher": tp.importance.FisherImportance()}
    groups = []
    for g in pruner.DG.get_all_groups(ignored_layers=pruner.ignored_layers, root_module_types=pruner.root_module_types):
        items = describe_group_c(g, names)
        groups.append({"root": names[g[0][0].target.module], "items": items,
                       "imp": {k: c(g).clone() for k, c in crits.items()}})
    torch.save({"cfg": cfg, "groups": groups}, os.path.join(OUT, "exp_importance_tiny.pt"))
    print("exp_importance", len(groups), os.path.getsize(os.path.join(OUT, "exp_importance_tiny.pt")))


def gen_ldm_tiny():
    """The latent-diffusion UNetModel (BASELINE configs[4]) from the UNMODIFIED reference modules
    (ldm_exp/ldm/modules/diffusionmodules/openaimodel.py + ldm_exp/ldm/modules/attention.py; omegaconf is stubbed, openaimodel.py:476):
    a small member of the cin256-v2 family whose zero-initialised convolutions are re-drawn (a random-init network otherwise outputs 0
    and back-propagates nothing into most layers): state-dict keys, eps_hat, loss and all gradients after two accumulated Taylor passes
    (q_sample with the LDM sqrt-linear schedule, mse loss — what `get_loss_at_t` returns, ddpm.py:881-889,1022-1056); plus the parameter
    count of the full cin256-v2 network."""
    import types
    sys.path.insert(0, os.path.join(ref_shim.REF, "ldm_exp"))
    oc, lc = types.ModuleType("omegaconf"), types.ModuleType("omegaconf.listconfig")
    lc.ListConfig = type("ListConfig", (list,), {})
    oc.listconfig = lc
    sys.modules.setdefault("omegaconf", oc)
    sys.modules.setdefault("omegaconf.listconfig", lc)
    from ldm.modules.diffusionmodules.openaimodel import UNetModel as RefUNet
    from diff_pruning_b200 import ldm as L
    cfg = dict(L.LDM_TINY_CONFIG)
    torch.manual_seed(0)
    m = RefUNet(**cfg).eval()
    g = torch.Generator().manual_seed(5)
    redrawn = []
    for k, p in m.named_parameters():
        if float(p.detach().abs().sum()) == 0 and p.dim() > 1:
            p.data.copy_(torch.randn(p.shape, generator=g) * 0.05)
            redrawn.append(k)
    betas = torch.linspace(0.0015 ** 0.5, 0.0195 ** 0.5, 1000, dtype=torch.float64) ** 2
    ac = torch.cumprod(1.0 - betas, dim=0).to(torch.float32)
    clean, noise = inputs(2, 16)
    ctx = torch.randn(2, 1, cfg["context_dim"], generator=g)
    m.zero_grad()
    losses = []
    for tt in (7, 400):
        t = (tt * torch.ones(2)).long()
        xt = (ac[t] ** 0.5).reshape(-1, 1, 1, 1) * clean + ((1 - ac[t]) ** 0.5).reshape(-1, 1, 1, 1) * noise
        out = m(xt, t, context=ctx)
        loss = torch.nn.functional.mse_loss(out, noise)
        loss.backward()
        losses.append(loss.item())
    torch.manual_seed(0)
    n_full = sum(p.numel() for p in RefUNet(**L.CIN256_V2_CONFIG).parameters())
    import hashlib
    sha = hashlib.sha256(b"".join(v.detach().numpy().tobytes() for v in m.state_dict().values())).hexdigest()
    # weights are reproducible (seed 0 construction + the redraw loop above with Generator(5), context drawn right after): only their digest is stored
    torch.save({"cfg": cfg, "redrawn": redrawn, "sd_keys": list(m.state_dict().keys()), "sd_sha": sha, "context": ctx, "losses": losses,
                "out_last": out.detach(), "grads": {k: p.grad.clone() for k, p in m.named_parameters()}, "alphas_cumprod_fp": fp(ac),
                "cin256_v2_params": n_full}, os.path.join(OUT, "ldm_tiny.pt"))
    print("ldm_tiny", losses, n_full, len(redrawn), os.path.getsize(os.path.join(OUT, "ldm_tiny.pt")))


def gen_ref_pickle():
    """A whole-module pickle exactly as the reference writes it (`torch.save(model)`, ddpm_prune.py:135) for a small member of the
    family after a `--pruner magnitude` prune at ratio 0.3 — default AttnProcessor2_0 objects, FrozenDict config and all — plus eps_hat
    of that network (legacy processor, the only one that runs on pruned widths).  Pins `torch.load(pruned_ckpt)` at ddpm_train.py:292
    / ddpm_sample.py:27 against this package's classes."""
    os.chdir("/tmp")
    cfg = dict(dp.TINY_TEST_CONFIG, block_out_channels=(16, 32))
    torch.manual_seed(0)
    m = UNet2DModel(**cfg).eval()
    example = {"sample": torch.randn(1, 3, 16, 16), "timestep": torch.ones((1,)).long()}
    pruner = tp.pruner.MagnitudePruner(m, example, importance=tp.importance.MagnitudeImportance(), iterative_steps=1,
                                       channel_groups={}, ch_sparsity=0.3, ignored_layers=[m.conv_out])
    for g in pruner.step(interactive=True):
        g.prune()
    for mod in m.modules():
        if isinstance(mod, (Upsample2D, Downsample2D)):
            mod.channels = mod.conv.in_channels
    m.zero_grad()
    del pruner
    torch.save(m, os.path.join(OUT, "ref_pruned_small.pth"))
    legacy_attn(m)
    sched = DDPMScheduler(num_train_timesteps=1000)
    clean, noise = inputs(2, 16)
    t = torch.tensor([3, 950]).long()
    with torch.no_grad():
        out = m(sched.add_noise(clean, noise, t), t).sample
    torch.save({"cfg": cfg, "t": t, "eps": out, "shapes": {k: list(v.shape) for k, v in m.state_dict().items()},
                "scales": {n: float(a.scale) for n, a in m.named_modules() if isinstance(a, Attention)}},
               os.path.join(OUT, "ref_pruned_small_out.pt"))
    print("ref_pickle", os.path.getsize(os.path.join(OUT, "ref_pruned_small.pth")), sum(p.numel() for p in m.parameters()))


def gen_prune_script():
    """ddpm_prune.py run UNMODIFIED through tests/run_script_traced.py (compat/ first on sys.path, trace mode) as `--pruner magnitude
    --pruning_ratio 0.3 --device cpu` on a saved seed-0 TINY pipeline.  Without a GPU the script stops at its hard-coded
    `pipeline.to("cuda")` (ddpm_prune.py:144), after everything kept here: the #Params / #MACS lines it printed, the files it saved,
    their JSON configs, and the shapes and digest of its whole-module pickle of the pruned UNet."""
    import shutil
    import subprocess
    import tempfile
    tmp = tempfile.mkdtemp()
    src, dst = os.path.join(tmp, "tiny_cifar_pipeline"), os.path.join(tmp, "pruned")     # "cifar" in the path: 32x32 example inputs
    torch.manual_seed(0)
    dp.DDPMPipeline(unet=dp.UNet2DModel(**dp.TINY_TEST_CONFIG), scheduler=dp.DDPMScheduler(num_train_timesteps=1000)).save_pretrained(src)
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(ROOT, "diff-pruning_b200", "compat"), ROOT]))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "run_script_traced.py"), os.path.join(ref_shim.REF, "ddpm_prune.py"),
                        "--model_path", src, "--save_path", dst, "--pruner", "magnitude", "--pruning_ratio", "0.3", "--device", "cpu",
                        "--batch_size", "2"], cwd=ROOT, env=env, capture_output=True, text=True)
    assert r.returncode == 0 or "cuda" in r.stderr.lower(), r.stderr[-2000:]
    printed = [l for l in r.stdout.splitlines() if l.startswith(("#Params", "#MACS"))]
    files = sorted(os.path.relpath(os.path.join(d, f), dst) for d, _, fs in os.walk(dst) for f in fs)
    describe = ("import hashlib, json, sys, torch, diffusers\nm = torch.load(sys.argv[1], map_location='cpu')\nh = hashlib.sha256()\n"
                "for k, v in m.state_dict().items():\n    h.update(k.encode()); h.update(v.contiguous().numpy().tobytes())\n"
                "print(json.dumps({'class': type(m).__name__, 'shapes': {k: list(v.shape) for k, v in m.state_dict().items()}, "
                "'state_dict_sha256': h.hexdigest()}))")
    pickle = json.loads(subprocess.run([sys.executable, "-c", describe, os.path.join(dst, "pruned", "unet_pruned.pth")], env=env,
                                       capture_output=True, text=True, check=True).stdout)
    json.dump({"printed": printed, "files": files, "configs": {f: json.load(open(os.path.join(dst, f))) for f in files if f.endswith(".json")},
               "pruned_pickle": pickle}, open(os.path.join(OUT, "ddpm_prune_magnitude_tiny.json"), "w"), indent=1)
    shutil.rmtree(tmp)
    print("prune_script", printed, len(files), pickle["state_dict_sha256"][:16])


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--skip-cfg1", action="store_true")
    ap.add_argument("--only", default=None)
    a = ap.parse_args()
    torch.set_num_threads(8)     # tests/test_oracle_golden.py GOLDEN_THREADS: the oracle re-sums in the same order
    jobs = {"prune_script": gen_prune_script, "ldm_tiny": gen_ldm_tiny, "exp_importance": gen_exp_importance, "ref_pickle": gen_ref_pickle, "lsun_struct": gen_lsun_struct, "lr": gen_lr, "ckpt": gen_ckpt, "ddim": gen_ddim, "tiny": gen_tiny, "blocks": gen_blocks, "finetune": gen_finetune, "cifar_fwd": gen_cifar_fwd,
            "cfg1_s3": gen_cfg1_s3, "cfg3_s3": gen_cfg3_s3, "cfg1": gen_cfg1}
    for name, fn in jobs.items():
        if a.only and name != a.only:
            continue
        if name.startswith("cfg") and a.skip_cfg1:
            continue
        fn()
