"""Pin the oracle (oracle/unet_oracle.py) against fixtures generated from the unmodified reference
(tools/gen_golden.py).  CPU only."""
import copy

import pytest
import torch

from conftest import expand, load_golden, max_rel, rel_err
import diff_pruning_b200 as dp
from oracle import unet_oracle as orc

# tools/gen_golden.py runs with this many intra-op threads.  The CPU's fp32 reductions (convolution weight gradients, GEMMs) split
# their sums by thread, and the gradients that are zero in exact arithmetic (conftest.worst_grad_err) hold nothing but that rounding:
# they match the fixtures only when the oracle sums in the same order.
GOLDEN_THREADS = 8


@pytest.fixture(autouse=True)
def golden_thread_count():
    n = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_THREADS)
    yield
    torch.set_num_threads(n)


def seeded_sd(cfg, seed=0):
    torch.manual_seed(seed)
    m = dp.UNet2DModel(**cfg)
    return {k: v.detach().clone() for k, v in m.state_dict().items()}


def inputs(b, hw):
    g1, g2 = torch.Generator().manual_seed(1), torch.Generator().manual_seed(2)
    return torch.randn(b, 3, hw, hw, generator=g1), torch.randn(b, 3, hw, hw, generator=g2)


def test_tiny_unet_two_accumulated_passes():
    G = load_golden("tiny_unet.pt")
    cfg = G["cfg"]
    sd = {k: v.requires_grad_(True) for k, v in seeded_sd(cfg).items()}
    ac = orc.alphas_cumprod()
    clean, noise = inputs(2, 16)
    losses = []
    for tt in (7, 400):
        t = (tt * torch.ones(2)).long()
        losses.append(orc.taylor_pass(sd, cfg, ac, clean, noise, t).item())
    assert losses == pytest.approx(G["losses"], rel=1e-6)
    for k, g in G["grads"].items():
        if not k.endswith("to_k.bias"):   # identically-zero gradient, see conftest.worst_grad_err
            assert rel_err(sd[k].grad, g) < 2e-5, k
    with torch.no_grad():
        out2 = orc.unet_forward(sd, cfg, orc.add_noise(ac, clean, noise, G["t2"]), G["t2"])
    assert max_rel(out2, G["out_t2"]) < 1e-6


def test_blocks():
    G = load_golden("blocks.pt")
    r = G["resnet"]
    sd = {"b." + k: v.clone().requires_grad_(True) for k, v in r["sd"].items()}
    x, temb = r["x"].clone().requires_grad_(True), r["temb"].clone().requires_grad_(True)
    y = orc.resnet_block(sd, "b", x, temb, groups=8, eps=1e-6)
    assert max_rel(y, r["y"]) < 1e-6
    y.backward(r["gy"])
    assert rel_err(x.grad, r["gx"]) < 1e-5 and rel_err(temb.grad, r["gtemb"]) < 1e-5
    for k, g in r["grads"].items():
        assert rel_err(sd["b." + k].grad, g) < 1e-5, k
    a = G["attn"]
    sd = {"a." + k: v.clone().requires_grad_(True) for k, v in a["sd"].items()}
    xa = a["x"].clone().requires_grad_(True)
    ya = orc.attention_block(sd, "a", xa, groups=8, eps=1e-6, scale=a["scale"])
    assert max_rel(ya, a["y"]) < 1e-6
    ya.backward(a["gy"])
    assert rel_err(xa.grad, a["gx"]) < 1e-5
    for k, g in a["grads"].items():
        assert rel_err(sd["a." + k].grad, g) < 1e-5, k


def test_cifar_state_dict_and_eps():
    G = load_golden("cifar_fwd.pt")
    cfg = dp.CIFAR10_DDPM_CONFIG
    sd = seeded_sd(cfg)
    assert sum(v.numel() for v in sd.values()) == G["n_params"] == 35746307
    for k, f in G["sd_fp"].items():
        v = sd[k].double()
        assert [float(v.sum()), float(v.abs().sum()), float((v * v).sum())] == pytest.approx(f, rel=1e-12, abs=1e-12), k
    ac = orc.alphas_cumprod()
    clean16, noise16 = inputs(16, 32)
    clean, noise = clean16[:2], noise16[:2]
    with torch.no_grad():
        for tt, ref in G["eps_b2"].items():
            t = (tt * torch.ones(2)).long()
            assert max_rel(orc.unet_forward(sd, cfg, orc.add_noise(ac, clean, noise, t), t), ref) < 1e-5, tt
        t = (50 * torch.ones(16)).long()
        out = orc.unet_forward(sd, cfg, orc.add_noise(ac, clean16, noise16, t), t)
        assert torch.nn.functional.mse_loss(out, noise16).item() == pytest.approx(G["kat_losses_b16"][50], rel=2e-6)
        assert G["kat_losses_b16"][50] == pytest.approx(1.1101333, rel=1e-6)   # SURVEY.md §8(d) KAT


def test_cifar_one_pass_grads():
    G = load_golden("cifar_fwd.pt")
    cfg = dp.CIFAR10_DDPM_CONFIG
    sd = {k: v.requires_grad_(True) for k, v in seeded_sd(cfg).items()}
    ac = orc.alphas_cumprod()
    clean16, noise16 = inputs(16, 32)
    t = (500 * torch.ones(2)).long()
    loss = orc.taylor_pass(sd, cfg, ac, clean16[:2], noise16[:2], t)
    assert loss.item() == pytest.approx(G["loss_b2_t500"], rel=2e-6)
    for k, s in G["grad_samples_b2_t500"].items():
        assert rel_err(sd[k].grad.flatten()[:64], s) < 1e-3 or float((sd[k].grad.flatten()[:64] - s).abs().max()) < 1e-7, k
    for k, f in G["grad_fp_b2_t500"].items():
        g = sd[k].grad.double()
        assert float((g * g).sum()) == pytest.approx(f[2], rel=1e-3), k


def test_finetune_two_steps():
    G = load_golden("finetune_tiny.pt")
    cfg = G["cfg"]
    params = {k: v.requires_grad_(True) for k, v in seeded_sd(cfg).items()}
    ema = {k: v.detach().clone() for k, v in params.items()}
    opt = torch.optim.Adam(list(params.values()), lr=2e-4, betas=(0.9, 0.999), weight_decay=0.0, eps=1e-8)
    ac = orc.alphas_cumprod()
    for st in G["steps"]:
        loss, gn = orc.finetune_step(params, cfg, ac, st["clean"], st["noise"], st["t"], opt, ema)
        assert loss.item() == pytest.approx(st["loss"], rel=1e-5)
        assert gn.item() == pytest.approx(st["grad_norm"], rel=1e-4)
    for k in params:
        assert rel_err(params[k], G["params"][k]) < 1e-6, k
        assert rel_err(ema[k], G["ema"][k]) < 1e-6, k


def _replay_variant(V, weights, grads, variant, check_imp_rtol):
    """Re-run the interactive group sequence with the oracle's scoring + selection on (weights, grads) dicts;
    slices tensors like the reference's pruners (function.py) so later groups see earlier pruning."""
    n_flip = 0
    for g in V["groups"]:
        items = [(n, k, expand(i)) for n, k, i in g["items"]]
        imp = orc.group_importance(items, weights, grads, variant)
        assert imp.shape == g["imp"].shape
        assert rel_err(imp, g["imp"]) < check_imp_rtol, g["root"]
        sel = orc.select_pruning_idxs(imp, g["ch_groups"], g["n_pruned"])
        if sorted(sel) != sorted(g["idxs"]):
            n_flip += 1
        for n, k, idx in items:   # apply the GOLDEN selection so the sequence stays aligned
            parts = len(idx) // g["channels"]   # merged concat halves: positional mapping per part
            drop = sorted(idx[q * g["channels"] + j] for q in range(parts) for j in g["idxs"])
            for store in (weights, grads):
                w = store[n + ".weight"]
                if k == "in":
                    keep = [c for c in range(w.shape[1]) if c not in set(drop)]
                    store[n + ".weight"] = w[:, keep].contiguous()
                else:
                    keep = [c for c in range(w.shape[0]) if c not in set(drop)]
                    store[n + ".weight"] = w[keep].contiguous()
                    if k in ("out", "gn") and (n + ".bias") in store and store[n + ".bias"] is not None:
                        store[n + ".bias"] = store[n + ".bias"][keep].contiguous()
    return n_flip


def test_cfg1_three_steps_scores_and_masks():
    """BASELINE config 1 with 3 timesteps: oracle grads -> interactive scores -> masks == reference, bit-exact."""
    G = load_golden("cifar_cfg1_s3.pt")
    cfg = dp.CIFAR10_DDPM_CONFIG
    sd = {k: v.requires_grad_(True) for k, v in seeded_sd(cfg).items()}
    ac = orc.alphas_cumprod()
    clean, noise = inputs(G["B"], 32)
    for k in range(G["n_steps"]):
        t = (k * torch.ones(G["B"])).long()
        assert orc.taylor_pass(sd, cfg, ac, clean, noise, t).item() == pytest.approx(G["losses"][k], rel=2e-6)
    for variant, V in G["variants"].items():
        weights = {k: v.detach().clone() for k, v in sd.items()}
        grads = {k: v.grad.detach().clone() for k, v in sd.items()}
        assert _replay_variant(V, weights, grads, variant, 2e-4) == 0, variant
        assert {k: list(v.shape) for k, v in weights.items()} == V["pruned_shapes"], variant
        assert V["pruned"][1] == sum(v.numel() for v in weights.values())


def test_cfg1_published_counts():
    G = load_golden("cifar_cfg1.pt")
    V = G["variants"]["vendored"]
    assert round(V["base"][1] / 1e6, 3) == 35.746 and round(V["pruned"][1] / 1e6, 3) == 19.851   # assets/exp.png
    assert round(V["pruned"][0] / 1e9, 3) == 3.392
    assert len(V["groups"]) == 50 and sum(len(g["idxs"]) for g in V["groups"]) == 3164
    assert G["losses"][0] == pytest.approx(1.1193706, rel=1e-6) and G["losses"][99] == pytest.approx(1.1028205, rel=1e-6)


def test_exp_importance_variants_match_the_vendored_classes():
    """FullTaylor(order 1, 2) / AbsTaylor / Fisher (ddpm_exp/torch_pruning/importance.py:438-781): the oracle's item scores on the
    fixture's groups, with gradients re-derived by the oracle's own two accumulated passes."""
    from conftest import expand
    G = load_golden("exp_importance_tiny.pt")
    cfg = G["cfg"]
    torch.manual_seed(0)
    import diff_pruning_b200 as dp
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in dp.UNet2DModel(**cfg).state_dict().items()}
    g1, g2 = torch.Generator().manual_seed(1), torch.Generator().manual_seed(2)
    clean, noise = torch.randn(2, 3, 16, 16, generator=g1), torch.randn(2, 3, 16, 16, generator=g2)
    for tt in (7, 400):
        orc.taylor_pass(sd, cfg, orc.alphas_cumprod(), clean, noise, (tt * torch.ones(2)).long())
    w = {k: v.detach() for k, v in sd.items()}
    dw = {k: v.grad for k, v in sd.items()}
    assert len(G["groups"]) == 22
    for g in G["groups"]:
        items = [(n, k, expand(i)) for n, k, i in g["items"]]
        for variant in orc.EXP_VARIANTS:
            got = orc.group_importance(items, w, dw, variant)
            ref = g["imp"][variant]
            assert float((got - ref).abs().max()) <= 2e-4 * float(ref.abs().max()) + 1e-12, (g["root"], variant)


def fp(t):
    t = t.detach().double()
    return [float(t.sum()), float(t.abs().sum()), float((t * t).sum())]


def ldm_tiny_model(G):
    """Rebuild the fixture's weights: seed-0 construction, then the zero-initialised convolutions re-drawn exactly as tools/gen_golden.py did."""
    import hashlib
    from diff_pruning_b200 import ldm
    torch.manual_seed(0)
    m = ldm.UNetModel(**G["cfg"]).eval()
    g = torch.Generator().manual_seed(5)
    redrawn = []
    for k, p in m.named_parameters():
        if float(p.detach().abs().sum()) == 0 and p.dim() > 1:
            p.data.copy_(torch.randn(p.shape, generator=g) * 0.05)
            redrawn.append(k)
    ctx = torch.randn(2, 1, G["cfg"]["context_dim"], generator=g)
    assert redrawn == G["redrawn"] and list(m.state_dict().keys()) == G["sd_keys"]
    assert hashlib.sha256(b"".join(v.detach().numpy().tobytes() for v in m.state_dict().values())).hexdigest() == G["sd_sha"]
    assert torch.equal(ctx, G["context"])
    return m


def test_ldm_module_tree_and_oracle_match_the_reference():
    """BASELINE configs[4] (ldm_exp UNetModel): this package's module tree reproduces the reference's parameters bit for bit (state-dict
    keys + digest; 400 920 579 parameters for cin256-v2), and the LDM oracle reproduces the reference's loss / eps_hat / gradients of two
    accumulated Taylor passes (tests/golden/ldm_tiny.pt, generated from the unmodified reference modules)."""
    from oracle import ldm_oracle as lorc
    from diff_pruning_b200 import ldm
    G = load_golden("ldm_tiny.pt")
    assert G["cin256_v2_params"] == 400920579
    m = ldm_tiny_model(G)
    ac = lorc.alphas_cumprod()
    assert fp(ac) == pytest.approx(G["alphas_cumprod_fp"], rel=1e-6)
    assert torch.equal(ac, ldm.ldm_alphas_cumprod())
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in m.state_dict().items()}
    g1, g2 = torch.Generator().manual_seed(1), torch.Generator().manual_seed(2)
    clean, noise = torch.randn(2, 3, 16, 16, generator=g1), torch.randn(2, 3, 16, 16, generator=g2)
    losses = [lorc.taylor_pass(sd, G["cfg"], ac, clean, noise, (tt * torch.ones(2)).long(), G["context"]).item() for tt in (7, 400)]
    assert losses == pytest.approx(G["losses"], rel=1e-6)
    for k, v in sd.items():
        assert float((v.grad - G["grads"][k]).abs().max()) <= 2e-5 * float(G["grads"][k].abs().max()) + 1e-9, k
    # trace-mode forward of the module tree == oracle forward
    with dp.trace_mode(), torch.no_grad():
        t = (400 * torch.ones(2)).long()
        out = m(lorc.q_sample(ac, clean, noise, t), t, context=G["context"])
    assert max_rel(out, G["out_last"]) < 1e-5
