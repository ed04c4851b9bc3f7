"""GroupNorm outputs written already split for the tensor-core convolutions (dp_groupnorm_fwd_split + DP_CONV_X_SPLIT).

* the split output rebuilds the fp32-mode GroupNorm output to the 22 bits the split keeps, under a bound B >= max|y| known in advance;
* fprop / wgrad reading the split buffer are bitwise equal to the same launches reading fp32 x with the same amax slot value;
* plan level: which GroupNorms go split, and a C1-sized pass gives the same loss / gradients / masks with DPB200_PRESPLIT off and on."""
import ctypes as C
import math

import pytest
import torch

from conftest import worst_grad_err

pytestmark = pytest.mark.gpu

X_SPLIT = 4      # DP_CONV_X_SPLIT


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from diff_pruning_b200 import _lib as L
    lib = L.load()
    if not lib.dp_tc_available():
        pytest.fail("tensor-core path (tcgen05/TMA) not available on this device: conv_tc.cu must run on sm_100a")
    return lib


def S():
    return torch.cuda.current_stream().cuda_stream


def slot_exp(slot):
    return min(max((int(slot.view(torch.int32)[0]) >> 23) & 0xFF, 14), 254)


def unsplit(ys, C_, E):
    v = ys[..., :C_].double()
    return (v[:, 0] + v[:, 1] * 2.0 ** -11) * 2.0 ** (E - 140)


def torch_split(x, E, pitch):
    """What the kernels' split2 makes of x with the scale of exponent E, in the [rows][2][pitch] layout (pad channels zero)."""
    s = 2.0 ** (140 - E)
    xs = x.float() * s
    hi = xs.half()
    lo = ((xs - hi.float()) * 2048.0).half()
    out = torch.zeros((x.shape[0], 2, pitch), dtype=torch.float16, device=x.device)
    out[:, 0, :x.shape[1]], out[:, 1, :x.shape[1]] = hi, lo
    return out


def gn_args(L, N, HW, C_, G, x, gamma, beta, silu, p_drop):
    a = L.GnArgs()
    a.N, a.HW, a.C, a.G, a.eps, a.silu = N, HW, C_, G, 1e-5, silu
    a.x, a.ldx = x.data_ptr(), C_
    a.gamma, a.beta = gamma.data_ptr(), beta.data_ptr()
    if p_drop:
        a.dropout_p, a.dropout_seed = p_drop, 1234
    return a


@pytest.mark.parametrize("C_,G", [(96, 32), (128, 32), (180, 36)])
@pytest.mark.parametrize("N,H", [(1, 256), (2, 32), (8, 4)])
@pytest.mark.parametrize("act", ["none", "silu", "silu+dropout"])
def test_groupnorm_split_output(lib, C_, G, N, H, act):
    from diff_pruning_b200 import _lib as L
    if H == 256 and (C_ != 128 or act == "silu+dropout"):
        pytest.skip("one 256x256 case is enough")
    torch.manual_seed(C_ + H)
    HW = H * H
    x = (torch.randn(N, HW, C_, device="cuda") * 3 + 1).contiguous()
    gamma, beta = torch.randn(C_, device="cuda"), torch.randn(C_, device="cuda") * 0.5
    silu, p = int(act != "none"), (0.1 if "dropout" in act else 0.0)
    ws = torch.empty(lib.dp_groupnorm_workspace_bytes(N, HW, C_, G) // 4 + 64, device="cuda")
    pitch = lib.dp_tc_weight_row(C_)
    # fp32 mode
    a = gn_args(L, N, HW, C_, G, x, gamma, beta, silu, p)
    y = torch.empty_like(x)
    st = torch.empty(2 * N * G, device="cuda")
    slot_y = torch.zeros(1, dtype=torch.int32, device="cuda")
    a.y, a.ldy, a.mean, a.rstd, a.workspace, a.amax_y = y.data_ptr(), C_, st.data_ptr(), st.data_ptr() + 4 * N * G, ws.data_ptr(), slot_y.data_ptr()
    assert lib.dp_groupnorm_fwd(C.byref(a), S()) == 0
    # split mode only
    b = gn_args(L, N, HW, C_, G, x, gamma, beta, silu, p)
    ys = torch.zeros((N * HW, 2, pitch), dtype=torch.float16, device="cuda")
    st2 = torch.empty(2 * N * G, device="cuda")
    slot_b = torch.zeros(1, dtype=torch.int32, device="cuda")
    b.mean, b.rstd, b.workspace, b.amax_y = st2.data_ptr(), st2.data_ptr() + 4 * N * G, ws.data_ptr(), slot_b.data_ptr()
    assert lib.dp_groupnorm_fwd_split(C.byref(b), ys.data_ptr(), pitch, S()) == 0
    torch.cuda.synchronize()
    B = float(slot_b.view(torch.float32)[0])
    ymax = float(y.abs().max())
    assert B >= ymax > 0
    n = C_ // G * HW
    assert B <= (float(gamma.abs().max()) * math.sqrt(n - 1) + float(beta.abs().max())) * (1 / 0.9 if p else 1) * 1.01 + 0.3
    print(f"C={C_} {H}x{H} {act}: log2(B / max|y|) = {math.log2(B / ymax):.2f}")
    assert torch.equal(st, st2)
    E = slot_exp(slot_b)
    yr = unsplit(ys, C_, E)
    ref = y.reshape(-1, C_).double()
    err = (yr - ref).abs()
    assert bool((err <= ref.abs() * 2.0 ** -22 + B * 2.0 ** -48).all()), float((err / (ref.abs() + B * 2.0 ** -48)).max())
    assert not bool(ys[..., C_:].any())          # pad channels untouched
    # the kernels' own split of the fp32 y with the same scale: bitwise the same pairs
    assert torch.equal(ys, torch_split(y.reshape(-1, C_), E, pitch))


def test_groupnorm_split_rejects_unsupported(lib):
    from diff_pruning_b200 import _lib as L
    N, HW, C_, G = 2, 64, 179, 179
    x = torch.randn(N, HW, C_, device="cuda")
    gamma, beta = torch.ones(C_, device="cuda"), torch.zeros(C_, device="cuda")
    a = gn_args(L, N, HW, C_, G, x, gamma, beta, 1, 0.0)
    ws = torch.empty(lib.dp_groupnorm_workspace_bytes(N, HW, C_, G) // 4 + 64, device="cuda")
    st = torch.empty(2 * N * G, device="cuda")
    slot = torch.zeros(1, dtype=torch.int32, device="cuda")
    a.mean, a.rstd, a.workspace, a.amax_y = st.data_ptr(), st.data_ptr() + 4 * N * G, ws.data_ptr(), slot.data_ptr()
    ys = torch.zeros((N * HW, 2, 192), dtype=torch.float16, device="cuda")
    assert lib.dp_groupnorm_fwd_split(C.byref(a), ys.data_ptr(), 192, S()) == -3       # C % 4: no float4 kernel
    a.C, a.G = 176, 16
    a.amax_y = None
    assert lib.dp_groupnorm_fwd_split(C.byref(a), ys.data_ptr(), 192, S()) == -5       # the bound needs its slot


CASES = [
    # N, C, H, W, K, R
    (2, 128, 32, 32, 128, 3),     # 128->128 3x3 @32x32 (long K loop: the raw path would run TS)
    (2, 256, 16, 16, 256, 3),
    (8, 256, 4, 4, 256, 3),       # split-K level
    (4, 256, 8, 8, 256, 3),       # split-K level
    (2, 384, 16, 16, 128, 3),     # up path
    (2, 96, 16, 16, 96, 3),       # pruned widths, pitch 128
    (2, 180, 16, 16, 90, 3),      # pruned widths, pitch 192
    (2, 128, 32, 32, 384, 1),     # fused qkv projection (short K loop: SS on both paths)
    (2, 40, 16, 16, 64, 1),       # pitch 40 < one 64-channel box
]


@pytest.mark.parametrize("N,C_,H,W,K,R", CASES)
def test_conv_split_operand_bitwise(lib, N, C_, H, W, K, R):
    from diff_pruning_b200 import _lib as L
    torch.manual_seed(N * C_ + K)
    x = torch.randn(N, H, W, C_, device="cuda")
    wt = torch.randn(K, C_, R, R, device="cuda") / math.sqrt(C_ * R * R)
    Kld = (K + 3) // 4 * 4                      # dy pitch as the plan lays it out (16-byte rows for TMA)
    dy = torch.randn(N, H, W, Kld, device="cuda")
    Cp, Kp = lib.dp_tc_weight_row(C_), lib.dp_tc_weight_row(K)
    packs = [torch.empty(n, device="cuda", dtype=torch.float16) for n in (R * R * K * Cp, R * R * K * Cp, R * R * C_ * Kp, R * R * C_ * Kp)]
    wslot = torch.zeros(1, dtype=torch.int32, device="cuda")
    assert lib.dp_pack_conv_weight_tc(wt.data_ptr(), K, C_, R, R, *[p.data_ptr() for p in packs], wslot.data_ptr(), S()) == 0
    wck = torch.empty(wt.numel(), device="cuda")
    wkc = torch.empty(wt.numel(), device="cuda")
    assert lib.dp_pack_conv_weight(wt.data_ptr(), K, C_, R, R, wck.data_ptr(), wkc.data_ptr(), S()) == 0
    # slot preset to a loose bound (as the GroupNorm's B is): both forms use the same scale
    xslot = torch.tensor([8.0 * float(x.abs().max())], device="cuda").view(torch.int32)
    yslot = torch.zeros(1, dtype=torch.int32, device="cuda")
    assert lib.dp_amax(dy.data_ptr(), Kld, N * H * W, K, yslot.data_ptr(), S()) == 0
    torch.cuda.synchronize()
    ys = torch_split(x.reshape(-1, C_), slot_exp(xslot), Cp)

    def args(split):
        a = L.ConvArgs()
        a.N, a.H, a.W, a.C, a.P, a.Q, a.K, a.R, a.S = N, H, W, C_, H, W, K, R, R
        a.stride, a.pad_t, a.pad_l, a.splits = 1, (R - 1) // 2, (R - 1) // 2, 1
        a.flags = X_SPLIT if split else 0
        a.x, a.ldx = (ys.data_ptr(), Cp) if split else (x.data_ptr(), C_)
        a.w, a.w_tc_hi, a.w_tc_lo = wck.data_ptr(), packs[0].data_ptr(), packs[1].data_ptr()
        a.amax_x, a.amax_w, a.amax_y = xslot.data_ptr(), wslot.data_ptr(), yslot.data_ptr()
        return a

    assert lib.dp_conv_presplit_eligible(C.byref(args(True))) == 0
    outs = []
    for split in (False, True):
        a = args(split)
        y = torch.full((N, H, W, K), float("nan"), device="cuda")
        a.y, a.ldy = y.data_ptr(), K
        need = lib.dp_conv_splitk_workspace_floats(C.byref(a), 0)
        ws = torch.full((max(need, 1),), float("nan"), device="cuda")
        if need > 0:
            a.workspace = ws.data_ptr()
        assert lib.dp_conv2d_fprop(C.byref(a), S()) == 0
        wa = args(split)
        splits = 3
        wws = torch.full((splits * K * R * R * C_,), float("nan"), device="cuda")
        wa.y, wa.ldy, wa.splits, wa.workspace = dy.data_ptr(), Kld, splits, wws.data_ptr()
        assert lib.dp_conv2d_wgrad(C.byref(wa), S()) == 0
        torch.cuda.synchronize()
        outs.append((y, wws))
    (y0, w0), (y1, w1) = outs
    assert not torch.isnan(y0).any() and not torch.isnan(w0).any()
    assert torch.equal(y0, y1)
    assert torch.equal(w0, w1)
    # and the fp32 reference is still met (the split keeps 22 bits of x whatever the scale)
    ref = torch.nn.functional.conv2d(x.permute(0, 3, 1, 2).double(), wt.double(), padding=(R - 1) // 2).permute(0, 2, 3, 1)
    assert float((y1.double() - ref).norm() / ref.norm()) < 2e-5


def test_split_operand_never_falls_back_to_simt(lib):
    from diff_pruning_b200 import _lib as L
    a = L.ConvArgs()
    N, H, W, C_, K = 2, 16, 16, 64, 64
    x = torch.zeros((N * H * W, 2, 64), dtype=torch.float16, device="cuda")
    y = torch.empty(N, H, W, K, device="cuda")
    wt = torch.empty(K * C_ * 9, device="cuda")
    a.N, a.H, a.W, a.C, a.P, a.Q, a.K, a.R, a.S = N, H, W, C_, H // 2, W // 2, K, 3, 3
    a.stride, a.pad_t, a.pad_l, a.flags = 2, 1, 1, X_SPLIT      # stride 2: outside the split form
    a.x, a.ldx, a.y, a.ldy, a.w = x.data_ptr(), 64, y.data_ptr(), K, wt.data_ptr()
    assert lib.dp_conv_presplit_eligible(C.byref(a)) != 0
    assert lib.dp_conv2d_fprop(C.byref(a), S()) == -3


def _c1_plan_pass(presplit):
    import diff_pruning_b200 as dp
    from diff_pruning_b200 import engine as E
    from diff_pruning_b200.scoring import TaylorScorer
    old = E.PRESPLIT, E.AUDIT_SLOTS
    E.PRESPLIT = presplit
    E.AUDIT_SLOTS = presplit          # every amax slot, the split operands' bounds B included, checked against the operand it scales
    try:
        torch.manual_seed(0)
        cfg = dict(dp.TINY_TEST_CONFIG)
        model = dp.UNet2DModel(**cfg).cuda().eval()
        g = torch.Generator().manual_seed(1)
        clean, noise = torch.randn(4, 3, 32, 32, generator=g), torch.randn(4, 3, 32, 32, generator=g)
        model.zero_grad()
        sc = TaylorScorer(model, clean.cuda(), noise.cuda(), use_graph=False)
        loss = float(sc.step(7))
        torch.cuda.synchronize()
        n_gn = sum(isinstance(m, torch.nn.GroupNorm) for m in model.modules())
        grads = {k: p.grad.detach().clone() for k, p in model.named_parameters()}
        return loss, grads, sc.plan, n_gn
    finally:
        E.PRESPLIT, E.AUDIT_SLOTS = old


def test_plan_presplit_same_results(lib):
    l0, g0, p0, _ = _c1_plan_pass(False)
    l1, g1, plan, n_gn = _c1_plan_pass(True)
    assert p0.split_gn == []
    # every resnet and attention GroupNorm writes split; conv_out's (SIMT convolution, 3 output channels) keeps fp32
    print("split GroupNorm outputs:", plan.split_gn)
    assert len(plan.split_gn) == n_gn - 1
    assert plan.audit_log
    assert abs(l1 - l0) <= 1e-5 * abs(l0)
    assert worst_grad_err(g1.items(), g0) < 1e-4
