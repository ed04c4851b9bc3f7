"""Planned sm_100a executor for the UNet2DModel forward + backward (the Taylor-scoring / finetune hot path).

Instead of dispatching ~1000 ATen ops per pass through autograd (SURVEY.md §3.1: ddpm_prune.py:100-102 ->
unet_2d.py:219 -> autograd), the engine walks the module tree ONCE per (batch, resolution), lays every
activation / gradient out in HBM as fp32 NHWC views, and records two static launch lists (forward, backward)
of libdpb200 C-ABI calls with pre-built argument structs.  Static shapes + no allocation + no sync make the
whole pass CUDA-graph capturable (scoring.py does that).

HBM layout decisions (DESIGN.md §3):
  * NHWC fp32 activations so an implicit-GEMM conv reads K-contiguous rows; weights packed K-major per tap.
  * torch.cat([h, skip]) (unet_2d_blocks.py:1822,2035) never copies: the skip tensor and the up-path tensor
    are written by their producers straight into the two channel ranges of one wider buffer (views with a
    pixel stride), and so are their gradients.
  * residual adds, bias adds and the per-image temb add are conv epilogues; GroupNorm backward takes the
    residual-branch gradient as an addend; the 1x1 shortcut accumulates in place; dW accumulates into the
    Parameter.grad arena across timesteps (ddpm_prune.py:102 has no zero_grad in the loop).
"""
from __future__ import annotations

import ctypes as C
import math
import os
from typing import Callable, Dict, List, Optional, Tuple

import torch
import torch.nn as nn

from . import _lib as L
from .models import (Attention, Downsample2D, ResnetBlock2D, UNet2DModel, Upsample2D, sinusoidal_frequencies)

_byref = C.byref
Step = Callable[[int], None]


_SM_COUNT = 148            # B200; the wgrad kernel runs one CTA per SM (192 KB of shared memory)
_WGRAD_CTA_OVERHEAD = 8    # per-CTA prologue + pipeline fill + TMEM->workspace epilogue, in units of one 64-pixel stage


def _wgrad_splits(tiles, chunks, env=os.environ.get("DPB200_WGRAD_WAVES")):
    """Split-K factor of the tensor-core wgrad: grid = tiles x splits CTAs, each walking ceil(chunks / splits) pixel chunks.
    One CTA per SM, so the launch runs in ceil(grid / 148) strict waves: pick the split count whose modelled time
    waves x (overhead + chunks per CTA) is smallest (ties: fewer splits = smaller workspace), so a grid never overshoots a
    wave boundary by a few CTAs (592 -> 594 CTAs used to cost a fifth, almost empty, wave) and no trailing split is empty."""
    max_waves = int(env) if env else 8
    hi = max(1, min(chunks, max(2, (max_waves * _SM_COUNT) // tiles)))
    best = None
    for sp in range(1, hi + 1):
        cps = -(-chunks // sp)
        if cps * (sp - 1) >= chunks:                 # would leave the last split empty: same as a smaller split count
            continue
        cost = -(-(tiles * sp) // _SM_COUNT) * (_WGRAD_CTA_OVERHEAD + cps)
        if best is None or cost < best[0]:
            best = (cost, sp)
    return best[1]


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


class View:
    """fp32 NHWC view: channels [off, off+C) of a contiguous (N, H, W, Ctot) buffer."""
    __slots__ = ("t", "N", "H", "W", "C", "off", "ld", "g")

    def __init__(self, t: torch.Tensor, off: int = 0, C_: Optional[int] = None):
        assert t.dim() == 4 and t.is_contiguous() and t.dtype == torch.float32
        self.t = t
        self.N, self.H, self.W, self.ld = t.shape
        self.off = off
        self.C = self.ld - off if C_ is None else C_
        self.g: Optional["View"] = None

    @property
    def ptr(self) -> int:
        return self.t.data_ptr() + 4 * self.off

    @property
    def rows(self) -> int:
        return self.N * self.H * self.W

    def torch(self) -> torch.Tensor:
        return self.t[..., self.off:self.off + self.C]


class BItem:
    """Backward work of one forward op: launches in execution order + the gradient views it writes."""
    __slots__ = ("steps", "writes")

    def __init__(self):
        self.steps: List[Step] = []
        # (gradient target view, setter(first_write: bool), amax_setter(slot) or None when the writing kernel cannot report max|value|)
        self.writes: List[Tuple[View, Callable[[bool], None], Optional[Callable[[int], None]]]] = []


def _copy_args(a):
    b = type(a)()
    C.memmove(C.byref(b), C.byref(a), C.sizeof(a))
    return b


AMAX_SLOTS = 8192  # capacity of a plan's amax-slot arrays (one uint32 per tensor-core operand use)
AUDIT_SLOTS = False  # tests: plans built while this is set check every amax slot against torch.amax of its operand right before the
                     # consuming launch (eager runs only: the check synchronises)
SIDE_WGRAD = True  # backward: weight-gradient launches (wgrad + split-K reduce) run on a second stream.  They only feed Parameter.grad, so the
                   # dgrad -> GroupNorm chain does not wait for them, and the small latency-bound kernels of that chain share SMs with wgrad CTAs
SPLITK = True      # small-M fprop / dgrad launches split their K loop over idle SMs (dp_conv_splitk_workspace_floats)
# GroupNorm outputs read only by tensor-core fprop / wgrad launches are written already split into fp16 hi / lo' (dp_groupnorm_fwd_split):
# the convolutions skip their in-kernel split.  DPB200_PRESPLIT=0 plans the fp32 operands instead (A/B runs in one process tree).
PRESPLIT = os.environ.get("DPB200_PRESPLIT", "1") != "0"
CONV_X_SPLIT = 4   # dp_conv_args.flags: DP_CONV_X_SPLIT
ARENA_ALIGN = 64   # floats: every parameter's slice of a flat arena starts on a 256-byte boundary


def arena_offsets(params):
    """Offsets of the parameters inside a flat fp32 arena (gradients / parameters / Adam moments / EMA), each aligned to ARENA_ALIGN
    floats.  Pruned widths (179, 358, 90 ...) otherwise leave every later tensor at an odd float offset: bias / weight pointers then
    fail the 16-byte test of the float4 epilogues and TMA descriptors and the kernels fall back to scalar paths (the round-1 'pruned
    finetune is as slow as the unpruned pass' anomaly).  Gap elements stay zero in every arena (zero grad -> zero Adam update)."""
    offs, o = [], 0
    for p in params:
        offs.append(o)
        o += (p.numel() + ARENA_ALIGN - 1) // ARENA_ALIGN * ARENA_ALIGN
    return offs, o


class Plan:
    """Static forward/backward launch lists for one (model, batch, H, W)."""

    def __init__(self, model: UNet2DModel, batch: int, height: int, width: int, device, training: bool = False,
                 need_grad: bool = True, fused_scores: bool = False, compute: str = "fp32"):
        self.lib = L.load()
        self.tc = bool(self.lib.dp_tc_available()) if torch.device(device).type == "cuda" else False
        if compute not in ("fp32", "bf16"):
            raise ValueError(f"compute must be 'fp32' (3 x fp16 split, fp32-grade) or 'bf16' (single-pass tensor tier), got {compute!r}")
        if compute == "bf16" and not (torch.device(device).type == "cuda" and self.lib.dp_bf16_available()):
            raise RuntimeError("diff_pruning_b200: the bf16 tensor tier needs an sm_100a device (no fallback)")
        # bf16 tier (ddpm_train.py --mixed_precision bf16 -> torch.autocast: conv / linear operands in bf16, everything else fp32):
        # eligible convolutions read bf16 operands (written by GroupNorm+SiLU directly, or by dp_cvt_bf16) on the kind::f16 kernels
        self.compute = compute
        self.bf16 = compute == "bf16"
        self._bf_cache: Dict[Tuple[int, int, int], Tuple[torch.Tensor, int]] = {}
        self._bf_packs: Dict[int, Tuple[torch.Tensor, torch.Tensor]] = {}
        self.n_bf16_convs = 0
        # GroupNorm outputs planned in split form: (buffer address, channel offset, channels) -> (fp16 [rows][2][pitch], pitch)
        self._split_cache: Dict[Tuple[int, int, int], Tuple[torch.Tensor, int]] = {}
        self.split_gn: List[str] = []     # shape tags of those GroupNorms, in plan order
        self.model = model
        self.B, self.H, self.W = batch, height, width
        self.dev = torch.device(device)
        self.need_grad = need_grad
        self.training = training
        self.fwd: List[Step] = []
        self.bwd: List[BItem] = []      # appended in forward order, executed reversed
        self.pack: List[Step] = []      # weight packing launches (re-run when weights change)
        self._keep: list = []           # tensors / structs that must stay alive
        self._ginit: set = set()
        self._gbuf: Dict[int, torch.Tensor] = {}
        self._scratch: Dict[str, torch.Tensor] = {}
        self._scratch_need: Dict[str, int] = {}
        self._late: List[Callable[[], None]] = []   # pointer fix-ups once scratch buffers exist
        self._packs: Dict[int, Tuple[torch.Tensor, torch.Tensor]] = {}
        # amax slots of the tensor-core operands (3 x fp16 split, conv_tc.cu): activations / gradients get a slot per use, zeroed at the
        # start of every forward and filled by dp_amax right before the launch that reads it; weights keep theirs across passes
        self._slots = torch.zeros(AMAX_SLOTS, device=self.dev, dtype=torch.int32)
        self._wslots = torch.zeros(AMAX_SLOTS, device=self.dev, dtype=torch.int32)
        self._n_slots = self._n_wslots = 0
        self._amax_fwd: Dict[Tuple[int, int, int, int], int] = {}
        # producer-filled slots, keyed by the activation tensor's base address: forward = every kernel writing into the tensor adds
        # max|written| (an upper bound for any sub-view a consumer reads); backward = the same for the tensor's gradient buffer, bound
        # at _finalize_build once all writers are known (a writer without amax support keeps the consumer's dp_amax launch)
        self._slot_tags: List[str] = []
        self._fslot: Dict[int, int] = {}
        self._fslot_bad: set = set()
        self._bslot: Dict[int, dict] = {}
        one = torch.tensor([1.0], dtype=torch.float32).view(torch.int32).to(self.dev)
        self._wslots[AMAX_SLOTS - 1:] = one            # constant slot: bound 1.0 (softmax probabilities)
        self._one_slot = self._wslots.data_ptr() + 4 * (AMAX_SLOTS - 1)
        self.audit_log: list = []
        self.audit = AUDIT_SLOTS
        self.params = [p for p in model.parameters()]
        self.dropout_seed_dev = torch.zeros(1, device=self.dev, dtype=torch.int64)
        self._n_dropout = 0
        self.fused_scores = fused_scores and need_grad
        self.lin_macs = 0
        self.conv_macs = 0             # MACs of one forward over the 4-D-weight convolutions (set while building)
        self.generation = 0            # forward counter of the autograd boundary (see _UNetFunction)
        self._calls = 0                # module-forward counter: advances the dropout stream on the autograd / compat path
        self.scores: Dict[int, Tuple[torch.Tensor, torch.Tensor]] = {}
        if self.fused_scores:   # one flat vector: [out-channel | in-channel] signed scores of every conv / linear weight
            n = sum(p.shape[0] + p.shape[1] for p in self.params if p.dim() >= 2)
            self.score_arena = torch.zeros(n, device=self.dev, dtype=torch.float32)
            self._score_off = 0
        self._build()

    # ------------------------------------------------------------------ memory helpers
    def new(self, N, H, W, C_) -> View:
        """Activation buffer; the pixel stride is rounded up to 4 floats so every view is TMA-addressable (16-byte pitch)
        even for pruned widths such as 179 or 358."""
        t = torch.empty((N, H, W, (C_ + 3) // 4 * 4), device=self.dev, dtype=torch.float32)
        self._keep.append(t)
        return View(t, 0, C_)

    def gradof(self, v: View) -> View:
        """Gradient view mirroring v (same buffer geometry, so concat views stay views)."""
        if v.g is None:
            gt = self._gbuf.get(v.t.data_ptr())
            if gt is None:
                gt = torch.empty_like(v.t)
                self._gbuf[v.t.data_ptr()] = gt
            v.g = View(gt, v.off, v.C)
        return v.g

    def g_is_init(self, v: View) -> bool:
        g = self.gradof(v)
        p = g.t.data_ptr()
        return any(q == p and off <= g.off and g.off + g.C <= off + c for (q, off, c) in self._ginit)

    def g_mark(self, v: View):
        g = self.gradof(v)
        self._ginit.add((g.t.data_ptr(), g.off, g.C))

    def scratch(self, name: str, nfloats: int) -> str:
        """Shared temporary (always consumed right after it is produced)."""
        self._scratch_need[name] = max(self._scratch_need.get(name, 0), int(nfloats))
        return name

    def sptr(self, name: str) -> int:
        return self._scratch[name].data_ptr()

    # ------------------------------------------------------------------ parameter plumbing
    def pgrad(self, p: nn.Parameter) -> int:
        return self._grad_views[id(p)].data_ptr()

    def _setup_param_grads(self):
        offs, total = arena_offsets(self.params)
        self.grad_arena = torch.zeros(total, device=self.dev, dtype=torch.float32)
        self._grad_views = {}
        for p, o in zip(self.params, offs):
            self._grad_views[id(p)] = self.grad_arena[o:o + p.numel()].view_as(p)

    def attach_grads(self):
        """Make every Parameter.grad the plan's arena view (accumulating semantics are preserved)."""
        for p in self.params:
            gv = self._grad_views[id(p)]
            if p.grad is None:
                gv.zero_()
                p.grad = gv
            elif p.grad.data_ptr() != gv.data_ptr():
                gv.copy_(p.grad)
                p.grad = gv

    def signature(self):
        return tuple((p.data_ptr(), tuple(p.shape)) for p in self.params)

    def weight_version(self):
        """(sum of autograd version counters, explicit weights epoch of the model).  The version counters catch optimiser steps and
        load_state_dict; writes torch does not track — `param.data.copy_()` (how EMAModel.copy_to / restore write weights,
        training_utils.py:216-224 of the reference's diffusers) and kernels that update the parameter arena through raw pointers
        (FinetuneStepper) — are covered by the epoch, bumped by invalidate_packs()."""
        return (sum(p._version for p in self.params), self.model.__dict__.get("_dpb200_weights_epoch", 0))

    def _score_views(self, w: nn.Parameter, K: int, Cin: int):
        got = self.scores.get(id(w))
        if got is None:
            o = self._score_off
            got = (self.score_arena[o:o + K], self.score_arena[o + K:o + K + Cin])
            self._score_off = o + K + Cin
            self.scores[id(w)] = got
        return got

    # ------------------------------------------------------------------ launch recording
    def _rec(self, lst: List[Step], fn, args=None, what="", info=""):
        check = L.check
        if args is not None:
            self._keep.append(args)
            ref = _byref(args)

            def run(s, fn=fn, ref=ref, what=what):
                rc = fn(ref, s)
                if rc:
                    check(rc, what)
        else:
            def run(s, fn=fn, what=what):
                rc = fn(s)
                if rc:
                    check(rc, what)
        run.what = what
        run.info = info          # shape tag for per-layer timing tables (bench.py, scripts/trace_pass.py)
        lst.append(run)

    def _bitem(self) -> BItem:
        it = BItem()
        self.bwd.append(it)
        return it

    # ------------------------------------------------------------------ op emitters
    def _packed(self, w: nn.Parameter):
        """(w_ck, w_kc): K-major packed copies of an OIHW / (out,in) weight; the packing launch is recorded once."""
        got = self._packs.get(id(w))
        if got is not None:
            return got
        K, Cin = w.shape[0], w.shape[1]
        R = w.shape[2] if w.dim() == 4 else 1
        S = w.shape[3] if w.dim() == 4 else 1
        wck = torch.empty(w.numel(), device=self.dev, dtype=torch.float32)
        wkc = torch.empty(w.numel(), device=self.dev, dtype=torch.float32)
        lib = self.lib
        self._rec(self.pack, lambda s, w=w, K=K, Cin=Cin, R=R, S=S, a=wck, b=wkc:
                  lib.dp_pack_conv_weight(w.data_ptr(), K, Cin, R, S, a.data_ptr(), b.data_ptr(), s), what="pack")
        tc = None
        if self.tc and K * Cin >= 256:
            RS = R * S
            na, nb = RS * K * lib.dp_tc_weight_row(Cin), RS * Cin * lib.dp_tc_weight_row(K)   # rows padded for aligned TMA box rows
            wslot = self._wslots.data_ptr() + 4 * self._n_wslots
            self._n_wslots += 1
            assert self._n_wslots < AMAX_SLOTS
            # fp16 kc_hi kc_lo ck_hi ck_lo + the weight's amax slot (one power-of-two scale per tensor)
            tc = tuple(torch.empty(n, device=self.dev, dtype=torch.float16) for n in (na, na, nb, nb)) + (wslot,)
            self._rec(self.pack, lambda s, w=w, K=K, Cin=Cin, R=R, S=S, t=tc:
                      lib.dp_pack_conv_weight_tc(w.data_ptr(), K, Cin, R, S, t[0].data_ptr(), t[1].data_ptr(), t[2].data_ptr(),
                                                 t[3].data_ptr(), t[4], s), what="pack tc")
        self._packs[id(w)] = (wck, wkc, tc)
        return wck, wkc, tc

    def _new_slot(self, tag: str = "") -> int:
        """Device address of a fresh per-pass amax slot (zeroed by the first launch of every forward)."""
        self._slot_tags.append(tag)
        slot = self._slots.data_ptr() + 4 * self._n_slots
        self._n_slots += 1
        assert self._n_slots <= AMAX_SLOTS, "raise engine.AMAX_SLOTS"
        return slot

    def _amax(self, lst: List[Step], ptr_get, ld: int, rows: int, cols: int, fwd_key=None) -> int:
        """Records dp_amax over a [rows][cols] view into a fresh amax slot; returns the slot's device address.  Forward activations are
        written once per pass, so consumers of the same view share one slot (fwd_key)."""
        if fwd_key is not None and fwd_key in self._amax_fwd:
            return self._amax_fwd[fwd_key]
        slot = self._new_slot(f"amax {rows}x{cols}")
        lib = self.lib
        self._rec(lst, lambda s, g=ptr_get: lib.dp_amax(g(), ld, rows, cols, slot, s), what="amax")
        if fwd_key is not None:
            self._amax_fwd[fwd_key] = slot
        return slot

    def _out_slot(self, out: View) -> Optional[int]:
        """Producer side (forward): the slot of the tensor `out` lives in; the producing kernel adds max|values written|."""
        if not self.tc:
            return None
        k = out.t.data_ptr()
        if k not in self._fslot:
            self._fslot[k] = self._new_slot(f"out {out.N}x{out.H}x{out.W}x{out.t.shape[-1]}")
        return self._fslot[k]

    def _alias_slot(self, out: View, src: View):
        """`out` holds copies of src's values only (nearest-neighbour upsampling): src's bound is out's bound."""
        k = src.t.data_ptr()
        if self.tc and k in self._fslot and k not in self._fslot_bad:
            self._fslot[out.t.data_ptr()] = self._fslot[k]

    def _unslotted(self, out: View):
        """A kernel without amax support writes into this tensor: consumers must measure their operand themselves."""
        self._fslot_bad.add(out.t.data_ptr())

    def _x_slot(self, x: View) -> int:
        """Consumer side (forward): the producer-filled slot of x's tensor, else a dp_amax launch over the view."""
        k = x.t.data_ptr()
        if k in self._fslot and k not in self._fslot_bad:
            slot = self._fslot[k]
        else:
            slot = self._amax(self.fwd, lambda p=x.ptr: p, x.ld, x.rows, x.C, fwd_key=(x.ptr, x.ld, x.rows, x.C))
        sp = self._split_cache.get((x.t.data_ptr(), x.off, x.C))
        if sp is not None:     # only the split form is written: check the bound against the operand rebuilt from it
            self._audit(self.fwd, slot, lambda sp=sp, x=x, slot=slot: self._unsplit(sp, x, slot))
        else:
            self._audit(self.fwd, slot, lambda x=x: x.torch())
        return slot

    def _unsplit(self, sp: Tuple[torch.Tensor, int], x: View, slot: int) -> torch.Tensor:
        """(hi + lo' * 2^-11) / s of a split operand, s = the power of two the kernels derive from the slot (common.cuh scale_up)."""
        t, pitch = sp
        bits = int(self._slots[(slot - self._slots.data_ptr()) // 4])
        E = min(max((bits >> 23) & 0xFF, 14), 254)
        v = t.view(-1, 2, pitch)[:, :, :x.C].double()
        return ((v[:, 0] + v[:, 1] * 2.0 ** -11) * 2.0 ** (E - 140)).float()

    def presplit_ok(self, gn_in: View, x: View, out: View, w: nn.Parameter, stride: int = 1, pad: int = 1) -> bool:
        """Can the GroupNorm gn_in -> x write x in split form for its one consumer, the convolution x -> out with weight w?  Needs the
        tensor-core fprop and wgrad of that convolution to take a split operand, and one float4 GroupNorm launch (one scale per tensor)."""
        K, Cin = w.shape[0], w.shape[1]
        if not (PRESPLIT and self.tc and not self.bf16) or K * Cin < 256:
            return False
        if gn_in.C % 4 or gn_in.off % 4 or gn_in.C > self.GN_MAX_C:
            return False
        a = L.ConvArgs()
        a.N, a.H, a.W, a.C = x.N, x.H, x.W, x.C
        a.P, a.Q, a.K = out.H, out.W, K
        a.R = w.shape[2] if w.dim() == 4 else 1
        a.S = w.shape[3] if w.dim() == 4 else 1
        a.stride, a.pad_t, a.pad_l = stride, pad, pad
        return self.lib.dp_conv_presplit_eligible(_byref(a)) == 0

    def _split_of(self, x: View) -> Optional[Tuple[torch.Tensor, int]]:
        return self._split_cache.get((x.t.data_ptr(), x.off, x.C))

    def _dy_slot(self, steps: List[Step], v: View) -> int:
        """Consumer side (backward): slot of max|v.grad|.  The writers of v.grad are built later; _finalize_build hands them the slot and
        drops the dp_amax launch recorded here when every one of them can report its own maximum."""
        g = self.gradof(v)
        rec = self._bslot.get(v.t.data_ptr())
        if rec is None:
            rec = self._bslot[v.t.data_ptr()] = {"slot": self._new_slot(f"grad {v.N}x{v.H}x{v.W}x{v.t.shape[-1]}"), "flags": []}
        slot, flag, lib = rec["slot"], [True], self.lib
        rec["flags"].append(flag)

        def run(s, flag=flag, g=g):
            if flag[0]:
                L.check(lib.dp_amax(g.ptr, g.ld, g.rows, g.C, slot, s), "amax")
        run.what, run.info = "amax", ""
        steps.append(run)
        self._audit(steps, slot, lambda g=g: g.torch())
        return slot

    def _audit(self, lst: List[Step], slot: int, get):
        if not self.audit:
            return

        def run(s, slot=slot, get=get):
            torch.cuda.current_stream().synchronize()
            arr = self._slots if self._slots.data_ptr() <= slot < self._slots.data_ptr() + 4 * AMAX_SLOTS else self._wslots
            bound = float(arr.view(torch.float32)[(slot - arr.data_ptr()) // 4])
            true = float(get().abs().max())
            if not (bound >= true):
                raise AssertionError(f"amax slot {bound} below the operand's maximum {true}")
            self.audit_log.append((bound, true))
        run.what, run.info = "audit", ""
        lst.append(run)

    # ------------------------------------------------------------------ bf16 tier plumbing
    def _bf_geom(self, x: View, out: View, w: nn.Parameter, stride: int, pad: int) -> "L.ConvBf16Args":
        a = L.ConvBf16Args()
        a.N, a.H, a.W, a.C = x.N, x.H, x.W, x.C
        a.P, a.Q, a.K = out.H, out.W, w.shape[0]
        a.R = w.shape[2] if w.dim() == 4 else 1
        a.S = w.shape[3] if w.dim() == 4 else 1
        a.stride, a.pad_t, a.pad_l, a.splits = stride, pad, pad, 1
        a.ldx, a.lddy, a.ld_out = (x.C + 7) // 8 * 8, (w.shape[0] + 7) // 8 * 8, max(out.ld, x.ld)
        return a

    def conv_bf16_ok(self, x: View, out: View, w: nn.Parameter, stride: int = 1, pad: int = 1, need_dx: bool = True) -> bool:
        """Does this convolution run on the bf16 kernels?  All of its launches (fprop, wgrad, dgrad) or none.  Small GEMMs (the
        time-embedding MLP, per-image temb projections: rows = batch) and 3-channel ends (conv_in / conv_out) stay fp32-grade:
        they are launch-latency-sized and cost nothing to keep exact."""
        if not self.bf16 or x.rows < 256 or w.shape[1] < 16 or w.shape[0] < 16:
            return False
        g = self._bf_geom(x, out, w, stride, pad)
        ops = [0] + ([2] + ([1] if need_dx else []) if self.need_grad else [])
        return all(self.lib.dp_conv_bf16_eligible(_byref(g), op) == 0 for op in ops)

    def _bf_new(self, rows: int, C_: int) -> Tuple[torch.Tensor, int]:
        ld = (C_ + 7) // 8 * 8
        t = torch.empty((rows, ld), device=self.dev, dtype=torch.bfloat16)
        self._keep.append(t)
        return t, ld

    def _bf16_of(self, v: View) -> Tuple[torch.Tensor, int]:
        """The bf16 operand copy of an activation view: written by its producer when one registered it (GroupNorm), else by ONE
        dp_cvt_bf16 launch recorded at the first consumer (the buffer is stable from there to the end of the backward pass)."""
        key = (v.t.data_ptr(), v.off, v.C)
        got = self._bf_cache.get(key)
        if got is None:
            got = self._bf_new(v.rows, v.C)
            self._bf_cache[key] = got
            t, ld = got
            self._rec(self.fwd, lambda s, p=v.ptr, ldv=v.ld, r=v.rows, c=v.C, d=t.data_ptr(), ld=ld:
                      self.lib.dp_cvt_bf16(p, ldv, r, c, d, ld, s), what="cvt bf16")
        return got

    def _packed_bf16(self, w: nn.Parameter):
        got = self._bf_packs.get(id(w))
        if got is None:
            K, Cin = w.shape[0], w.shape[1]
            R = w.shape[2] if w.dim() == 4 else 1
            S = w.shape[3] if w.dim() == 4 else 1
            lib = self.lib
            kc = torch.empty(R * S * K * lib.dp_bf16_weight_row(Cin), device=self.dev, dtype=torch.bfloat16)
            ck = torch.empty(R * S * Cin * lib.dp_bf16_weight_row(K), device=self.dev, dtype=torch.bfloat16)
            self._rec(self.pack, lambda s, w=w, K=K, Cin=Cin, R=R, S=S, a=kc, b=ck:
                      lib.dp_pack_conv_weight_bf16(w.data_ptr(), K, Cin, R, S, a.data_ptr(), b.data_ptr(), s), what="pack bf16")
            got = (kc, ck)
            self._bf_packs[id(w)] = got
        return got

    def _colsum_tree(self, steps: List[Step], src_ptr: int, ld: int, rows: int, per_img: int, cols: int,
                     seg_name: Optional[str], tmp: Tuple[str, str] = ("cs_a", "cs_b")) -> str:
        """Deterministic hierarchical column sums of a [rows][cols] view down to per-image sums (dense [N][cols]);
        returns the scratch name holding them."""
        lib = self.lib
        get = (lambda p=src_ptr: p)
        cur_ld, cur_rows, cur_per, level = ld, rows, per_img, 0
        while True:
            s_rows = 256 if (cur_per > 256 and cur_per % 256 == 0) else cur_per
            nseg = cur_rows // s_rows
            last = cur_per == s_rows
            out_name = seg_name if (last and seg_name) else tmp[level & 1]
            self.scratch(out_name, nseg * cols)
            self._rec(steps, lambda s, g=get, ld_=cur_ld, r=cur_rows, sr=s_rows, o=out_name:
                      lib.dp_colsum(g(), ld_, r, cols, sr, self.sptr(o), cols, 0, s), what="colsum")
            get = (lambda o=out_name: self.sptr(o))
            cur_ld, cur_rows, cur_per = cols, nseg, cur_per // s_rows
            level += 1
            if last:
                return out_name

    def conv(self, x: View, w: nn.Parameter, b: Optional[nn.Parameter], out: View, stride=1, pad=1,
             rowadd: Optional[View] = None, residual: Optional[View] = None, accumulate_out=False, need_dx=True,
             dx_scratch: Optional[str] = None, seg_out: Optional[str] = None, dy_dense: Optional[str] = None,
             dx_into: Optional[View] = None):
        """Records fprop (fwd) and bias-grad / wgrad / dgrad (bwd).
        dgrad target: `dx_scratch` (shared dense scratch [rows][C]) or the gradient view of `dx_into` / `x`.
        dy source: out.grad, or the dense scratch `dy_dense` ([rows][K]) when the consumer provides it."""
        lib = self.lib
        K, Cin = w.shape[0], w.shape[1]
        R = w.shape[2] if w.dim() == 4 else 1
        S = w.shape[3] if w.dim() == 4 else 1
        assert x.C == Cin and out.C == K, (x.C, Cin, out.C, K)
        use_bf = dy_dense is None and self.conv_bf16_ok(x, out, w, stride, pad, need_dx)
        if use_bf:
            return self._conv_bf16(x, w, b, out, stride, pad, rowadd, residual, accumulate_out, need_dx, dx_scratch, seg_out, dx_into)
        wck, wkc, wtc = self._packed(w)
        a = L.ConvArgs()
        if wtc is not None:
            a.w_tc_hi, a.w_tc_lo, a.amax_w = wtc[0].data_ptr(), wtc[1].data_ptr(), wtc[4]
            a.amax_x = self._x_slot(x)
        xs = self._split_of(x)
        if xs is not None:
            assert wtc is not None, "a split operand needs the tensor-core path"
        a.N, a.H, a.W, a.C = x.N, x.H, x.W, x.C
        a.P, a.Q, a.K = out.H, out.W, K
        a.R, a.S, a.stride, a.pad_t, a.pad_l = R, S, stride, pad, pad
        a.flags = (1 if accumulate_out else 0) | (CONV_X_SPLIT if xs is not None else 0)
        a.splits = 1
        a.x, a.ldx, a.y, a.ldy = x.ptr, x.ld, out.ptr, out.ld
        if xs is not None:
            a.x, a.ldx = xs[0].data_ptr(), xs[1]
        a.amax_out = self._out_slot(out)
        a.w = wck.data_ptr()
        a.bias = b.data_ptr() if b is not None else None
        if rowadd is not None:
            a.rowadd, a.ld_rowadd = rowadd.ptr, rowadd.ld
        if residual is not None:
            a.residual, a.ld_res = residual.ptr, residual.ld
        info = f"{Cin}->{K} {R}x{S}" + (f" s{stride}" if stride != 1 else "") + f" @{out.H}x{out.W}"
        if w.dim() == 4:
            self.conv_macs += out.rows * K * Cin * R * S      # 4-D-weight convolutions only: the roofline denominator (SURVEY.md §8d)
        else:
            self.lin_macs += out.rows * K * Cin               # nn.Linear layers (the LDM transformer blocks are linear-heavy)
        self._splitk(a, 0)
        self._rec(self.fwd, lib.dp_conv2d_fprop, a, "conv fprop", info)
        if not self.need_grad:
            return
        it = self._bitem()
        steps = it.steps
        # The time-embedding branch of a resnet (per-image sums of conv1's dy -> bias / time_emb_proj gradients -> d silu(temb)) only meets
        # the main chain again at the very end of the backward: all of it runs on the side stream (fp32-grade plans; scratch of its own)
        temb_side = SIDE_WGRAD and not self.bf16 and (dy_dense is not None or seg_out is not None)
        n_steps0 = len(steps)
        if dy_dense is not None:
            self.scratch(dy_dense, out.rows * K)
            dy_get, dy_ld = (lambda n=dy_dense: self.sptr(n)), K
        else:
            dout = self.gradof(out)
            dy_get, dy_ld = (lambda p=dout.ptr: p), dout.ld
        # 1. bias gradient (and per-image sums for the caller when seg_out is set).  Without seg_out the bias gradient falls out of the
        #    wgrad kernel's pass over dy (bias_ws -> dp_conv2d_wgrad_reduce): no column-sum launches at all
        bias_in_wgrad = b is not None and seg_out is None and dy_dense is None
        if (b is not None or seg_out is not None) and not bias_in_wgrad:
            if dy_dense is not None and out.H * out.W == 1:
                seg = dy_dense  # already dense per-image rows
            else:
                seg = None
            if seg is None:
                # src pointer may be late-bound (dense scratch) -> wrap
                if dy_dense is not None:
                    raise NotImplementedError("dense dy with spatial extent")
                seg = self._colsum_tree(steps, dout.ptr, dout.ld, out.rows, out.H * out.W, K, seg_out,
                                        ("cs_a_side", "cs_b_side") if temb_side else ("cs_a", "cs_b"))
            if b is not None:
                self._rec(steps, lambda s, seg=seg, b=b, n=x.N: lib.dp_colsum(self.sptr(seg), K, n, K, n, self.pgrad(b), K, 1, s),
                          what="bias grad")
            if temb_side:
                for f in steps[n_steps0:]:
                    f.side = 1
                steps[n_steps0].side = 2
        # 2. wgrad -> split-K workspace -> fixed-order reduce into Parameter.grad
        TC = R * S * Cin
        tiles = ((K + 127) // 128) * ((Cin + 127) // 128) * R * S   # the kernel's grid: out-channel tiles x in-channel tiles x taps
        chunks = max(1, out.rows // 64)              # tensor-core wgrad walks 64-pixel chunks
        splits = _wgrad_splits(tiles, chunks)
        # dy in a per-tensor gradient buffer stays valid for the rest of the backward: its weight gradient may run on the side stream
        # (own scratch: the main stream's wgrads — the temb projections, whose dy lives in a reused scratch — must not share it)
        side = SIDE_WGRAD and (dy_dense is None or temb_side)
        ws_name, bws_name = ("wgrad_ws_side", "bias_ws_side") if side else ("wgrad_ws", "bias_ws")
        n_steps1 = len(steps)
        self.scratch(ws_name, splits * K * TC)
        amax_dy = None
        if wtc is not None:
            amax_dy = self._amax(steps, dy_get, dy_ld, out.rows, K) if dy_dense is not None else self._dy_slot(steps, out)
        wa = _copy_args(a)
        wa.amax_y, wa.amax_out = amax_dy, None
        wa.flags, wa.splits = a.flags & CONV_X_SPLIT, splits
        wa.ldy = dy_ld
        wa.rowadd, wa.residual, wa.bias = None, None, None
        self._late.append(lambda wa=wa, g=dy_get, n=ws_name: (setattr(wa, "y", g()), setattr(wa, "workspace", self.sptr(n))))
        if bias_in_wgrad:
            self.scratch(bws_name, splits * K)
            self._late.append(lambda wa=wa, n=bws_name: setattr(wa, "bias_ws", self.sptr(n)))
        self._rec(steps, lib.dp_conv2d_wgrad, wa, "conv wgrad", info)
        steps[-1].side = 2 if side else 0          # 2: first launch of a side group (waits for the main stream's progress so far)
        ra = L.WgradReduceArgs()
        ra.K, ra.C, ra.R, ra.S, ra.splits = K, Cin, R, S, splits
        ra.dw = self.pgrad(w)
        if self.fused_scores:   # signed first-order Taylor terms sum_k W*dW_t fall out of the split-K reduce (ddpm_prune.py:60)
            so, si = self._score_views(w, K, Cin)
            ra.w, ra.score_out, ra.score_in = w.data_ptr(), so.data_ptr(), si.data_ptr()
        self._late.append(lambda ra=ra, n=ws_name: setattr(ra, "workspace", self.sptr(n)))
        if bias_in_wgrad:
            ra.db = self.pgrad(b)
            self._late.append(lambda ra=ra, n=bws_name: setattr(ra, "bias_ws", self.sptr(n)))
        self._rec(steps, lib.dp_conv2d_wgrad_reduce, ra, "conv wgrad reduce")
        steps[-1].side = 1 if side else 0
        # 3. dgrad
        if need_dx:
            da = _copy_args(a)
            da.ldy = dy_ld
            da.w = wkc.data_ptr()
            if wtc is not None:
                da.w_tc_hi, da.w_tc_lo, da.amax_y = wtc[2].data_ptr(), wtc[3].data_ptr(), amax_dy
            da.flags = 0
            da.amax_out = None
            da.rowadd, da.residual, da.bias = None, None, None
            self._late.append(lambda da=da, g=dy_get: setattr(da, "y", g()))
            if dx_scratch is not None:
                self.scratch(dx_scratch, x.rows * x.C)
                da.ldx = x.C
                self._late.append(lambda da=da, n=dx_scratch: setattr(da, "x", self.sptr(n)))
            else:
                tgt = dx_into if dx_into is not None else x
                gx = self.gradof(tgt)
                da.x, da.ldx = gx.ptr, gx.ld
                it.writes.append((tgt, lambda init, da=da: setattr(da, "flags", 1 if init else 0),
                                  lambda slot, da=da: setattr(da, "amax_out", slot)))
            da.workspace = None
            self._splitk(da, 1, "splitk_ws_side" if (temb_side and dy_dense is not None) else "splitk_ws")
            self._rec(steps, lib.dp_conv2d_dgrad, da, "conv dgrad", info)
        if temb_side and dy_dense is not None:      # the time_emb_proj convolution: amax(dy), wgrad, reduce, dgrad all on the side stream
            for f in steps[n_steps1:]:
                f.side = 1
            steps[n_steps1].side = 2

    FUSE_QKV = True      # to_q / to_k / to_v of an attention block as one projection (conv_qkv); tests / A-B runs may clear it before planning

    def qkv_fusable(self, x: View, lins) -> bool:
        ws = [l.weight for l in lins]
        inner, Cin = ws[0].shape[0], ws[0].shape[1]
        return bool(self.FUSE_QKV and self.tc and not self.bf16 and all(tuple(w.shape) == (inner, Cin) for w in ws)
                    and inner * Cin >= 256 and x.rows >= 128 and len({l.bias is None for l in lins}) == 1)

    def conv_qkv(self, x: View, lins) -> Tuple[View, View, View]:
        """q, k, v = to_q(x), to_k(x), to_v(x) (attention_processor.py:432-441; ldm attention.py:172-176) as ONE 1x1 convolution over the
        concatenated out-channels, q / k / v being channel ranges of one [N][H][W][3 inner] buffer: x is read once instead of three
        times, and the backward needs one dgrad over K = 3 inner instead of three launches of which two read-modify-write dx.  The
        weight gradients stay three launches (one per Parameter: their .grad slices are not adjacent in the arena), each over its
        channel range of the shared dy buffer, on the side stream like every other wgrad.  The fused fp32 operand [3 inner][C] is
        gathered from the three Parameters by the pack list (re-run whenever the weights change) and packed like any other weight;
        one amax slot covers q, k and v (an upper bound is all a slot has to be).  Pruned widths (inner = 179 ...): every part starts on a
        multiple of 4 channels (16-byte aligned views for TMA); the pad channels have zero weight rows and zero bias, so the forward
        writes zeros there, and their gradient columns are zeroed once here and never written again."""
        lib = self.lib
        ws = [l.weight for l in lins]
        bs = [l.bias for l in lins]
        inner, Cin = ws[0].shape[0], ws[0].shape[1]
        ip = (inner + 3) // 4 * 4          # channel pitch of a part inside the fused buffer
        K = 3 * ip
        assert x.C == Cin
        qkv = self.new(x.N, x.H, x.W, K)
        parts = tuple(View(qkv.t, i * ip, inner) for i in range(3))
        wf = torch.zeros((K, Cin), device=self.dev, dtype=torch.float32)
        self._keep.append(wf)
        for i, w in enumerate(ws):
            self._rec(self.pack, lambda s, w=w, d=wf.data_ptr() + 4 * i * ip * Cin:
                      lib.dp_copy_rows(w.data_ptr(), Cin, d, Cin, inner, Cin, s), what="pack qkv")
        has_bias = bs[0] is not None
        bf = None
        if has_bias:
            bf = torch.zeros(K, device=self.dev, dtype=torch.float32)
            self._keep.append(bf)
            for i, b in enumerate(bs):
                self._rec(self.pack, lambda s, b=b, d=bf.data_ptr() + 4 * i * ip:
                          lib.dp_copy_rows(b.data_ptr(), inner, d, inner, 1, inner, s), what="pack qkv")
        wck, wkc, wtc = self._packed(wf)
        assert wtc is not None
        a = L.ConvArgs()
        a.w_tc_hi, a.w_tc_lo, a.amax_w = wtc[0].data_ptr(), wtc[1].data_ptr(), wtc[4]
        a.amax_x = self._x_slot(x)
        a.N, a.H, a.W, a.C = x.N, x.H, x.W, Cin
        a.P, a.Q, a.K = x.H, x.W, K
        a.R, a.S, a.stride, a.pad_t, a.pad_l = 1, 1, 1, 0, 0
        a.flags, a.splits = 0, 1
        a.x, a.ldx, a.y, a.ldy = x.ptr, x.ld, qkv.ptr, qkv.ld
        xs = self._split_of(x)
        if xs is not None:
            a.flags, a.x, a.ldx = CONV_X_SPLIT, xs[0].data_ptr(), xs[1]
        a.amax_out = self._out_slot(qkv)
        a.w = wck.data_ptr()
        a.bias = bf.data_ptr() if has_bias else None
        info = f"{Cin}->{K} 1x1 @{x.H}x{x.W}"
        self.lin_macs += qkv.rows * K * Cin
        self._splitk(a, 0)
        self._rec(self.fwd, lib.dp_conv2d_fprop, a, "conv fprop", info)
        if not self.need_grad:
            return parts
        it = self._bitem()
        steps = it.steps
        dout = self.gradof(qkv)
        if ip != inner:
            dout.t.zero_()                 # pad columns of dy: read by the fused dgrad (against zero weights), written by nobody
        amax_dy = self._dy_slot(steps, qkv)
        # weight (and bias) gradients: one launch per Parameter over its channel range of dy, side stream
        pinfo = f"{Cin}->{inner} 1x1 @{x.H}x{x.W}"
        tiles = ((inner + 127) // 128) * ((Cin + 127) // 128)
        splits = _wgrad_splits(tiles, max(1, qkv.rows // 64))
        side = SIDE_WGRAD
        ws_name, bws_name = ("wgrad_ws_side", "bias_ws_side") if side else ("wgrad_ws", "bias_ws")
        self.scratch(ws_name, splits * inner * Cin)
        if has_bias:
            self.scratch(bws_name, splits * inner)
        for i, (w, b) in enumerate(zip(ws, bs)):
            wa = _copy_args(a)
            wa.K = inner
            wa.y, wa.ldy = dout.ptr + 4 * i * ip, dout.ld
            wa.amax_y, wa.amax_out = amax_dy, None
            wa.flags, wa.splits = a.flags & CONV_X_SPLIT, splits
            wa.rowadd, wa.residual, wa.bias, wa.workspace = None, None, None, None
            self._late.append(lambda wa=wa, n=ws_name: setattr(wa, "workspace", self.sptr(n)))
            if has_bias:
                self._late.append(lambda wa=wa, n=bws_name: setattr(wa, "bias_ws", self.sptr(n)))
            self._rec(steps, lib.dp_conv2d_wgrad, wa, "conv wgrad", pinfo)
            steps[-1].side = 2 if side else 0
            ra = L.WgradReduceArgs()
            ra.K, ra.C, ra.R, ra.S, ra.splits = inner, Cin, 1, 1, splits
            ra.dw = self.pgrad(w)
            if self.fused_scores:
                so, si = self._score_views(w, inner, Cin)
                ra.w, ra.score_out, ra.score_in = w.data_ptr(), so.data_ptr(), si.data_ptr()
            self._late.append(lambda ra=ra, n=ws_name: setattr(ra, "workspace", self.sptr(n)))
            if has_bias:
                ra.db = self.pgrad(b)
                self._late.append(lambda ra=ra, n=bws_name: setattr(ra, "bias_ws", self.sptr(n)))
            self._rec(steps, lib.dp_conv2d_wgrad_reduce, ra, "conv wgrad reduce")
            steps[-1].side = 1 if side else 0
        # one dgrad over all 3 inner channels of dy
        da = _copy_args(a)
        da.y, da.ldy = dout.ptr, dout.ld
        da.w = wkc.data_ptr()
        da.w_tc_hi, da.w_tc_lo, da.amax_y = wtc[2].data_ptr(), wtc[3].data_ptr(), amax_dy
        da.flags = 0
        da.amax_out = None
        da.rowadd, da.residual, da.bias = None, None, None
        gx = self.gradof(x)
        da.x, da.ldx = gx.ptr, gx.ld
        it.writes.append((x, lambda init, da=da: setattr(da, "flags", 1 if init else 0),
                          lambda slot, da=da: setattr(da, "amax_out", slot)))
        da.workspace = None
        self._splitk(da, 1)
        self._rec(steps, lib.dp_conv2d_dgrad, da, "conv dgrad", info)
        return parts

    def _splitk(self, a, op: int, name: str = "splitk_ws"):
        """Small-M launches (4x4 .. 16x16 levels) split their K loop over the idle SMs: one shared scratch, bound late."""
        need = int(self.lib.dp_conv_splitk_workspace_floats(C.byref(a), op)) if SPLITK else 0
        if need > 0:
            self.scratch(name, need)
            self._late.append(lambda a=a, n=name: setattr(a, "workspace", self.sptr(n)))

    def _conv_bf16(self, x, w, b, out, stride, pad, rowadd, residual, accumulate_out, need_dx, dx_scratch, seg_out, dx_into):
        """conv() on the bf16 tensor tier: same launch structure and fp32 outputs, operands as bf16 copies."""
        lib = self.lib
        K, Cin = w.shape[0], w.shape[1]
        R = w.shape[2] if w.dim() == 4 else 1
        S = w.shape[3] if w.dim() == 4 else 1
        kc, ck = self._packed_bf16(w)
        xb, ldxb = self._bf16_of(x)
        self.n_bf16_convs += 1
        self._unslotted(out)        # the bf16 kernels do not report max|out|
        a = self._bf_geom(x, out, w, stride, pad)
        a.flags = 1 if accumulate_out else 0
        a.x_bf16, a.ldx = xb.data_ptr(), ldxb
        a.out, a.ld_out = out.ptr, out.ld
        a.w_bf16 = kc.data_ptr()
        a.bias = b.data_ptr() if b is not None else None
        if rowadd is not None:
            a.rowadd, a.ld_rowadd = rowadd.ptr, rowadd.ld
        if residual is not None:
            a.residual, a.ld_res = residual.ptr, residual.ld
        info = f"{Cin}->{K} {R}x{S}" + (f" s{stride}" if stride != 1 else "") + f" @{out.H}x{out.W} bf16"
        if w.dim() == 4:
            self.conv_macs += out.rows * K * Cin * R * S
        else:
            self.lin_macs += out.rows * K * Cin
        self._rec(self.fwd, lib.dp_conv2d_fprop_bf16, a, "conv fprop", info)
        if not self.need_grad:
            return
        it = self._bitem()
        steps = it.steps
        dout = self.gradof(out)
        # 1. bias gradient / per-image sums (fp32, from the fp32 dy)
        if b is not None or seg_out is not None:
            seg = self._colsum_tree(steps, dout.ptr, dout.ld, out.rows, out.H * out.W, K, seg_out)
            if b is not None:
                self._rec(steps, lambda s, seg=seg, b=b, n=x.N: lib.dp_colsum(self.sptr(seg), K, n, K, n, self.pgrad(b), K, 1, s),
                          what="bias grad")
        # 2. dy -> bf16 once for wgrad and dgrad
        lddyb = (K + 7) // 8 * 8
        self.scratch("dy_bf16", (out.rows * lddyb + 1) // 2)
        self._rec(steps, lambda s, p=dout.ptr, ld=dout.ld, r=out.rows: lib.dp_cvt_bf16(p, ld, r, K, self.sptr("dy_bf16"), lddyb, s),
                  what="cvt bf16")
        # 3. wgrad -> split-K workspace -> fixed-order reduce into Parameter.grad
        TC = R * S * Cin
        ctw = lib.dp_bf16_wgrad_ctile(Cin)
        tiles = ((K + 127) // 128) * ((Cin + ctw - 1) // ctw) * R * S
        chunks = max(1, out.rows // 64)
        splits = _wgrad_splits(tiles, chunks)
        self.scratch("wgrad_ws", splits * K * TC)
        wa = _copy_args(a)
        wa.flags, wa.splits, wa.lddy = 0, splits, lddyb
        wa.rowadd, wa.residual, wa.bias, wa.out = None, None, None, None
        self._late.append(lambda wa=wa: (setattr(wa, "dy_bf16", self.sptr("dy_bf16")), setattr(wa, "workspace", self.sptr("wgrad_ws"))))
        self._rec(steps, lib.dp_conv2d_wgrad_bf16, wa, "conv wgrad", info)
        ra = L.WgradReduceArgs()
        ra.K, ra.C, ra.R, ra.S, ra.splits = K, Cin, R, S, splits
        ra.dw = self.pgrad(w)
        self._late.append(lambda ra=ra: setattr(ra, "workspace", self.sptr("wgrad_ws")))
        self._rec(steps, lib.dp_conv2d_wgrad_reduce, ra, "conv wgrad reduce")
        # 4. dgrad
        if need_dx:
            da = _copy_args(a)
            da.lddy, da.w_bf16, da.flags = lddyb, ck.data_ptr(), 0
            da.rowadd, da.residual, da.bias, da.x_bf16 = None, None, None, None
            self._late.append(lambda da=da: setattr(da, "dy_bf16", self.sptr("dy_bf16")))
            if dx_scratch is not None:
                self.scratch(dx_scratch, x.rows * x.C)
                da.ld_out = x.C
                self._late.append(lambda da=da, n=dx_scratch: setattr(da, "out", self.sptr(n)))
            else:
                tgt = dx_into if dx_into is not None else x
                gx = self.gradof(tgt)
                da.out, da.ld_out = gx.ptr, gx.ld
                it.writes.append((tgt, lambda init, da=da: setattr(da, "flags", 1 if init else 0), None))
            self._rec(steps, lib.dp_conv2d_dgrad_bf16, da, "conv dgrad", info)

    GN_MAX_C = 1024      # channels one dp_groupnorm launch handles (256 threads x 4 channel slots); wider tensors are split by groups

    def gn(self, x: View, norm: nn.Module, out: View, silu: bool, dropout_p: float = 0.0, bf16_only: bool = False, groups: Optional[int] = None,
           split_only: bool = False):
        """fwd: out = dropout?(silu?(GN(x))).  Returns the forward argument structs, one per channel part (the backward reuses stats /
        dropout seed).  Groups are independent, so a tensor wider than GN_MAX_C (the LDM's concatenated 1920-channel inputs) runs as
        k launches over k disjoint ranges of whole groups.  split_only (every consumer of `out` is a tensor-core fprop / wgrad that
        takes a split operand, see presplit_ok): write only the fp16 hi / lo' pair the convolutions read, scaled by a bound known in
        advance (dp_groupnorm_fwd_split); the fp32 tensor is left unwritten."""
        lib = self.lib
        G = groups if groups is not None else norm.num_groups
        parts = 1
        while x.C // parts > self.GN_MAX_C:
            parts += 1
            while G % parts or x.C % parts or (x.C // parts) % 4:
                parts += 1
                if parts > G:
                    raise NotImplementedError(f"GroupNorm over {x.C} channels in {G} groups cannot be split into parts of <= {self.GN_MAX_C}")
        if dropout_p > 0:
            self._n_dropout += 1
        yb = ldyb = None
        if bf16_only:   # every consumer of `out` is a bf16 convolution: write the operand directly, skip the fp32 tensor
            yb, ldyb = self._bf_new(out.rows, out.C)
            self._bf_cache[(out.t.data_ptr(), out.off, out.C)] = (yb, ldyb)
        ys = None
        if split_only:
            assert parts == 1 and not bf16_only
            pitch = lib.dp_tc_weight_row(out.C)     # the packed weights' row length: 128-byte box rows for C > 64
            ys = torch.zeros((out.rows, 2, pitch), device=self.dev, dtype=torch.float16)   # pad channels stay zero (finite for the MMA)
            self._keep.append(ys)
            self._split_cache[(out.t.data_ptr(), out.off, out.C)] = (ys, pitch)
            self.split_gn.append(f"{out.N}x{out.H}x{out.W}x{out.C}")
        cp, gp = x.C // parts, G // parts
        args = []
        yslot = self._out_slot(out) if not bf16_only else None   # the tensor-core convolutions that read `out` find its slot filled
        for i in range(parts):
            c0 = i * cp
            a = L.GnArgs()
            a.amax_y = yslot
            a.N, a.HW, a.C, a.G = x.N, x.H * x.W, cp, gp
            a.eps, a.silu = norm.eps, 1 if silu else 0
            a.x, a.ldx, a.y, a.ldy = x.ptr + 4 * c0, x.ld, out.ptr + 4 * c0, out.ld
            if bf16_only:
                a.y, a.y_bf16, a.ldyb = None, yb.data_ptr() + 2 * c0, ldyb
            if split_only:
                a.y = None
            a.gamma, a.beta = norm.weight.data_ptr() + 4 * c0, norm.bias.data_ptr() + 4 * c0
            stats = torch.empty(2 * x.N * gp, device=self.dev, dtype=torch.float32)
            self._keep.append(stats)
            a.mean, a.rstd = stats.data_ptr(), stats.data_ptr() + 4 * x.N * gp
            if dropout_p > 0:
                a.dropout_p = dropout_p
                a.dropout_seed = (0x9E3779B97F4A7C15 * self._n_dropout + 0x632BE59BD9B4E019 * i) & 0xFFFFFFFFFFFFFFFF
                a.dropout_seed_dev = self.dropout_seed_dev.data_ptr()
            self.scratch("gn_ws", (lib.dp_groupnorm_workspace_bytes(a.N, a.HW, a.C, a.G) + 3) // 4)
            self._late.append(lambda a=a: setattr(a, "workspace", self.sptr("gn_ws")))
            if split_only:
                self._rec(self.fwd, lambda ref, s, p=ys.data_ptr(), ld=ys.shape[-1]: lib.dp_groupnorm_fwd_split(ref, p, ld, s), a, "gn fwd")
            else:
                self._rec(self.fwd, lib.dp_groupnorm_fwd, a, "gn fwd")
            args.append((a, c0))
        return args

    def gn_bwd(self, a_fwd, x: View, norm: nn.Module, dy_get: Callable[[], int], lddy: int,
               add2: Optional[View] = None):
        """x.grad (=|+=) GN(+SiLU)(+dropout) backward (+ add2); dgamma/dbeta += .  a_fwd: what gn() returned."""
        lib = self.lib
        gx = self.gradof(x)
        it = self._bitem()
        parts = []
        for a_part, c0 in a_fwd:
            b = _copy_args(a_part)
            b.amax_y, b.amax_dx = None, None
            b.dx, b.lddx, b.lddy = gx.ptr + 4 * c0, gx.ld, lddy
            if add2 is not None:
                b.dx_add2, b.ldadd2 = add2.ptr + 4 * c0, add2.ld
            b.dgamma, b.dbeta = self.pgrad(norm.weight) + 4 * c0, self.pgrad(norm.bias) + 4 * c0
            self._late.append(lambda b=b, c0=c0: (setattr(b, "dy", dy_get() + 4 * c0), setattr(b, "workspace", self.sptr("gn_ws"))))
            parts.append((b, c0))
            side_param = b.HW > 1       # not the one-pixel LayerNorm shapes: their row kernels take dgamma / dbeta from x and dy
            if side_param:              # per-image channel sums in a buffer of this layer's own: dgamma / dbeta leave the dx chain
                fin = torch.empty(2 * b.N * b.C, device=self.dev, dtype=torch.float32)
                self._keep.append(fin)
                b.fin = fin.data_ptr()
            self._rec(it.steps, lib.dp_groupnorm_bwd, b, "gn bwd")
            if side_param:
                self._rec(it.steps, lib.dp_groupnorm_bwd_param, b, "gn bwd param")
                it.steps[-1].side = 2 if SIDE_WGRAD else 0     # only feeds Parameter.grad, like the weight gradients

        def resolve(init, parts=parts, gx=gx):
            if init:
                for b, c0 in parts:
                    b.dx_add, b.ldadd = gx.ptr + 4 * c0, gx.ld
        it.writes.append((x, resolve, lambda slot, parts=parts: [setattr(b, "amax_dx", slot) for b, _ in parts]))

    # ------------------------------------------------------------------ blocks
    def resnet(self, m: ResnetBlock2D, x: View, out: View):
        """ResnetBlock2D.forward — resnet.py:589-639."""
        assert m.output_scale_factor == 1.0, "output_scale_factor != 1 is outside the DDPM configs"
        Cout = m.conv1.out_channels
        p_drop = float(m.dropout.p) if (self.training and m.dropout.p > 0) else 0.0
        a1 = self.new(x.N, x.H, x.W, x.C)
        h1 = self.new(x.N, x.H, x.W, Cout)
        a2 = self.new(x.N, x.H, x.W, Cout)
        tp = self.new(self.B, 1, 1, Cout)
        has_sc = m.conv_shortcut is not None
        da = lambda: self.sptr("da")
        g1 = self.gn(x, m.norm1, a1, silu=True, bf16_only=self.conv_bf16_ok(a1, h1, m.conv1.weight),
                     split_only=self.presplit_ok(x, a1, h1, m.conv1.weight))
        if self.need_grad:
            self.gn_bwd(g1, x, m.norm1, da, x.C, add2=None if has_sc else self.gradof(out))
        # time_emb_proj(silu(temb)) -> per-image row added in conv1's epilogue; its dY are conv1's per-image sums
        self.conv(self.silu_temb, m.time_emb_proj.weight, m.time_emb_proj.bias, tp, pad=0, dy_dense="seg",
                  dx_into=self.silu_temb)
        self.conv(a1, m.conv1.weight, m.conv1.bias, h1, rowadd=tp, seg_out="seg", dx_scratch="da")
        g2 = self.gn(h1, m.norm2, a2, silu=True, dropout_p=p_drop, bf16_only=self.conv_bf16_ok(a2, out, m.conv2.weight),
                     split_only=self.presplit_ok(h1, a2, out, m.conv2.weight))
        if self.need_grad:
            self.gn_bwd(g2, h1, m.norm2, da, Cout)
        if has_sc:
            self.conv(a2, m.conv2.weight, m.conv2.bias, out, dx_scratch="da")
            self.conv(x, m.conv_shortcut.weight, m.conv_shortcut.bias, out, pad=0, accumulate_out=True)
        else:
            self.conv(a2, m.conv2.weight, m.conv2.bias, out, residual=x, dx_scratch="da")

    def attention(self, m: Attention, x: View, out: View):
        """Attention + legacy AttnProcessor — attention_processor.py:415-470 (heads = 1, explicit stale scale)."""
        if m.heads != 1:
            raise NotImplementedError("multi-head attention blocks are outside the DDPM UNet2DModel configs (heads=1)")
        assert m.rescale_output_factor == 1.0
        N, H, W = x.N, x.H, x.W
        inner = m.to_q.out_features
        xn = self.new(N, H, W, x.C)
        lins = (m.to_q, m.to_k, m.to_v)
        fuse = self.qkv_fusable(xn, lins)
        o = self.new(N, H, W, inner)
        if not fuse:
            q, k, v = (self.new(N, H, W, inner) for _ in range(3))
        g = self.gn(x, m.group_norm, xn, silu=False,
                    bf16_only=(not fuse) and all(self.conv_bf16_ok(xn, q, l.weight, 1, 0) for l in lins),
                    split_only=fuse and self.presplit_ok(x, xn, o, m.to_q.weight, 1, 0))
        if self.need_grad:
            self.gn_bwd(g, x, m.group_norm, lambda xn=xn: self.gradof(xn).ptr, x.C,
                        add2=self.gradof(out) if m.residual_connection else None)
        if fuse:
            q, k, v = self.conv_qkv(xn, lins)
        else:
            self.conv(xn, m.to_q.weight, m.to_q.bias, q, pad=0)
            self.conv(xn, m.to_k.weight, m.to_k.bias, k, pad=0)
            self.conv(xn, m.to_v.weight, m.to_v.bias, v, pad=0)
        self._attn_core(q, k, v, o, float(m.scale))
        self.conv(o, m.to_out[0].weight, m.to_out[0].bias, out, pad=0, residual=x if m.residual_connection else None)

    def _attn_core(self, q: View, k: View, v: View, o: View, sc: float):
        """o = softmax(sc * q k^T) v per image over the H*W tokens (single head) and its backward: tcgen05 NT GEMMs when the token
        count is a multiple of 128, the exact SIMT batched GEMM otherwise."""
        lib = self.lib
        N, H, W, inner = q.N, q.H, q.W, q.C
        T = H * W
        P = torch.empty((N, T, T), device=self.dev, dtype=torch.float32)
        self._keep.append(P)

        def gemm(M, Nn, Kd, A, a_rs, a_cs, a_bs, Bp, b_rs, b_cs, b_bs, Cp, ldc, c_bs, alpha):
            ga = L.GemmArgs()
            ga.M, ga.N, ga.Kd, ga.batch = M, Nn, Kd, N
            ga.A, ga.a_rs, ga.a_cs, ga.a_bs = A, a_rs, a_cs, a_bs
            ga.B, ga.b_rs, ga.b_cs, ga.b_bs = Bp, b_rs, b_cs, b_bs
            ga.C, ga.ldc, ga.c_bs, ga.alpha, ga.accumulate = Cp, ldc, c_bs, alpha, 0
            return ga
        Pp = P.data_ptr()
        if self.tc and T % 128 == 0 and inner > 64:      # the NT GEMM rides the 128-wide persistent kernel (N tiles of 128)
            return self._attention_core_tc(N, H, W, T, inner, q, k, v, o, P, sc)
        # S = scale * q k^T ; P = softmax(S) (in place) ; o = P v
        self._rec(self.fwd, lib.dp_gemm_batched, gemm(T, T, inner, q.ptr, q.ld, 1, T * q.ld, k.ptr, 1, k.ld, T * k.ld,
                                                      Pp, T, T * T, sc), "attn qk")
        self._rec(self.fwd, lambda s: lib.dp_softmax_fwd(Pp, Pp, N * T, T, s), what="softmax")
        self._rec(self.fwd, lib.dp_gemm_batched, gemm(T, inner, T, Pp, T, 1, T * T, v.ptr, v.ld, 1, T * v.ld,
                                                      o.ptr, o.ld, T * o.ld, 1.0), "attn pv")
        if self.need_grad:
            dq, dk, dv, do = (self.gradof(t) for t in (q, k, v, o))
            dP = torch.empty_like(P)
            self._keep.append(dP)
            dPp = dP.data_ptr()
            it = self._bitem()
            st = it.steps
            # dV = P^T dO ; dP = dO V^T ; dS = P*(dP - rowsum(dP*P)) ; dQ = scale dS K ; dK = scale dS^T Q
            self._rec(st, lib.dp_gemm_batched, gemm(T, inner, T, Pp, 1, T, T * T, do.ptr, do.ld, 1, T * do.ld,
                                                    dv.ptr, dv.ld, T * dv.ld, 1.0), "attn dV")
            self._rec(st, lib.dp_gemm_batched, gemm(T, T, inner, do.ptr, do.ld, 1, T * do.ld, v.ptr, 1, v.ld, T * v.ld,
                                                    dPp, T, T * T, 1.0), "attn dP")
            self._rec(st, lambda s: lib.dp_softmax_bwd(Pp, dPp, dPp, N * T, T, None, s), what="softmax bwd")
            self._rec(st, lib.dp_gemm_batched, gemm(T, inner, T, dPp, T, 1, T * T, k.ptr, k.ld, 1, T * k.ld,
                                                    dq.ptr, dq.ld, T * dq.ld, sc), "attn dQ")
            self._rec(st, lib.dp_gemm_batched, gemm(T, inner, T, dPp, 1, T, T * T, q.ptr, q.ld, 1, T * q.ld,
                                                    dk.ptr, dk.ld, T * dk.ld, sc), "attn dK")

    def _attention_core_tc(self, N, H, W, T, inner, q, k, v, o, P, sc):
        """softmax(scale q k^T) v and its backward on the tensor-core NT GEMM (dp_gemm_nt_tc): every product is written as
        C = A B^T with a K-contiguous activation A (TMA box of the token grid) and a pre-split fp16 hi/lo' B built by
        dp_split_h3 (optionally transposing); P^T / dS^T come from dp_transpose_batched.
          fwd : S = q k^T          B = split(k)            O  = P v         B = split^T(v)
          bwd : dV = P^T dO        A = P^T, B = split^T(dO)   dP = dO v^T    B = split(v)
                dQ = dS k          B = split^T(k)            dK = dS^T q    A = dS^T, B = split^T(q)
        Operand amax slots: q, k, v, dO come from the kernels that wrote those tensors, P / P^T are bounded by 1, dS by softmax_bwd."""
        lib = self.lib
        i8, t8 = (inner + 7) // 8 * 8, (T + 7) // 8 * 8
        nsplit = N * max(T * i8, inner * t8)          # fp16 elements; the scratch is counted in floats
        self.scratch("att_hi", (nsplit + 1) // 2); self.scratch("att_lo", (nsplit + 1) // 2); self.scratch("att_t", N * T * T)
        Pp = P.data_ptr()

        def split(lst, src: View, slot: int, transpose: int):   # src is an [N][T][inner] activation view
            self._rec(lst, lambda s, p=src.ptr, ld=src.ld, tr=transpose: lib.dp_split_h3(
                p, ld, T * ld, N, T, inner, tr, slot, self.sptr("att_hi"), self.sptr("att_lo"), s), what="attn split")

        def gemm(lst, A_get, ld_a, Kg, Nn, C_ptr, ldc, alpha, what, slot_a, slot_b, slot_out=None):
            ga = L.GemmNtArgs()
            ga.batch, ga.H, ga.W, ga.Kg, ga.N = N, H, W, Kg, Nn
            ga.ld_a, ga.C, ga.ldc, ga.alpha = ld_a, C_ptr, ldc, alpha
            ga.amax_a, ga.amax_b, ga.amax_out = slot_a, slot_b, slot_out
            self._late.append(lambda ga=ga, g=A_get: (setattr(ga, "A", g()), setattr(ga, "b_hi", self.sptr("att_hi")),
                                                      setattr(ga, "b_lo", self.sptr("att_lo"))))
            self._rec(lst, lib.dp_gemm_nt_tc, ga, what)
            return ga

        f = self.fwd
        sq, sk, sv, one = self._x_slot(q), self._x_slot(k), self._x_slot(v), self._one_slot
        split(f, k, sk, 0)
        gemm(f, lambda: q.ptr, q.ld, inner, T, Pp, T, sc, "attn qk (tc)", sq, sk)
        self._rec(f, lambda s: lib.dp_softmax_fwd(Pp, Pp, N * T, T, s), what="softmax")
        split(f, v, sv, 1)
        gemm(f, lambda: Pp, T, T, inner, o.ptr, o.ld, 1.0, "attn pv (tc)", one, sv, self._out_slot(o))
        if not self.need_grad:
            return
        dq, dk, dv, do = (self.gradof(t) for t in (q, k, v, o))
        dP = torch.empty_like(P)
        self._keep.append(dP)
        dPp = dP.data_ptr()
        it = self._bitem()
        st = it.steps
        tptr = lambda: self.sptr("att_t")
        sdo, sds = self._dy_slot(st, o), self._new_slot("dS")
        self._rec(st, lambda s: lib.dp_transpose_batched(Pp, tptr(), N, T, T, s), what="attn transpose")
        split(st, do, sdo, 1)
        g_dv = gemm(st, tptr, T, T, inner, dv.ptr, dv.ld, 1.0, "attn dV (tc)", one, sdo)
        split(st, v, sv, 0)
        gemm(st, lambda: do.ptr, do.ld, inner, T, dPp, T, 1.0, "attn dP (tc)", sdo, sv)
        self._rec(st, lambda s: lib.dp_softmax_bwd(Pp, dPp, dPp, N * T, T, sds, s), what="softmax bwd")
        split(st, k, sk, 1)
        g_dq = gemm(st, lambda: dPp, T, T, inner, dq.ptr, dq.ld, sc, "attn dQ (tc)", sds, sk)
        self._rec(st, lambda s: lib.dp_transpose_batched(dPp, tptr(), N, T, T, s), what="attn transpose")
        split(st, q, sq, 1)
        g_dk = gemm(st, tptr, T, T, inner, dk.ptr, dk.ld, sc, "attn dK (tc)", sds, sq)
        # dq / dk / dv are written (=) exactly once, by these GEMMs, which report their maxima to the 1x1 convolutions' dy slots
        for t_, g_ in ((q, g_dq), (k, g_dk), (v, g_dv)):
            it.writes.append((t_, lambda init: None, lambda slot, g_=g_: setattr(g_, "amax_out", slot)))

    # ------------------------------------------------------------------ whole network
    def _build(self):
        if hasattr(self.model, "input_blocks"):      # latent-diffusion UNetModel (ldm.py)
            return self._build_ldm()
        m, lib = self.model, self.lib
        B, H, W = self.B, self.H, self.W
        cfg = m.config
        self._setup_param_grads()
        # ---- inputs + timestep embedding chain (embeddings.py:22-62, 200-212)
        self.t_dev = torch.zeros(B, device=self.dev, dtype=torch.int64)
        # network input / output live in buffers padded to a multiple of 4 channels (zero pad) so their pixel stride is
        # 16-byte aligned: TMA can then read them and conv_in / conv_out run on the tensor-core path too
        def padded(c):
            t = torch.zeros((B, H, W, (c + 3) // 4 * 4), device=self.dev, dtype=torch.float32)
            self._keep.append(t)
            return View(t, 0, c)
        self.x_in = padded(cfg.in_channels)
        half = cfg.block_out_channels[0] // 2
        self.freqs = sinusoidal_frequencies(cfg.block_out_channels[0], cfg.freq_shift).to(self.dev)
        te = m.time_embedding
        temb0 = self.new(B, 1, 1, 2 * half)
        l1, s1 = self.new(B, 1, 1, te.linear_1.out_features), self.new(B, 1, 1, te.linear_1.out_features)
        emb = self.new(B, 1, 1, te.linear_2.out_features)
        self.silu_temb = self.new(B, 1, 1, emb.C)
        self._rec(self.fwd, lambda s: lib.dp_timestep_embedding(self.t_dev.data_ptr(), self.freqs.data_ptr(), temb0.ptr, B, half,
                                                                1 if cfg.flip_sin_to_cos else 0, s), what="temb")
        self.conv(temb0, te.linear_1.weight, te.linear_1.bias, l1, pad=0, need_dx=False)
        n1, n2 = B * l1.ld, B * emb.ld   # flat extents incl. pitch padding (pads are never read as channels)
        self._rec(self.fwd, lambda s: lib.dp_silu_fwd(l1.ptr, s1.ptr, n1, s), what="silu")
        if self.need_grad:
            self._rec(self._bitem().steps, lambda s: lib.dp_silu_bwd(l1.ptr, self.gradof(s1).ptr, self.gradof(l1).ptr, n1, 0, s),
                      what="silu bwd")
        self.conv(s1, te.linear_2.weight, te.linear_2.bias, emb, pad=0)
        self._rec(self.fwd, lambda s: lib.dp_silu_fwd(emb.ptr, self.silu_temb.ptr, n2, s), what="silu")
        if self.need_grad:
            self._rec(self._bitem().steps,
                      lambda s: lib.dp_silu_bwd(emb.ptr, self.gradof(self.silu_temb).ptr, self.gradof(emb).ptr, n2, 0, s),
                      what="silu bwd")
            self.bwd[-1].steps[-1].join = True     # d silu(temb) is complete only when the side stream's time-embedding branches are

        # ---- skip/concat geometry: every skip lives in the upper channel range of its consumer's concat buffer
        skip_shapes = []
        ch, hh, ww = m.conv_in.out_channels, H, W
        skip_shapes.append((hh, ww, ch))
        for blk in m.down_blocks:
            for r in blk.resnets:
                ch = r.conv2.out_channels
                skip_shapes.append((hh, ww, ch))
            if blk.downsamplers is not None:
                ch = blk.downsamplers[0].conv.out_channels
                hh, ww = hh // 2, ww // 2
                skip_shapes.append((hh, ww, ch))
        consumers = [r for blk in m.up_blocks for r in blk.resnets]
        assert len(consumers) == len(skip_shapes)
        cat_total = [0] * len(skip_shapes)
        for j, r in enumerate(consumers):
            cat_total[len(skip_shapes) - 1 - j] = r.norm1.num_channels
        counter = [0]

        def new_skip() -> View:
            i = counter[0]
            counter[0] += 1
            hh_, ww_, c = skip_shapes[i]
            buf = self.new(B, hh_, ww_, cat_total[i])
            assert cat_total[i] - c > 0
            return View(buf.t, cat_total[i] - c, c)

        def h_half(skip: View) -> View:   # channels [0, C_h) of the skip's concat buffer
            return View(skip.t, 0, skip.off)

        def cat_of(skip: View) -> View:
            return View(skip.t, 0, skip.off + skip.C)

        x = new_skip()
        self.conv(self.x_in, m.conv_in.weight, m.conv_in.bias, x, need_dx=False)
        skips = [x]
        for blk in m.down_blocks:
            has_attn = getattr(blk, "has_attention", False)
            for j, r in enumerate(blk.resnets):
                if has_attn:
                    mid = self.new(x.N, x.H, x.W, r.conv2.out_channels)
                    self.resnet(r, x, mid)
                    y = new_skip()
                    self.attention(blk.attentions[j], mid, y)
                else:
                    y = new_skip()
                    self.resnet(r, x, y)
                x = y
                skips.append(x)
            if blk.downsamplers is not None:
                d: Downsample2D = blk.downsamplers[0]
                y = new_skip()
                self.conv(x, d.conv.weight, d.conv.bias, y, stride=2, pad=d.padding)  # pad 0 => F.pad(0,1,0,1) folded
                x = y
                skips.append(x)

        # ---- mid (its last op writes straight into the h-half of the first concat)
        mb = m.mid_block
        y = self.new(x.N, x.H, x.W, x.C)
        self.resnet(mb.resnets[0], x, y)
        x = y
        if mb.attentions[0] is not None:
            y = self.new(x.N, x.H, x.W, x.C)
            self.attention(mb.attentions[0], x, y)
            x = y
        dest = h_half(skips[-1])
        assert dest.C == x.C and dest.H == x.H, (dest.C, x.C)
        self.resnet(mb.resnets[1], x, dest)

        # ---- up
        nblk = len(m.up_blocks)
        for bi, blk in enumerate(m.up_blocks):
            has_attn = getattr(blk, "has_attention", False)
            nres = len(blk.resnets)
            for j, r in enumerate(blk.resnets):
                cat = cat_of(skips.pop())
                if j < nres - 1:
                    dest = h_half(skips[-1])
                else:  # feeds the upsampler or the output head
                    dest = self.new(cat.N, cat.H, cat.W, r.conv2.out_channels)
                    assert blk.upsamplers is not None or bi == nblk - 1
                if has_attn:
                    mid = self.new(cat.N, cat.H, cat.W, r.conv2.out_channels)
                    self.resnet(r, cat, mid)
                    self.attention(blk.attentions[j], mid, dest)
                else:
                    self.resnet(r, cat, dest)
                x = dest
            if blk.upsamplers is not None:
                u: Upsample2D = blk.upsamplers[0]
                up = self.new(x.N, 2 * x.H, 2 * x.W, x.C)
                xx = x
                self._rec(self.fwd, lambda s, xx=xx, up=up: lib.dp_upsample2x_fwd(xx.ptr, xx.ld, up.ptr, up.ld, xx.N, xx.H, xx.W, xx.C, s),
                          what="upsample")
                self._alias_slot(up, xx)
                if self.need_grad:
                    it = self._bitem()
                    accf = [0]
                    it.writes.append((xx, lambda init, accf=accf: accf.__setitem__(0, 1 if init else 0), None))
                    self._rec(it.steps, lambda s, xx=xx, up=up, accf=accf: lib.dp_upsample2x_bwd(
                        self.gradof(up).ptr, up.ld, self.gradof(xx).ptr, self.gradof(xx).ld, xx.N, xx.H, xx.W, xx.C, accf[0], s),
                        what="upsample bwd")
                dest = h_half(skips[-1])
                self.conv(up, u.conv.weight, u.conv.bias, dest)
                x = dest
        assert not skips
        # ---- out head (unet_2d.py:302-304)
        a = self.new(x.N, x.H, x.W, x.C)
        g = self.gn(x, m.conv_norm_out, a, silu=True)
        if self.need_grad:
            self.gn_bwd(g, x, m.conv_norm_out, lambda: self.sptr("da"), x.C)
        self.y_out = padded(cfg.out_channels)
        self.gradof(self.y_out).t.zero_()
        self.conv(a, m.conv_out.weight, m.conv_out.bias, self.y_out, dx_scratch="da")

        self._finalize_build()

    def _finalize_build(self):
        # ---- allocate shared scratch, bind late pointers, resolve (=|+=) of every gradient write in EXECUTION order
        for name, n in self._scratch_need.items():
            self._scratch[name] = torch.empty(max(n, 1), device=self.dev, dtype=torch.float32)
        for fix in self._late:
            fix()
        self._late.clear()
        if self.need_grad:
            self.g_mark(self.silu_temb)   # zeroed at backward start; every resnet accumulates into it
            self.g_mark(self.y_out)       # loaded from the loss gradient
            for it in reversed(self.bwd):
                for view, setter, _ in it.writes:
                    setter(self.g_is_init(view))
                    self.g_mark(view)
            # gradient amax slots: when every writer of a tensor's gradient reports its own maximum, the consumers' dp_amax launches go
            writers: Dict[int, list] = {}
            for it in self.bwd:
                for view, _, amax_setter in it.writes:
                    writers.setdefault(view.t.data_ptr(), []).append(amax_setter)
            for key, rec in self._bslot.items():
                ws = writers.get(key, [])
                if ws and all(w is not None for w in ws):
                    for w in ws:
                        w(rec["slot"])
                    for flag in rec["flags"]:
                        flag[0] = False
        self._packed_version = None
        if self._n_slots:       # every activation / gradient amax slot starts the pass at zero
            zero: List[Step] = []
            n, ptr, lib = self._n_slots, self._slots.data_ptr(), self.lib
            self._rec(zero, lambda s: lib.dp_zero_u32(ptr, n, s), what="amax zero")
            self.fwd.insert(0, zero[0])
        self.bwd_steps: List[Step] = [f for it in reversed(self.bwd) for f in it.steps]
        self._has_side = any(getattr(f, "side", 0) for f in self.bwd_steps)
        self._side_stream = None

    # ------------------------------------------------------------------ latent-diffusion UNetModel (ldm.py; BASELINE configs[4])
    def _tokens(self, v: View) -> View:
        """The same storage seen as N*H*W one-pixel images (LayerNorm = GroupNorm with one group over the channels of a token)."""
        return View(v.t.view(v.rows, 1, 1, v.ld), v.off, v.C)

    def layernorm(self, x: View, ln: nn.LayerNorm, out: View, add2: Optional[View] = None):
        """nn.LayerNorm over the channel dimension of every token (attention.py:204-206), forward + backward (dx += add2: the residual
        branch's gradient)."""
        xt, ot = self._tokens(x), self._tokens(out)
        g = self.gn(xt, ln, ot, silu=False, groups=1)
        if self.need_grad:
            self.gn_bwd(g, xt, ln, lambda o=out: self.gradof(o).ptr, self.gradof(out).ld, add2=add2)

    def transformer_block(self, blk, x: View) -> View:
        """BasicTransformerBlock (attention.py:196-212) for a one-token context:
             x2 = attn1(LN1(x)) + x + attn2(LN2(.), context)      x3 = ff(LN3(x2)) + x2
        Cross-attention over ONE context token is softmax over a single logit = 1, so attn2(., c) = to_out(to_v(c)) for every query token
        whatever to_q / to_k / LN2 hold: a per-image row, added in the epilogue of attn1's output projection.  Their gradients are
        exactly zero in the reference as well (softmax backward of a single element), so nothing is launched for them."""
        lib = self.lib
        N, H, W, d = x.N, x.H, x.W, x.C
        a1, a2, ff = blk.attn1, blk.attn2, blk.ff
        if a1.heads != 1 or a2.heads != 1:
            raise NotImplementedError("multi-head transformer blocks (cin256-v2 uses num_heads = 1)")
        if self.ctx_in.H * self.ctx_in.W != 1:
            raise NotImplementedError("cross-attention over more than one context token")
        inner = a1.to_q.out_features
        # cross-attention contribution (per image): octx = to_out(to_v(context))
        vctx, octx = self.new(self.B, 1, 1, a2.to_v.out_features), self.new(self.B, 1, 1, d)
        self.conv(self.ctx_in, a2.to_v.weight, None, vctx, pad=0, need_dx=False)
        self.conv(vctx, a2.to_out[0].weight, a2.to_out[0].bias, octx, pad=0, dy_dense="seg_ctx")
        # self-attention
        x2 = self.new(N, H, W, d)
        h1 = self.new(N, H, W, d)
        self.layernorm(x, blk.norm1, h1, add2=self.gradof(x2))
        o = self.new(N, H, W, inner)
        lins = (a1.to_q, a1.to_k, a1.to_v)
        if all(l.bias is None for l in lins) and self.qkv_fusable(h1, lins):
            q, k, v = self.conv_qkv(h1, lins)
        else:
            q, k, v = (self.new(N, H, W, inner) for _ in range(3))
            self.conv(h1, a1.to_q.weight, None, q, pad=0)
            self.conv(h1, a1.to_k.weight, None, k, pad=0)
            self.conv(h1, a1.to_v.weight, None, v, pad=0)
        self._attn_core(q, k, v, o, float(a1.scale))
        self.conv(o, a1.to_out[0].weight, a1.to_out[0].bias, x2, pad=0, residual=x, rowadd=octx, seg_out="seg_ctx")
        # GEGLU feed-forward
        x3 = self.new(N, H, W, d)
        h3 = self.new(N, H, W, d)
        self.layernorm(x2, blk.norm3, h3, add2=self.gradof(x3))
        proj, lin2 = ff.net[0].proj, ff.net[2]
        I = lin2.in_features
        u, gg = self.new(N, H, W, 2 * I), self.new(N, H, W, I)
        self.conv(h3, proj.weight, proj.bias, u, pad=0)
        rows = u.rows
        self._rec(self.fwd, lambda s: lib.dp_geglu_fwd(u.ptr, u.ld, gg.ptr, gg.ld, rows, I, s), what="geglu")
        if self.need_grad:
            it = self._bitem()
            it.writes.append((u, lambda init: None, None))        # du is written (=) exactly once, by this op
            self._rec(it.steps, lambda s: lib.dp_geglu_bwd(u.ptr, u.ld, self.gradof(gg).ptr, gg.ld, self.gradof(u).ptr, u.ld, rows, I, s),
                      what="geglu bwd")
        self.conv(gg, lin2.weight, lin2.bias, x3, pad=0, residual=x2)
        return x3

    def spatial_transformer(self, m, x: View, out: View):
        """SpatialTransformer (attention.py:215-257): GroupNorm(32, eps 1e-6) -> 1x1 proj_in -> transformer blocks over the H*W tokens
        -> 1x1 proj_out ; + x."""
        h = self.new(x.N, x.H, x.W, m.proj_in.out_channels)
        xn = self.new(x.N, x.H, x.W, x.C)
        g = self.gn(x, m.norm, xn, silu=False, bf16_only=self.conv_bf16_ok(xn, h, m.proj_in.weight, 1, 0),
                    split_only=self.presplit_ok(x, xn, h, m.proj_in.weight, 1, 0))
        if self.need_grad:
            self.gn_bwd(g, x, m.norm, lambda xn=xn: self.gradof(xn).ptr, x.C, add2=self.gradof(out))
        self.conv(xn, m.proj_in.weight, m.proj_in.bias, h, pad=0)
        for blk in m.transformer_blocks:
            h = self.transformer_block(blk, h)
        self.conv(h, m.proj_out.weight, m.proj_out.bias, out, pad=0, residual=x)

    def _build_ldm(self):
        """UNetModel.forward (openaimodel.py:710-742) as a static launch plan; same HBM conventions as the DDPM UNet (NHWC fp32 views,
        zero-copy skip concatenation, epilogue-fused bias / embedding row / residual)."""
        from types import SimpleNamespace as NS
        m, lib = self.model, self.lib
        B, H, W = self.B, self.H, self.W
        cfg = m.config
        self._setup_param_grads()
        self.t_dev = torch.zeros(B, device=self.dev, dtype=torch.int64)

        def padded(n, h, w, c):
            t = torch.zeros((n, h, w, (c + 3) // 4 * 4), device=self.dev, dtype=torch.float32)
            self._keep.append(t)
            return View(t, 0, c)
        self.x_in = padded(B, H, W, cfg.in_channels)
        self.ctx_in = padded(B, 1, 1, cfg.context_dim)
        mc = cfg.model_channels
        half = mc // 2
        self.freqs = sinusoidal_frequencies(mc, 0).to(self.dev)        # exp(-ln(1e4) i / half), util.py:160-162
        temb0 = self.new(B, 1, 1, 2 * half)
        te1, te2 = m.time_embed[0], m.time_embed[2]
        l1, s1 = self.new(B, 1, 1, te1.out_features), self.new(B, 1, 1, te1.out_features)
        emb = self.new(B, 1, 1, te2.out_features)
        self.silu_temb = self.new(B, 1, 1, emb.C)
        # cos | sin order (util.py:164) = the DDPM kernel with the halves flipped
        self._rec(self.fwd, lambda s: lib.dp_timestep_embedding(self.t_dev.data_ptr(), self.freqs.data_ptr(), temb0.ptr, B, half, 1, s), what="temb")
        self.conv(temb0, te1.weight, te1.bias, l1, pad=0, need_dx=False)
        n1, n2 = B * l1.ld, B * emb.ld
        self._rec(self.fwd, lambda s: lib.dp_silu_fwd(l1.ptr, s1.ptr, n1, s), what="silu")
        if self.need_grad:
            self._rec(self._bitem().steps, lambda s: lib.dp_silu_bwd(l1.ptr, self.gradof(s1).ptr, self.gradof(l1).ptr, n1, 0, s), what="silu bwd")
        self.conv(s1, te2.weight, te2.bias, emb, pad=0)
        self._rec(self.fwd, lambda s: lib.dp_silu_fwd(emb.ptr, self.silu_temb.ptr, n2, s), what="silu")
        if self.need_grad:
            self._rec(self._bitem().steps,
                      lambda s: lib.dp_silu_bwd(emb.ptr, self.gradof(self.silu_temb).ptr, self.gradof(emb).ptr, n2, 0, s), what="silu bwd")
            self.bwd[-1].steps[-1].join = True     # d silu(temb) is complete only when the side stream's time-embedding branches are

        def as_resnet(rb):     # ResBlock (openaimodel.py:163-275) in the attribute vocabulary of Plan.resnet()
            sk = rb.skip_connection
            return NS(norm1=rb.in_layers[0], conv1=rb.in_layers[2], time_emb_proj=rb.emb_layers[1], norm2=rb.out_layers[0],
                      dropout=rb.out_layers[2], conv2=rb.out_layers[3], conv_shortcut=sk if isinstance(sk, nn.Conv2d) else None,
                      output_scale_factor=1.0)

        # ---- skip geometry: the output of every input block is concatenated (as the UPPER channels) in front of one output block
        shapes, ch, hh, ww = [], None, H, W
        for blk in m.input_blocks:
            for layer in blk:
                if isinstance(layer, nn.Conv2d):
                    ch = layer.out_channels
                elif hasattr(layer, "in_layers"):
                    ch = layer.out_channels
                elif hasattr(layer, "op"):
                    ch, hh, ww = layer.op.out_channels, hh // 2, ww // 2
            shapes.append((hh, ww, ch))
        consumers = [blk[0] for blk in m.output_blocks]
        assert len(consumers) == len(shapes)
        cat_total = [0] * len(shapes)
        for j, rb in enumerate(consumers):
            cat_total[len(shapes) - 1 - j] = rb.in_layers[0].num_channels
        counter = [0]

        def new_skip() -> View:
            i = counter[0]
            counter[0] += 1
            hh_, ww_, c = shapes[i]
            buf = self.new(B, hh_, ww_, cat_total[i])
            assert cat_total[i] - c > 0
            return View(buf.t, cat_total[i] - c, c)
        h_half = lambda skip: View(skip.t, 0, skip.off)
        cat_of = lambda skip: View(skip.t, 0, skip.off + skip.C)

        def run_layers(layers, x: View, dest: View) -> View:
            """A TimestepEmbedSequential: the last layer writes `dest`, the others fresh buffers."""
            layers = list(layers)
            for li, layer in enumerate(layers):
                last = li == len(layers) - 1
                if isinstance(layer, nn.Conv2d):
                    y = dest
                    self.conv(x, layer.weight, layer.bias, y, need_dx=False)
                elif hasattr(layer, "in_layers"):
                    y = dest if last else self.new(x.N, x.H, x.W, layer.out_channels)
                    self.resnet(as_resnet(layer), x, y)
                elif hasattr(layer, "transformer_blocks"):
                    y = dest if last else self.new(x.N, x.H, x.W, x.C)
                    self.spatial_transformer(layer, x, y)
                elif hasattr(layer, "op"):
                    y = dest
                    self.conv(x, layer.op.weight, layer.op.bias, y, stride=2, pad=1)
                elif hasattr(layer, "conv"):      # Upsample: nearest x2 then 3x3 conv
                    up = self.new(x.N, 2 * x.H, 2 * x.W, x.C)
                    xx = x
                    self._rec(self.fwd, lambda s, xx=xx, up=up: lib.dp_upsample2x_fwd(xx.ptr, xx.ld, up.ptr, up.ld, xx.N, xx.H, xx.W, xx.C, s),
                              what="upsample")
                    self._alias_slot(up, xx)
                    if self.need_grad:
                        it = self._bitem()
                        accf = [0]
                        it.writes.append((xx, lambda init, accf=accf: accf.__setitem__(0, 1 if init else 0), None))
                        self._rec(it.steps, lambda s, xx=xx, up=up, accf=accf: lib.dp_upsample2x_bwd(
                            self.gradof(up).ptr, up.ld, self.gradof(xx).ptr, self.gradof(xx).ld, xx.N, xx.H, xx.W, xx.C, accf[0], s),
                            what="upsample bwd")
                    y = dest
                    self.conv(up, layer.conv.weight, layer.conv.bias, y)
                else:
                    raise NotImplementedError(type(layer).__name__)
                x = y
            return x

        x, skips = self.x_in, []
        for blk in m.input_blocks:
            x = run_layers(blk, x, new_skip())
            skips.append(x)
        # the middle block's last layer writes straight into the h-half of the first concatenation
        dest = h_half(skips[-1])
        assert dest.C == x.C and dest.H == x.H, (dest.C, x.C)
        x = run_layers(m.middle_block, x, dest)
        nblk = len(m.output_blocks)
        for bi, blk in enumerate(m.output_blocks):
            cat = cat_of(skips.pop())
            layers = list(blk)
            out_ch = layers[0].out_channels
            up = hasattr(layers[-1], "conv") and not hasattr(layers[-1], "in_layers")
            if skips:
                dest = h_half(skips[-1])
                assert dest.C == out_ch and dest.H == cat.H * (2 if up else 1), (bi, dest.C, out_ch, dest.H, cat.H)
            else:
                dest = self.new(cat.N, cat.H, cat.W, out_ch)
            x = run_layers(layers, cat, dest)
        assert not skips
        a = self.new(x.N, x.H, x.W, x.C)
        g = self.gn(x, m.out[0], a, silu=True)
        if self.need_grad:
            self.gn_bwd(g, x, m.out[0], lambda: self.sptr("da"), x.C)
        self.y_out = padded(B, H, W, cfg.out_channels)
        self.gradof(self.y_out).t.zero_()
        self.conv(a, m.out[2].weight, m.out[2].bias, self.y_out, dx_scratch="da")
        self._finalize_build()

    def load_context(self, context: torch.Tensor):
        """context: (B, 1, context_dim) fp32 -> the plan's conditioning buffer (cross-attention input; no gradient)."""
        c = context.reshape(self.B, -1).to(device=self.dev, dtype=torch.float32)
        assert c.shape[1] == self.ctx_in.C, (tuple(context.shape), self.ctx_in.C)
        self.ctx_in.t.view(self.B, -1)[:, :self.ctx_in.C].copy_(c, non_blocking=True)

    # ------------------------------------------------------------------ execution
    def run_pack(self, s: Optional[int] = None):
        s = _stream() if s is None else s
        for f in self.pack:
            f(s)

    def ensure_packed(self, force: bool = False):
        v = self.weight_version()
        if force or v != self._packed_version:
            self.run_pack()
            self._packed_version = v

    def check_current(self):
        """Raises when the model's parameters were replaced (pruned / re-pointed) after this plan was built: its launch lists
        still address the old Parameter storage and would silently accumulate into an arena that is no longer `.grad`."""
        if tuple((p.data_ptr(), tuple(p.shape)) for p in self.model.parameters()) != self.signature():
            raise RuntimeError("diff_pruning_b200: the model's parameters were replaced after this plan was built "
                               "(pruning / load / re-pointing); create a new TaylorScorer / FinetuneStepper")

    def run_forward(self, s: Optional[int] = None):
        s = _stream() if s is None else s
        for f in self.fwd:
            f(s)

    def run_backward(self, s: Optional[int] = None):
        s = _stream() if s is None else s
        self.gradof(self.silu_temb).t.zero_()
        main = torch.cuda.current_stream(self.dev)
        if not self._has_side or main.cuda_stream != s or self.audit:
            for f in self.bwd_steps:
                f(s)
            return
        if self._side_stream is None:
            self._side_stream = torch.cuda.Stream(device=self.dev)
        side = self._side_stream
        s2 = side.cuda_stream
        for f in self.bwd_steps:
            k = getattr(f, "side", 0)
            if k == 2:                  # dy (and its amax slot) are final at this point of the main stream
                side.wait_stream(main)
            if k:
                f(s2)
            else:
                if getattr(f, "join", False):
                    main.wait_stream(side)
                f(s)
        main.wait_stream(side)          # Parameter.grad is complete when the pass ends (also closes a CUDA-graph capture's fork)

    def load_input_nchw(self, sample: torch.Tensor, timesteps: torch.Tensor):
        sample = sample.contiguous()
        self.t_dev.copy_(timesteps.to(torch.int64), non_blocking=True)
        L.check(self.lib.dp_nchw_to_nhwc(sample.data_ptr(), self.x_in.ptr, self.x_in.ld, self.B, self.x_in.C, self.H, self.W,
                                         _stream()), "nchw->nhwc")

    def output_nchw(self) -> torch.Tensor:
        out = torch.empty((self.B, self.y_out.C, self.H, self.W), device=self.dev, dtype=torch.float32)
        L.check(self.lib.dp_nhwc_to_nchw(self.y_out.ptr, self.y_out.ld, out.data_ptr(), self.B, self.y_out.C, self.H, self.W, 0,
                                         _stream()), "nhwc->nchw")
        return out

    def load_grad_nchw(self, gout: torch.Tensor):
        gout = gout.contiguous()
        gy = self.gradof(self.y_out)
        L.check(self.lib.dp_nchw_to_nhwc(gout.data_ptr(), gy.ptr, gy.ld, self.B, gy.C, self.H, self.W, _stream()),
                "grad nchw->nhwc")

    def bytes_allocated(self) -> int:
        n = sum(t.numel() * t.element_size() for t in self._keep if isinstance(t, torch.Tensor))
        n += sum(t.numel() * 4 for t in self._gbuf.values()) + sum(t.numel() * 4 for t in self._scratch.values())
        n += sum(a.numel() * 8 + (sum(t.numel() * 2 for t in tc[:4]) if tc else 0) for a, _, tc in self._packs.values())
        n += self.grad_arena.numel() * 4
        return n


# ----------------------------------------------------------------------------------------------------------
# autograd boundary: the whole UNet is ONE node, parameters are listed as inputs so backward() fires, and the
# engine writes Parameter.grad itself (accumulating), exactly what `loss.backward()` does at ddpm_prune.py:102.
# ----------------------------------------------------------------------------------------------------------
class _UNetFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, sample, timesteps, plan, *params):
        plan.load_input_nchw(sample, timesteps)
        plan.run_forward()
        ctx.plan = plan
        plan.generation += 1          # activations live in the plan's buffers: a later forward overwrites them
        ctx.generation = plan.generation
        return plan.output_nchw()

    @staticmethod
    def backward(ctx, gout):
        plan: Plan = ctx.plan
        if plan.generation != ctx.generation:
            raise RuntimeError("diff_pruning_b200: backward() of a UNet forward whose activations were overwritten by a later forward "
                               "of the same (batch, resolution) plan (two forwards before one backward: gradient accumulation over "
                               "micro-batches, or sampling between forward and backward).  Call backward() before the next forward.")
        plan.attach_grads()
        plan.load_grad_nchw(gout)
        plan.run_backward()
        return (None, None, None) + (None,) * len(plan.params)


BF16_TIER = True   # conv_bf16.cu is part of this build (bench.py reports the bf16 finetune leg separately)


def get_plan(model: UNet2DModel, batch: int, H: int, W: int, device, need_grad: bool, fused_scores: bool = False,
             compute: str = "fp32") -> Plan:
    cache = model.__dict__.setdefault("_dpb200_plans", {})
    training = bool(model.training)
    drop = tuple(float(mod.p) for mod in model.modules() if isinstance(mod, nn.Dropout)) if training else ()
    key = (batch, H, W, str(device), need_grad, training, fused_scores, drop, compute)   # dropout rates are baked into the launch plan
    plan = cache.get(key)
    sig = tuple((p.data_ptr(), tuple(p.shape)) for p in model.parameters())
    if plan is None or plan.signature() != sig:
        if plan is not None or any(pl.signature() != sig for pl in cache.values()):
            cache.clear()  # weights were replaced (e.g. pruned): every cached plan is stale
        plan = Plan(model, batch, H, W, device, training=training, need_grad=need_grad, fused_scores=fused_scores, compute=compute)
        cache[key] = plan
    return plan


def unet_apply(model, sample: torch.Tensor, timesteps: torch.Tensor, context: Optional[torch.Tensor] = None) -> torch.Tensor:
    """UNet2DModel.forward on CUDA (models.py).  unet_2d.py:219-316."""
    if sample.dtype != torch.float32:
        raise TypeError("diff_pruning_b200 engine computes in fp32; got %s" % sample.dtype)
    B, Cc, H, W = sample.shape
    need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in model.parameters())
    if need_grad and sample.requires_grad:
        raise RuntimeError("diff_pruning_b200: the engine does not produce d(loss)/d(sample) (the reference loops never need it: "
                           "noisy images are leaves without grad, ddpm_prune.py:99-100); detach the input")
    # `accelerator.prepare(model)` with mixed_precision="bf16" (compat/accelerate) selects the bf16 tier for TRAINING forwards, the
    # analogue of running the forward under torch.autocast(bfloat16) at ddpm_train.py:255-261,458
    compute = model.__dict__.get("_dpb200_compute", "fp32") if (need_grad and model.training) else "fp32"
    plan = get_plan(model, B, H, W, sample.device, need_grad, compute=compute)
    # Packed weight copies: this module-forward path cannot see every way weights get written (`param.data.copy_` leaves no trace),
    # so it re-packs on EVERY call (~230 small launches, < 1 ms at C1) unless the caller froze the weights for a loop
    # (frozen_weights(): the DDIM pipelines) — the explicit TaylorScorer / FinetuneStepper APIs manage their own packs.
    plan.ensure_packed(force=not model.__dict__.get("_dpb200_frozen", False))
    if plan.training and plan._n_dropout:
        plan._calls += 1                # a fresh dropout stream per forward (and per rank), like torch's advancing Philox offset
        plan.dropout_seed_dev.fill_(_dropout_seed(plan._calls))
    if hasattr(plan, "ctx_in"):
        if context is None:
            raise ValueError("the LDM UNetModel is cross-attention conditioned: pass context=(B, 1, context_dim)")
        plan.load_context(context)
    if need_grad:
        return _UNetFunction.apply(sample, timesteps, plan, *plan.params)
    plan.load_input_nchw(sample, timesteps)
    plan.run_forward()
    return plan.output_nchw()


def _dropout_seed(step: int) -> int:
    """Per-step dropout seed, decorrelated across data-parallel ranks (every rank must draw its own masks)."""
    rank = 0
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            rank = dist.get_rank()
    except Exception:
        rank = 0
    return (0x5DEECE66D * step + 0x9E3779B97F4A7C15 * rank) & 0x7FFFFFFFFFFF


def invalidate_packs(model: UNet2DModel) -> None:
    """Tell every cached plan of `model` that its weights changed through a path torch's version counters do not see
    (`param.data.copy_`, raw-pointer kernels).  The next forward of any plan re-packs."""
    model.__dict__["_dpb200_weights_epoch"] = model.__dict__.get("_dpb200_weights_epoch", 0) + 1


class frozen_weights:
    """`with frozen_weights(model):` — weights are packed once on entry and the per-call re-pack of the module-forward path is
    skipped inside (sampling loops: 100 forwards on fixed weights)."""

    def __init__(self, model: UNet2DModel):
        self.model = model

    def __enter__(self):
        invalidate_packs(self.model)            # the first forward inside packs whatever the weights are NOW
        self.prev = self.model.__dict__.get("_dpb200_frozen", False)
        self.model.__dict__["_dpb200_frozen"] = True
        return self

    def __exit__(self, *exc):
        self.model.__dict__["_dpb200_frozen"] = self.prev
        return False


def add_noise_cuda(sched, x0: torch.Tensor, noise: torch.Tensor, timesteps: torch.Tensor) -> torch.Tensor:
    """DDPMScheduler.add_noise on CUDA — scheduling_ddpm.py:408-429."""
    lib = L.load()
    dev = x0.device
    tab = sched._dev_tables.get(str(dev))
    if tab is None:
        tab = sched.alphas_cumprod.to(dev).contiguous()
        sched._dev_tables[str(dev)] = tab
    x0c, nz = x0.contiguous(), noise.contiguous()
    t = timesteps.to(device=dev, dtype=torch.int64).contiguous()
    out = torch.empty_like(x0c)
    B, Cc, H, W = x0c.shape
    L.check(lib.dp_add_noise(x0c.data_ptr(), nz.data_ptr(), t.data_ptr(), tab.data_ptr(), out.data_ptr(), B, Cc, H, W, 0, 0, _stream()),
            "add_noise")
    return out
