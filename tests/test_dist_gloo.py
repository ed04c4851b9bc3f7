"""world_size-2 gloo test of the timestep-sharding rule (SURVEY.md §8(e)): rank r takes t_k with k mod W == r,
one all-reduce(SUM) of the gradient arena reproduces the sequential accumulation.  CPU, uses the oracle as the
per-pass engine (test infrastructure)."""
import os
import sys

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(2)
    import diff_pruning_b200 as dp
    from oracle import unet_oracle as orc
    cfg = dp.TINY_TEST_CONFIG
    torch.manual_seed(0)
    sd = {k: v.detach().clone().requires_grad_(True) for k, v in dp.UNet2DModel(**cfg).state_dict().items()}
    ac = orc.alphas_cumprod()
    g1, g2 = torch.Generator().manual_seed(1), torch.Generator().manual_seed(2)
    clean, noise = torch.randn(2, 3, 16, 16, generator=g1), torch.randn(2, 3, 16, 16, generator=g2)
    ts = list(range(0, 60, 10))
    for k, t in enumerate(ts):
        if k % world == rank:
            orc.taylor_pass(sd, cfg, ac, clean, noise, (t * torch.ones(2)).long())
    arena = torch.cat([v.grad.flatten() for v in sd.values()])
    dist.all_reduce(arena, op=dist.ReduceOp.SUM)
    if rank == 0:
        ref = {k: v.detach().clone().requires_grad_(True) for k, v in sd.items()}
        for t in ts:
            orc.taylor_pass(ref, cfg, ac, clean, noise, (t * torch.ones(2)).long())
        ref_arena = torch.cat([v.grad.flatten() for v in ref.values()])
        q.put(float((arena - ref_arena).norm() / ref_arena.norm()))
    dist.barrier()
    dist.destroy_process_group()


def test_timestep_sharding_allreduce_equals_sequential():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    err = q.get(timeout=300)
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    assert err < 1e-6


# ---- the `--pruner diff-pruning` stop rule (ddpm_prune.py:104-106) through TaylorScorer.run(thr=...), host logic only: the
# per-pass engine is replaced by a stub that adds a known per-timestep "gradient" and returns a preset loss
LOSS_SEQ = [1.10, 1.25, 1.05, 0.90, 0.70, 0.40, 0.20, 0.061, 0.0624, 0.05, 0.30, 0.01]   # thr 0.05 -> stops at index 7 (0.061 < 0.0625)


def _reference_loop(losses, thr):
    """Literal transcription of ddpm_prune.py:97-106 on fp32 0-dim tensors; returns the timesteps whose backward ran."""
    used, loss_max = [], 0
    for k, v in enumerate(losses):
        loss = torch.tensor(v, dtype=torch.float32)
        used.append(k)                                   # loss.backward()
        if loss > loss_max:
            loss_max = loss
        if loss < loss_max * thr:
            break
    return used


def _stub_scorer():
    from types import SimpleNamespace
    from diff_pruning_b200.scoring import TaylorScorer
    sc = TaylorScorer.__new__(TaylorScorer)
    sc.dev = torch.device("cpu")
    sc.plan = SimpleNamespace(grad_arena=torch.zeros(16), fused_scores=True, score_arena=torch.zeros(4))

    def step(t):
        g = torch.Generator().manual_seed(1000 + t)
        sc.plan.grad_arena += torch.randn(16, generator=g)
        sc.plan.score_arena += float(t + 1)
        return torch.tensor([LOSS_SEQ[t]], dtype=torch.float32)
    sc.step = step
    return sc


def _expected(used):
    arena, score = torch.zeros(16), torch.zeros(4)
    for t in used:
        arena += torch.randn(16, generator=torch.Generator().manual_seed(1000 + t))
        score += float(t + 1)
    return arena, score


def test_threshold_stop_single_process_matches_reference_loop():
    sys.path.insert(0, ROOT)
    from diff_pruning_b200.scoring import threshold_stop
    for thr in (0.05, 0.5, 0.9, 1e-6, 1.0):
        used = _reference_loop(LOSS_SEQ, thr)
        assert threshold_stop(LOSS_SEQ, thr) == len(used)
        sc = _stub_scorer()
        losses = sc.run(range(len(LOSS_SEQ)), thr=thr)
        assert losses.numel() == len(used)
        assert torch.equal(losses, torch.tensor(LOSS_SEQ[:len(used)], dtype=torch.float32))
        arena, score = _expected(used)
        assert torch.equal(sc.plan.grad_arena, arena) and torch.equal(sc.plan.score_arena, score)
    assert _reference_loop(LOSS_SEQ, 0.05) == list(range(8))          # stops on 0.061 < fp32(1.25 * 0.05), keeps that step


def _thr_worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    out = []
    for thr in (0.05, 0.5, 1e-6):
        sc = _stub_scorer()
        losses = sc.run(range(len(LOSS_SEQ)), thr=thr)                  # sharded: rank r takes t = r, r + W, ...
        used = _reference_loop(LOSS_SEQ, thr)
        arena, score = _expected(used)
        out.append((losses.numel() == len(used), float((sc.plan.grad_arena - arena).abs().max()),
                    float((sc.plan.score_arena - score).abs().max())))
    if rank == 0:
        q.put(out)
    dist.barrier()
    dist.destroy_process_group()


def test_threshold_stop_sharded_over_ranks_equals_sequential():
    for world in (2, 3):
        ctx = mp.get_context("spawn")
        q = ctx.Queue()
        port = 31500 + (os.getpid() % 2000) + world
        procs = [ctx.Process(target=_thr_worker, args=(r, world, port, q)) for r in range(world)]
        for p in procs:
            p.start()
        out = q.get(timeout=300)
        for p in procs:
            p.join(60)
            assert p.exitcode == 0
        for ok, e_arena, e_score in out:
            assert ok and e_arena < 1e-5 and e_score == 0.0, (world, out)


# ---- accelerate shim (compat/accelerate): DDP semantics over torch.distributed — sharded batches, averaged gradients, barriers
def _acc_worker(rank, world, port, q):
    sys.path[:0] = [os.path.join(ROOT, "diff-pruning_b200", "compat"), ROOT]
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    torch.set_num_threads(1)
    from accelerate import Accelerator
    acc = Accelerator(gradient_accumulation_steps=1, mixed_precision="no", cpu=True)   # gloo on the host, also where GPUs are visible
    assert acc.num_processes == world and acc.process_index == rank and acc.is_main_process == (rank == 0)
    torch.manual_seed(0)
    model = torch.nn.Linear(4, 3)
    data = torch.arange(8 * 4, dtype=torch.float32).view(8, 4) / 10.0
    loader = torch.utils.data.DataLoader(torch.utils.data.TensorDataset(data), batch_size=2, shuffle=False)
    opt = torch.optim.SGD(model.parameters(), lr=0.1)
    model, opt, loader = acc.prepare(model, opt, loader)
    assert len(loader) == 2                        # 4 batches over 2 processes
    seen = []
    for (xb,) in loader:
        seen.append(xb.clone())
        with acc.accumulate(model):
            opt.zero_grad()
            loss = model(xb).square().sum()
            acc.backward(loss)
            assert acc.sync_gradients
            acc.clip_grad_norm_(model.parameters(), 1e9)
        break
    acc.wait_for_everyone()
    q.put((rank, seen[0].tolist(), model.weight.grad.tolist()))   # plain lists: tensors would travel as shared-memory handles
    acc.wait_for_everyone()
    torch.distributed.destroy_process_group()


def test_accelerate_shim_shards_batches_and_averages_gradients():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_acc_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = sorted([q.get(timeout=120) for _ in range(2)], key=lambda t: t[0])
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    (r0, x0, g0), (r1, x1, g1) = [(r, torch.tensor(x), torch.tensor(g)) for r, x, g in got]
    data = torch.arange(8 * 4, dtype=torch.float32).view(8, 4) / 10.0
    assert torch.equal(x0, data[0:2]) and torch.equal(x1, data[2:4])       # batch k -> process k mod world
    assert torch.equal(g0, g1)                                             # identical after the all-reduce
    torch.manual_seed(0)
    ref = torch.nn.Linear(4, 3)
    gs = []
    for xb in (x0, x1):
        ref.zero_grad()
        ref(xb).square().sum().backward()
        gs.append(ref.weight.grad.clone())
    assert torch.allclose(g0, (gs[0] + gs[1]) / 2, rtol=1e-6, atol=1e-7)   # the MEAN over processes (DDP)
