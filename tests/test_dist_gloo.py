"""world_size-2 gloo tests (CPU) of the host-side multi-GPU logic: flat gradient
bucket averaging, the priority-max reduction that makes sharded IS weights equal
the single-replay formula, slot sharding, and bench.py's reference arm under
torchrun (rank != 0 exits quietly)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, REPO)
    from distributed_rl_b200 import dist as D
    from oracle import oracle as O
    out = {}
    # 1. flat bucket: mean of per-rank gradients, grads stay views of the bucket
    torch.manual_seed(0)
    lin = torch.nn.Sequential(torch.nn.Linear(4, 3, bias=False), torch.nn.Linear(3, 2, bias=False))
    bucket = D.FlatGradBucket(lin.parameters())
    x = torch.full((5, 4), float(rank + 1))
    lin(x).sum().backward()
    local = bucket.flat.clone()
    bucket.all_reduce_mean()
    both = [torch.zeros_like(local) for _ in range(world)]
    dist.all_gather(both, local)
    out["bucket_ok"] = bool(torch.allclose(bucket.flat, sum(both) / world))
    out["views_ok"] = all(p.grad.data_ptr() >= bucket.flat.data_ptr() for p in lin.parameters())
    # 1b. overlapped variant: early params reduced from the autograd hook, late ones in finish()
    lin2 = torch.nn.Sequential(torch.nn.Linear(4, 3, bias=False), torch.nn.Linear(3, 2, bias=False))
    b2 = D.FlatGradBucket(lin2.parameters())
    b2.enable_overlap([lin2[1].weight])          # the last layer's gradient is ready first
    lin2(x).sum().backward()
    b2.finish()
    # the early all-reduce runs asynchronously in place, so this rank's own gradients come from a replica
    ref2 = torch.nn.Sequential(torch.nn.Linear(4, 3, bias=False), torch.nn.Linear(3, 2, bias=False))
    ref2.load_state_dict(lin2.state_dict())
    ref2(x).sum().backward()
    ok = True
    for p, r in zip(lin2.parameters(), ref2.parameters()):
        g = [torch.zeros_like(r.grad) for _ in range(world)]
        dist.all_gather(g, r.grad)
        ok = ok and bool(torch.allclose(p.grad, sum(g) / world))
    out["overlap_ok"] = ok
    # 1c. early gradients that bypass AccumulateGrad (linear.WeightGradSink): the sink's on_ready callback
    #     stands in for the autograd hook and launches the early all-reduce
    lin3 = torch.nn.Sequential(torch.nn.Linear(4, 3, bias=False), torch.nn.Linear(3, 2, bias=False))
    b3 = D.FlatGradBucket(lin3.parameters())
    b3.enable_overlap([lin3[1].weight])

    class _Sink:                       # the part of WeightGradSink the bucket uses
        on_ready = {}
    b3.attach_sink(_Sink)
    w_early = lin3[1].weight
    h3 = lin3[0](x)
    gw_early = torch.ones(5, 2).T @ h3.detach()            # d(sum)/dW of the last layer, computed "elsewhere"
    torch.autograd.backward(h3 @ w_early.detach().T, torch.ones(5, 2))   # autograd only sees the late layer
    w_early.grad.add_(gw_early)
    _Sink.on_ready[id(w_early)](w_early)                   # what sink.accumulate() does after the add
    local3 = [p.grad.clone() for p in lin3.parameters()]   # the early part may already be reduced in place: compare sums
    b3.finish()
    ref3 = torch.nn.Sequential(torch.nn.Linear(4, 3, bias=False), torch.nn.Linear(3, 2, bias=False))
    ref3.load_state_dict(lin3.state_dict())
    ref3(x).sum().backward()
    ok3 = True
    for p, r in zip(lin3.parameters(), ref3.parameters()):
        g = [torch.zeros_like(r.grad) for _ in range(world)]
        dist.all_gather(g, r.grad)
        ok3 = ok3 and bool(torch.allclose(p.grad, sum(g) / world, atol=1e-6))
    out["sink_ok"] = ok3
    # 1d. regression (round 1, found by tests/test_gpu_20_multigpu.py): torch runs post-accumulate-grad hooks even
    #     when a custom Function returns None for a parameter.  With a sink attached those calls must not count:
    #     the early all-reduce may only start after the sink has reported EVERY early gradient.
    class _NoWeightGrad(torch.autograd.Function):
        @staticmethod
        def forward(ctx, x, w):
            ctx.save_for_backward(x, w)
            return x @ w.T

        @staticmethod
        def backward(ctx, gy):
            x, w = ctx.saved_tensors
            return gy @ w, None                         # dL/dW is produced "elsewhere" (the sink)

    wa = torch.nn.Parameter(torch.randn(3, 4)); wb = torch.nn.Parameter(torch.randn(2, 3))
    b4 = D.FlatGradBucket([wa, wb])
    b4.enable_overlap([wa, wb])

    class _Sink4:
        on_ready = {}
    b4.attach_sink(_Sink4)
    x4 = torch.randn(5, 4, requires_grad=True)
    _NoWeightGrad.apply(_NoWeightGrad.apply(x4, wa), wb).sum().backward()    # fires both autograd hooks, no grads
    started_early = b4._work is not None
    ga, gb = torch.full_like(wa, float(rank + 1)), torch.full_like(wb, float(2 * rank + 1))
    wb.grad.add_(gb); _Sink4.on_ready[id(wb)](wb)
    after_one = b4._work is not None
    wa.grad.add_(ga); _Sink4.on_ready[id(wa)](wa)
    b4.finish()
    mean_a = sum(float(r + 1) for r in range(world)) / world
    mean_b = sum(float(2 * r + 1) for r in range(world)) / world
    out["none_grad_hooks_ok"] = (not started_early) and (not after_one) and \
        bool(torch.allclose(wa.grad, torch.full_like(wa, mean_a))) and bool(torch.allclose(wb.grad, torch.full_like(wb, mean_b)))
    # 1e. two overlapped groups (heads | conv_2, conv_3) + a late rest (conv_1), reported through the sink in the
    #     order the learner's two lanes do; wait_group(0) (the early optimizer step's gate) finishes group 0 alone
    ws = [torch.nn.Parameter(torch.randn(3, 3)) for _ in range(5)]
    b5 = D.FlatGradBucket(ws)
    b5.enable_overlap([ws[3], ws[4]], [ws[1], ws[2]])

    class _Sink5:
        on_ready = {}
    b5.attach_sink(_Sink5)
    gs5 = [torch.full((3, 3), float((i + 1) * (rank + 1))) for i in range(5)]
    gate_before = b5.wait_group(0)
    for i in (4, 3):                                     # heads' lane
        ws[i].grad.add_(gs5[i]); _Sink5.on_ready[id(ws[i])](ws[i])
    gate_after = b5.wait_group(0)
    heads_final = all(bool(torch.allclose(ws[i].grad, torch.full((3, 3), (i + 1) * (world + 1) / 2.0))) for i in (3, 4))
    for i in (2, 1):                                     # conv lane
        ws[i].grad.add_(gs5[i]); _Sink5.on_ready[id(ws[i])](ws[i])
    ws[0].grad.add_(gs5[0])                              # conv_1: plain late gradient
    b5.finish()
    out["two_groups_ok"] = (not gate_before) and gate_after and heads_final and all(
        bool(torch.allclose(ws[i].grad, torch.full((3, 3), (i + 1) * (world + 1) / 2.0))) for i in range(5))
    # 2. priority-max reduction: shard-local IS weights / global max == single-replay formula
    n, beta = 1024, 0.4
    rng = np.random.default_rng(100 + rank)
    p = ((np.abs(rng.standard_normal(n)).clip(max=1) + 1e-7) ** 0.6).astype(np.float32)
    t = O.SumTreeOracle(n); t.build(p)
    idx, _ = t.sample(rng.random(64))
    w_local, prob, max_w_local = O.is_weights(p[idx], t.total, t.min_priority, n, beta)
    mw = torch.tensor([float(max_w_local)])
    D.all_reduce_max_(mw)
    w_global = (w_local * (max_w_local / np.float32(mw.item()))).astype(np.float32)
    # single-process statement of SURVEY §8e: P(i) = (1/G) p_i / S_g, N = G n, w = (N P)^-beta / max
    shards = [torch.zeros(n) for _ in range(world)]
    dist.all_gather(shards, torch.from_numpy(p))
    NP = []
    for sp in shards:
        spn = sp.numpy().astype(np.float64)
        NP.append((world * n) * (1.0 / world) * spn / spn.sum())
    max_all = max(float((x ** -beta).max()) for x in NP)
    expect = (NP[rank][idx] ** -beta) / max_all
    out["isw_ok"] = bool(np.allclose(w_global, expect, rtol=2e-6))
    out["mw"] = float(mw.item())
    # 3. slot sharding covers [0, N) without overlap
    rs = [D.shard_slots(1000, r, world) for r in range(world)]
    out["shard_ok"] = sorted(i for r in rs for i in r) == list(range(1000))
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def test_world2_gloo_data_parallel_logic():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 300
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for r in (0, 1):
        assert res[r]["bucket_ok"] and res[r]["views_ok"] and res[r]["isw_ok"] and res[r]["shard_ok"], res[r]
        assert res[r]["overlap_ok"], res[r]
        assert res[r]["sink_ok"], res[r]
        assert res[r]["none_grad_hooks_ok"], res[r]
        assert res[r]["two_groups_ok"], res[r]
    assert res[0]["mw"] == res[1]["mw"]


def test_bench_reference_arm_under_torchrun_only_rank0_prints(tmp_path):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", str(29950 + os.getpid() % 40),
           os.path.join(REPO, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0",
           "--log2n", "12", "--batch", "8"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=tmp_path)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    j = json.loads(lines[0])
    assert j["impl"] == "reference" and j["n_gpus"] == 2 and j["cpu_baseline"]["kind"] == "port"
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["value"] > 0
