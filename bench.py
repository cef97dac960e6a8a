#!/usr/bin/env python
"""bench.py — learner transitions/s for the Ape-X hot path (sample + gather +
target + priority update, inside a full learner step) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[1], SURVEY.md §8d C2): Ape-X DQN, 2^20-slot
device-resident sum-tree per GPU, synthetic (4,84,84) uint8 frame stacks (59.2 GB
payload per GPU), batch 512 per GPU.  One "step" = one learner step:
  tree sample (512) -> IS weights -> TMA gather of a, r, done (s and s' are read by the fused
  gather + conv_1 kernels straight from the replay payload) -> Q(s), Q(s'), Qbar(s') ->
  fused double-DQN n-step target / clipped TD / priority / dLoss/dQ -> backward ->
  centered RMSprop -> tree priority write-back
N > 1: one process per GPU, replay sharded (2^20 slots each, weak scaling),
NCCL all-reduce of the gradients (AVG) and of the max IS weight (MAX) — the
only inter-GPU traffic (SURVEY.md §8e).

`value` = transitions/s with everything resident in HBM, the whole step replayed
as one CUDA graph (with parallel branches: the three forward passes, the weight
gradients, the tree update).  `e2e` = the same loop through the public Python API
with HOST buffers: every step ingests 512 new transitions from pinned host memory
(Replay.begin_ingest / commit_ingest -> b2rl_replay_reserve / copy_payload / commit,
the copy overlapping the step) and reads the step's scalars back.

--impl reference times the CPU port of the reference learner loop
(oracle/cpu_learner.py; the reference is pure Python and /root/reference does not
exist on the GPU box) on the host cores, rank 0 only.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

METRIC = "learner transitions/sec (sample+target+prio-update)"
UNIT = "transitions/s"
ALG_BYTES_PER_TRANSITION_GATHER = 2 * 28224 + 4 + 4 + 1   # SURVEY.md §8d: 56 457 B read per transition


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 1000 for apex, 40 for r2d2 / impala)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="apex", choices=["apex", "r2d2", "impala"],
                    help="apex = BASELINE.json configs[1] (the headline the driver runs); r2d2 / impala = configs[2] / "
                         "configs[3] (secondary lines, same JSON contract; --steps defaults apply to apex only)")
    ap.add_argument("--log2pool", type=int, default=14, help="r2d2: log2 of distinct stored sequences (payload pool)")
    ap.add_argument("--log2rollouts", type=int, default=15, help="impala: log2 of rollouts kept per GPU")
    ap.add_argument("--log2n", type=int, default=20, help="log2 of replay slots per GPU")
    ap.add_argument("--batch", type=int, default=512, help="batch per GPU")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--nchw", action="store_true", help="keep the network in NCHW (default: channels_last)")
    ap.add_argument("--unfused-conv1", action="store_true", help="stage the batch and let cuDNN run conv_1")
    ap.add_argument("--cudnn-conv1-wgrad", action="store_true", help="conv_1 weight gradient through a staged fp32 copy + cuDNN instead of csrc/conv1_wgrad.cu")
    ap.add_argument("--inline-wgrad", action="store_true", help="weight gradients inline in backward instead of on a side stream")
    ap.add_argument("--serial-forwards", action="store_true", help="the three forward passes of a step on one stream")
    ap.add_argument("--unfused-tail", action="store_true", help="dueling tail as separate PyTorch ops instead of csrc/dueling.cu")
    ap.add_argument("--cublas-dense", action="store_true", help="dense heads as cuBLAS fp32 GEMMs instead of the 3xTF32 tcgen05 kernel (csrc/gemm.cu)")
    ap.add_argument("--torch-optim", action="store_true", help="torch.optim.RMSprop instead of the fused kernel")
    ap.add_argument("--blaslt", action="store_true", help="route fp32 GEMMs through cuBLASLt")
    ap.add_argument("--tf32-matmul", action="store_true",
                    help="INFORMATIONAL ONLY: let the dense heads use TF32 like cuDNN's convolutions already do "
                         "(PyTorch's default, which the reference runs, is fp32 matmul; the headline keeps fp32)")
    ap.add_argument("--log2n-build", type=int, default=23, help="also time the bulk tree build at this log2 N (0: skip)")
    ap.add_argument("--e2e-steps", type=int, default=200, help="steps per end-to-end segment (3 segments, median reported)")
    ap.add_argument("--quick", action="store_true",
                    help="profiling aid: only the device-resident loop (no per-kernel timing, e2e or CPU baseline); "
                         "the line it prints is NOT a bench result")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=48)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 1000 if args.workload == "apex" else 40
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl b200)")
    return args


def reproducible_cudnn():
    """cuDNN picks the conv_2 / conv_3 algorithms with its heuristics (mode B) among the deterministic ones instead
    of timing candidates (cudnn.benchmark).  Timing can pick differently from run to run; one step that rounds
    differently changes the priorities and with them the minibatches of every later step.  This way the same
    arguments compute the same outputs on every run.  Must run before the process's first convolution."""
    import torch
    os.environ.setdefault("TORCH_CUDNN_USE_HEURISTIC_MODE_B", "1")
    torch.backends.cudnn.benchmark = False
    torch.backends.cudnn.deterministic = True


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(outdir, outputs, rank=0):
    """Write a step's returned tensors as `outdir/<name>.npy` so that two builds can be compared output for output:
    fp32 (and narrower) floats as float32, everything else (int64 indices, fp64) as float64.  Past
    DUMP_LIMIT_BYTES in all, every array is cut to the same fixed, seeded sample of its elements.  Rank r > 0
    of a multi-GPU run writes `<name>_rank<r>.npy`."""
    import numpy as np
    import torch

    arrays = {}
    for name, t in outputs.items():
        t = torch.as_tensor(t).detach()
        small_float = t.is_floating_point() and t.element_size() <= 4
        arrays[name] = t.to("cpu", torch.float32 if small_float else torch.float64).numpy()
    total = sum(a.nbytes for a in arrays.values())
    os.makedirs(outdir, exist_ok=True)
    for name, a in arrays.items():
        if total > DUMP_LIMIT_BYTES:
            keep = max(1, a.size * DUMP_LIMIT_BYTES // total)
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(outdir, name + (f"_rank{rank}" if rank else "") + ".npy"), a)


# --------------------------------------------------------------------------- #
# clocks                                                                        #
# --------------------------------------------------------------------------- #
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 8]
        os.unlink(self.f.name)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except ValueError:
                continue
            for nm, v in zip(names, r[5:9]):
                if "Active" in v and "Not" not in v:
                    reasons.add(nm)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out


# --------------------------------------------------------------------------- #
# reference arm / cpu baseline                                                  #
# --------------------------------------------------------------------------- #
def run_cpu_port(n_slots, batch, steps, warmup, threads=None):
    """`steps` train steps of the CPU port, sampled/assembled `m` at a time like the reference."""
    import torch
    from oracle.cpu_learner import CpuApexLearner

    cores = threads or os.cpu_count() or 1
    torch.set_num_threads(cores)
    m = max(1, min(16, steps))
    L = CpuApexLearner(n_slots, batch, m=m, pool=2048, threads=cores)
    cycles = max(1, (steps + m - 1) // m)
    for _ in range(max(0, (warmup + m - 1) // m)):
        L.cycle()
    tot_t, tot_n, parts = 0.0, 0, {"t_buffer": 0.0, "t_train": 0.0, "t_update": 0.0}
    for _ in range(cycles):
        r = L.cycle()
        tot_t += r["t_total"]; tot_n += r["transitions"]
        for k in parts:
            parts[k] += r[k]
    return {"value": tot_n / tot_t, "seconds": tot_t, "transitions": tot_n, "cores": cores, "m": m,
            "cycles": cycles, "parts": {k: v / cycles for k, v in parts.items()}}


def run_cpu_cycles(make, cycles, warm_cycles=0):
    """Time `cycles` reference cycles (buffer -> m train steps -> write-back) of a CPU port."""
    L = make()
    for _ in range(warm_cycles):
        L.cycle()
    tot_t, tot_n, parts = 0.0, 0, {"t_buffer": 0.0, "t_train": 0.0, "t_update": 0.0}
    for _ in range(cycles):
        r = L.cycle()
        tot_t += r["t_total"]; tot_n += r["transitions"]
        for k in parts:
            parts[k] += r[k]
    return {"value": tot_n / tot_t, "seconds": tot_t, "transitions": tot_n, "cycles": cycles,
            "parts": {k: v / cycles for k, v in parts.items()}}


def best_threads(make_for_threads, probe_cycles=1):
    """The reference leaves torch's intra-op thread count at its default (= all cores), which oversubscribes the
    small convolutions badly on a many-core host: probe a few counts, keep the fastest (reported as `cores`)."""
    import torch
    ncpu = os.cpu_count() or 1
    tried = {}
    for th in sorted({min(8, ncpu), min(32, ncpu), ncpu}):
        torch.set_num_threads(th)
        tried[th] = round(run_cpu_cycles(lambda: make_for_threads(th), probe_cycles)["value"], 1)
    best = max(tried, key=tried.get)
    torch.set_num_threads(best)
    return best, tried


def cpu_c1_legs(threads):
    """SURVEY §8d C1 (BASELINE.json configs[0]): the reference's own CPU-runnable case, N = 2^16, B = 32, m = 16 —
    once with the flat `PER` store the learners use and once with `SumTree` / `PrioritizedMemory`
    (baseline/sumtree.py, baseline/utils.py:328-360) substituted for it."""
    import torch
    from oracle.cpu_learner import CpuApexLearner, CpuApexSumTreeLearner
    torch.set_num_threads(threads)
    out = {}
    for name, cls in (("per_flat", CpuApexLearner), ("sumtree", CpuApexSumTreeLearner)):
        r = run_cpu_cycles(lambda: cls(1 << 16, 32, m=16, pool=1024, threads=threads), 2, 1)
        out[name] = {"value": r["value"], "unit": UNIT, "seconds": r["seconds"], "parts_s_per_cycle": r["parts"]}
    out["config"] = "Ape-X, N=2^16, batch 32, m=16 minibatches per buffer(), 2 cycles after 1 warm-up"
    out["cores"] = threads
    return out


def best_cpu_port(n_slots, batch, steps, warmup):
    """The reference leaves torch's intra-op thread count at its default (= all cores).  On a
    many-core host that oversubscribes the small convolutions badly (measured: 64 tr/s at 128
    threads vs 3200 tr/s at 32), so a 2-step probe picks the fastest of a few thread counts and the
    bounded sample is then timed at that count (reported as `cores`)."""
    ncpu = os.cpu_count() or 1
    tried = {}
    for th in sorted({min(8, ncpu), min(32, ncpu), ncpu}):
        tried[th] = round(run_cpu_port(n_slots, batch, 2, 1, threads=th)["value"], 1)
    best_th = max(tried, key=tried.get)
    best = run_cpu_port(n_slots, batch, steps, warmup, threads=best_th)
    best["tried_threads"] = tried
    return best


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = 1 << args.log2n
    steps = max(1, min(args.steps, 48))  # bounded sample: <= 48 train steps of 512 (about 10 s of CPU work)
    warm = min(args.warmup, 1)
    r = best_cpu_port(n, args.batch, steps, warm)
    sample = (f"{r['cycles']} cycle(s) of {r['m']} train steps x batch {args.batch} at N=2^{args.log2n} "
              f"priorities (payload pool of 2048 pickled records), after {warm} warm-up step(s)")
    line = {
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": r["cycles"] * r["m"], "warmup": warm, "ms_per_step": 1e3 * r["seconds"] / (r["cycles"] * r["m"]),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port", "sample": sample,
                         "parts_s_per_cycle": r["parts"], "tried_threads_tr_per_s": r["tried_threads"],
                         "host_cpus": os.cpu_count()},
        "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(args, world):
    return {"workload": f"Ape-X DQN learner step, 2^{args.log2n}-slot device sum-tree per GPU, synthetic (4,84,84) "
                        f"uint8 frame stacks, batch={args.batch} per GPU (BASELINE.json configs[1])",
            "slots_per_gpu": 1 << args.log2n, "batch_per_gpu": args.batch, "global_batch": args.batch * world,
            "record_bytes": ALG_BYTES_PER_TRANSITION_GATHER,
            "parallelism": f"replay-sharded dp{world}" if world > 1 else "single GPU",
            "l2": "inputs >> L2: every step gathers random rows of a 59 GB payload (no L2 flush needed)",
            "network": "dueling DQN of cfg/ape_x.json; conv_1 forward and weight gradient fused with the gather on tcgen05 "
                       "(int8 digits, fp32-exact), dense heads as 3xTF32 tcgen05 GEMMs at fp32 accuracy, fused dueling tail; "
                       "conv_2/conv_3 in cuDNN at PyTorch's default precision (TF32 convs) = what the reference runs"}


# --------------------------------------------------------------------------- #
# secondary workloads: R2D2 (BASELINE.json configs[2]) and IMPALA (configs[3])      #
# --------------------------------------------------------------------------- #
def secondary_reference_arm(args):
    """--impl reference for --workload r2d2 / impala: the CPU ports of those learners (oracle/cpu_learner.py)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    from oracle import cpu_learner as CL
    threads = min(32, os.cpu_count() or 1)
    torch.set_num_threads(threads)
    if args.workload == "r2d2":
        B = args.batch if args.batch != 512 else 64
        r = run_cpu_cycles(lambda: CL.CpuR2D2Learner(1 << args.log2n, B, m=1, pool=32, threads=threads), 2)
        what = f"R2D2 CPU port: 2 cycles of (buffer + 1 train step) at batch {B} x 80, N=2^{args.log2n} priorities"
    else:
        B = args.batch if args.batch != 512 else 1024
        r = run_cpu_cycles(lambda: CL.CpuImpalaLearner(1 << args.log2rollouts, B, m=1, pool=256, threads=threads), 2)
        what = f"IMPALA CPU port: 2 cycles of (bufferSave + 1 train step) at batch {B} x 20"
    line = {"impl": "reference", "metric": METRIC, "value": r["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": r["cycles"], "warmup": 0, "ms_per_step": 1e3 * r["seconds"] / r["cycles"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload},
            "cpu_baseline": {"value": r["value"], "unit": UNIT, "cores": threads, "kind": "port", "sample": what,
                             "parts_s_per_cycle": r["parts"], "host_cpus": os.cpu_count()},
            "e2e": {"value": r["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def secondary_workload(args):
    """R2D2 (2^20 sequence slots x 80 steps, batch 64) or IMPALA (20-step rollouts, batch 1024) on one GPU:
    sample -> conv_1 over the sampled sequences' frames read IN PLACE in the replay payload -> rest of the
    network -> target / V-trace kernel -> backward -> optimizer -> priority write-back, eager (no CUDA graph:
    the step is milliseconds long).  Same JSON contract as the Ape-X line."""
    import numpy as np
    import torch
    from distributed_rl_b200 import _lib, replay as R
    from distributed_rl_b200.hostmem import pinned_empty, on_gpu_node

    if int(os.environ.get("WORLD_SIZE", "1")) != 1:
        raise SystemExit("--workload r2d2/impala are single-GPU lines (the N-GPU headline is --workload apex)")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    reproducible_cudnn()
    lib = _lib.load()
    steps = args.steps
    warm = max(3, min(args.warmup, 5))
    g = torch.Generator(device=dev); g.manual_seed(0xB200 + 7)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))

    if args.workload == "r2d2":
        from distributed_rl_b200 import r2d2
        N, P, T = 1 << args.log2n, 1 << args.log2pool, 80
        B = args.batch if args.batch != 512 else 64
        cfg = r2d2.R2D2Config(BATCHSIZE=B, REPLAY_MEMORY_LEN=N, BUFFER_SIZE=0, PAYLOAD_POOL=P, FIXED_TRAJECTORY=T,
                              MEM=20, LEARNER_DEVICE=str(dev))
        torch.manual_seed(0)
        L = r2d2.Learner(cfg)
        mem = L.memory
        pool, tree = mem.pool, mem.store
        pool.fill_hash(P, seed=0xB203)
        pool.field_view("action").copy_(torch.randint(0, 6, (P, T), device=dev, generator=g, dtype=torch.int32))
        pool.field_view("reward").copy_(torch.randn(P, T, device=dev, generator=g))
        pool.field_view("h0").copy_(torch.randn(P, 512, device=dev, generator=g) * 0.1)
        pool.field_view("h1").copy_(torch.randn(P, 512, device=dev, generator=g) * 0.1)
        pool.field_view("notdone").copy_((torch.rand(P, device=dev, generator=g) > 0.02).float())
        tree.build((torch.randn(N, device=dev, generator=g).abs().clamp(max=1) + 1e-7) ** cfg.ALPHA)
        tree.seed(1234, 0)
        unit_bytes = T * 28224 + T * 8 + 2 * 512 * 4 + 8                       # SURVEY §8d: 2.263 MB / sequence
        units, frames_per_step, ingest_store = B, B * T, pool
        step_fn = L.fused_step
        scal = lambda o: o["scalars"]
        host = [pinned_empty((B, T, 4, 84, 84), torch.uint8, dev), pinned_empty((B, T), torch.int32, dev),
                pinned_empty((B, T), torch.float32, dev), pinned_empty((B, 512), torch.float32, dev),
                pinned_empty((B, 512), torch.float32, dev), pinned_empty((B,), torch.float32, dev)]
        host[0].random_(0, 256); host[1].random_(0, 6); host[2].normal_(); host[3].normal_(); host[4].normal_()
        host[5].fill_(1.0)
        hp = pinned_empty((B,), torch.float32, dev).fill_(1.0)
        wl = {"workload": f"R2D2 learner step, 2^{args.log2n}-slot device sum-tree, sequences of {T} x (4,84,84) uint8 frames "
                          f"with stored LSTM state, batch={B} sequences (BASELINE.json configs[2])",
              "slots": N, "payload_pool_sequences": P, "batch_sequences": B,
              "pool_note": f"2^{args.log2n} x 2.26 MB = 2.4 TB does not fit HBM: {P} distinct sequences "
                           f"({P * T * 28224 / 1e9:.1f} GB) are stored and slot s reads row s % {P} (SURVEY §8d C3)",
              "record_bytes": unit_bytes, "burn_in": cfg.MEM, "n_step": cfg.UNROLL_STEP,
              "l2": "inputs >> L2: every step reads 64 random 2.26 MB sequences of a 37 GB payload",
              "network": "conv stack -> LSTM(3136,512) -> dueling heads of cfg/r2d2.json; conv_1 (all 80x64 frames, online + "
                         "target) fused with the in-place gather on tcgen05; conv_2/3 + LSTM cuDNN; heads 3xTF32 tcgen05; Adam"}
        conv_rows, c_out, nets = (T - cfg.MEM) * B, 32, 2
    else:
        from distributed_rl_b200 import impala
        cap, T = 1 << args.log2rollouts, 20
        B = args.batch if args.batch != 512 else 1024
        cfg = impala.ImpalaConfig(BATCHSIZE=B, REPLAY_MEMORY_LEN=cap, BUFFER_SIZE=0, UNROLL_STEP=T, LEARNER_DEVICE=str(dev))
        torch.manual_seed(0)
        L = impala.Learner(cfg)
        st = L._memory.store
        st.fill_hash(cap, seed=0xB204)
        st.field_view("action").copy_(torch.randint(0, 6, (cap, T), device=dev, generator=g, dtype=torch.int32))
        st.field_view("mu").copy_(torch.rand(cap, T, device=dev, generator=g) * 0.85 + 0.05)
        st.field_view("reward").copy_(torch.randn(cap, T, device=dev, generator=g))
        st.field_view("done").copy_((torch.rand(cap, device=dev, generator=g) > 0.05).float())
        st.build(torch.ones(cap, device=dev))
        unit_bytes = (T + 1) * 28224 + T * 12 + 4                               # SURVEY §8d: 592.9 KB / rollout
        units, frames_per_step, ingest_store = B, B * (T + 1), st
        step_fn = L.fused_step
        scal = lambda o: torch.stack([o["criticLoss"], o["objActor"]])
        host = [pinned_empty((B, T + 1, 28224), torch.uint8, dev), pinned_empty((B, T), torch.int32, dev),
                pinned_empty((B, T), torch.float32, dev), pinned_empty((B, T), torch.float32, dev),
                pinned_empty((B,), torch.float32, dev)]
        host[0].random_(0, 256); host[1].random_(0, 6); host[2].uniform_(0.05, 0.9); host[3].normal_(); host[4].fill_(1.0)
        hp = pinned_empty((B,), torch.float32, dev).fill_(1.0)
        wl = {"workload": f"IMPALA learner step, uniform replay of 2^{args.log2rollouts} synthetic {T}-step rollouts "
                          f"((T+1) x (4,84,84) uint8 frames), batch={B} rollouts, V-trace (BASELINE.json configs[3])",
              "rollouts_kept": cap, "batch_rollouts": B, "record_bytes": unit_bytes,
              "l2": f"inputs >> L2: every step reads {B} random 593 KB rollouts of a {cap * unit_bytes / 1e9:.1f} GB payload",
              "network": "the reference's runnable policy (cfg/impala.json: conv 8x8s4-16, 4x4s2-32, MLP 2592-256-7): its "
                         "'ResNet-small' (baseNetwork.py:796-820) is broken upstream (SURVEY §8d C4); conv_1 of all "
                         "21 x 1024 frames fused with the in-place gather on tcgen05 (C_OUT=16)"}
        conv_rows, c_out, nets = (T + 1) * B, 16, 1

    def timed_region(k):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(k):
            out = step_fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), out

    for _ in range(warm):
        step_fn()
    torch.cuda.synchronize()
    clocks = ClockSampler(0)
    time.sleep(0.3)
    c0 = lib.b2rl_launch_count()
    ms, out = timed_region(steps)
    launches = lib.b2rl_launch_count() - c0
    clock_info = clocks.stop()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, out)
    value = units * (T if args.workload == "r2d2" else T) * steps / (ms / 1e3)

    # ---- dominant hand-written kernel alone: fused in-place gather + conv_1 over one step's frames ----
    frames = ingest_store.field_view("state").view(-1, 4, 84, 84)
    pack = R.Conv1Pack(nets, dev, c_out)
    wsrc = getattr(L.model, L.model.first_conv_node()).conv_1.weight
    for i in range(nets):
        pack.pack(i, wsrc)
    reps = 5
    rows = [torch.randint(0, frames.shape[0], (conv_rows,), device=dev, generator=g) for _ in range(reps)]
    outc = torch.empty((nets, conv_rows, 20, 20, c_out), device=dev)
    for r_ in rows[:2]:
        R.conv1_fused(frames, r_, pack, relu=True, out=outc)
    torch.cuda.synchronize()
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    for r_ in rows:
        R.conv1_fused(frames, r_, pack, relu=True, out=outc)
    t1.record(); torch.cuda.synchronize()
    c_us = t0.elapsed_time(t1) * 1e3 / reps
    alg = conv_rows * (28224 + nets * 400 * c_out * 4)
    c_ach = alg / (c_us * 1e-6) / 1e9
    data_path = units * unit_bytes / ((ms / steps) * 1e-3) / 1e9
    roofline = {"kernel": f"k_conv1_fused<{nets},{c_out}> — fused in-place gather + im2col + tcgen05 conv_1 over one step's "
                          f"{conv_rows} frame stacks", "bound": "hbm", "achieved": c_ach, "peak": peak, "unit": "GB/s",
                "frac": c_ach / peak, "traffic": None, "launch_us": c_us, "algorithmic_bytes_per_launch": alg,
                "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650",
                "whole_step_data_path": {"bytes_per_unit": unit_bytes, "units_per_step": units,
                                         "achieved_GBs": data_path, "frac": data_path / peak,
                                         "note": "SURVEY §8d per-unit gather bytes x units / step time: the step is bound by the "
                                                 "network (cuDNN conv_2/3, LSTM), not by the replay data path"}}
    del outc, rows

    # ---- e2e: every step ingests `units` new records from pinned host memory + reads the step's scalars back ----
    h2d = sum(t.numel() * t.element_size() for t in host) + hp.numel() * 4
    host_scal = pinned_empty(2, torch.float32, dev)
    ingest_store.push_begin(host, units)

    def e2e_step():
        ingest_store.push_commit(hp)                  # previous copy done -> records sampleable
        ingest_store.push_begin(host, units)          # H2D of the next records on the ingest stream, overlapping the step
        o = step_fn()
        host_scal.copy_(scal(o), non_blocking=True)

    with on_gpu_node(dev) as bound:
        for _ in range(3):
            e2e_step()
        torch.cuda.synchronize()
        k2 = max(10, steps // 2)
        s0 = torch.cuda.Event(enable_timing=True); s1 = torch.cuda.Event(enable_timing=True)
        s0.record()
        for _ in range(k2):
            e2e_step()
        s1.record()
        torch.cuda.synchronize()
    ms2 = s0.elapsed_time(s1)
    e2e = {"value": units * T * k2 / (ms2 / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
           "steps": k2, "ms_per_step": ms2 / k2, "h2d_GBs": h2d * k2 / (ms2 / 1e3) / 1e9,
           "host_thread_bound_to_gpu_numa_node": bool(bound),
           "what": f"push_commit + push_begin of {units} new records from pinned host memory (H2D on the ingest stream) + "
                   "fused_step() + D2H of the step's scalars"}

    cpu = None
    if not args.no_cpu_baseline:
        from oracle import cpu_learner as CL
        threads = min(32, os.cpu_count() or 1)
        torch.set_num_threads(threads)
        if args.workload == "r2d2":
            r = run_cpu_cycles(lambda: CL.CpuR2D2Learner(N, B, m=1, pool=32, threads=threads), 2)
        else:
            r = run_cpu_cycles(lambda: CL.CpuImpalaLearner(cap, B, m=1, pool=256, threads=threads), 2)
        cpu = {"value": r["value"], "unit": UNIT, "cores": threads, "kind": "port", "host_cpus": os.cpu_count(),
               "sample": f"2 cycles of (batch assembly + 1 train step) at batch {B} x {T}, {r['seconds']:.1f} s of CPU work",
               "parts_s_per_cycle": r["parts"]}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": steps, "warmup": warm,
            "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": wl, "units_per_s": units * steps / (ms / 1e3),
            "unit_name": "sequences" if args.workload == "r2d2" else "rollouts",
            "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
            "clocks": clock_info, "cuda_graph": False}
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- #
# our arm                                                                       #
# --------------------------------------------------------------------------- #
def main():
    args = parse()
    if args.workload != "apex":
        (secondary_reference_arm if args.impl == "reference" else secondary_workload)(args)
        return
    if args.impl == "reference":
        reference_arm(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from distributed_rl_b200 import _lib, replay as R
    from distributed_rl_b200.apex import ApexConfig, Learner

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # library knobs for the PyTorch remainder of the network (no precision change: fp32 matmul, TF32 conv)
    reproducible_cudnn()
    if args.cudnn_conv1_wgrad:
        from distributed_rl_b200.apex import _Conv1Gathered
        _Conv1Gathered.fused_wgrad = False
    if args.blaslt:
        torch.backends.cuda.preferred_blas_library("cublaslt")
    if args.tf32_matmul:
        torch.backends.cuda.matmul.allow_tf32 = True
    if world > 1:
        # NCCL_DEBUG is left as the launcher set it (the driver reads the INFO lines to check the rank count);
        # the JSON line is the only line of stdout that starts with '{'.
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.load()

    N, B = 1 << args.log2n, args.batch
    cfg = ApexConfig(BATCHSIZE=B, REPLAY_MEMORY_LEN=N, BUFFER_SIZE=0, LEARNER_DEVICE=str(dev),
                     CHANNELS_LAST=not args.nchw, FUSED_CONV1=not args.unfused_conv1,
                     FUSED_OPTIM=not args.torch_optim, DENSE_3XTF32=not args.cublas_dense, FUSED_DUELING_TAIL=not args.unfused_tail, PARALLEL_FORWARDS=not args.serial_forwards, DEFERRED_WGRAD=not args.inline_wgrad,
                     CUDNN_BENCHMARK=False)
    torch.manual_seed(0)
    learner = Learner(cfg, connect=None, start_replay=False)
    if world > 1:   # identical initial weights on every rank
        for p in list(learner.model.parameters()) + list(learner.target_model.parameters()):
            dist.broadcast(p.data, 0)
        learner.enable_data_parallel()
    store = learner.memory.store
    # ---- pre-fill: synthetic frames by counter hash, typed scalars, priorities (SURVEY §8d) ----
    store.fill_hash(N, seed=0xB200 + rank)
    g = torch.Generator(device=dev); g.manual_seed(0xB200 + 1 + rank)
    store.field_view("action").copy_(torch.randint(0, cfg.ACTION_SIZE, (N,), device=dev, generator=g, dtype=torch.int32))
    store.field_view("reward").copy_(torch.randn(N, device=dev, generator=g).clamp_(-1, 1))
    store.field_view("done").copy_((torch.rand(N, device=dev, generator=g) < 0.02).to(torch.uint8))
    prios = (torch.randn(N, device=dev, generator=g).abs().clamp(max=1) + 1e-7) ** cfg.ALPHA
    store.build(prios)
    store.seed(1234 + rank, 0)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm: the whole step as one CUDA graph --------------------------
    use_graph = not args.no_graph
    for _ in range(max(3, args.warmup)):     # first call builds (3 eager warm-ups + capture)
        learner.fused_step(use_graph=use_graph)
    per_step_launches = learner.launches_per_step
    barrier()
    clocks = ClockSampler(local) if rank == 0 else None
    time.sleep(0.3)
    barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        out = learner.fused_step(use_graph=use_graph)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    clock_info = clocks.stop() if clocks else None
    value = B * world * args.steps / (ms / 1e3)
    scal = out["scalars"].tolist()
    if args.dump_outputs:     # before anything else replays the step graph, whose outputs `out` holds
        dump_outputs(args.dump_outputs, out, rank)

    if args.quick:
        if rank == 0:
            print(json.dumps({"quick": True, "not_a_bench_result": True, "ms_per_step": ms / args.steps,
                              "gpu_launches_per_step": per_step_launches}), flush=True)
        return
    # ---- dominant hand-written kernels, each timed alone with CUDA events (graph of `reps`
    #      launches on distinct index sets -> no Python launch overhead, no L2 reuse of the rows) ----
    reps = 20
    idxs = [store.sample(B, beta=cfg.BETA, want_prob=False)[0] for _ in range(reps)]

    def time_graph(fn):
        for i in range(3):
            fn(idxs[i])
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for i in range(reps):
                fn(idxs[i])
        gr.replay(); torch.cuda.synchronize()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record(); gr.replay(); t1.record(); torch.cuda.synchronize()
        del gr
        return t0.elapsed_time(t1) * 1e3 / reps

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write)" if peaks else "fallback 6650"
    outb = store.alloc_batch(B)
    gather_us = time_graph(lambda ix: store.gather(ix, outb))
    g_ach = ALG_BYTES_PER_TRANSITION_GATHER * B / (gather_us * 1e-6) / 1e9
    kernels = {"k_gather_bulk": {"launch_us": gather_us, "algorithmic_bytes_per_launch": ALG_BYTES_PER_TRANSITION_GATHER * B,
                                 "achieved_GBs": g_ach, "frac": g_ach / peak,
                                 "note": "whole minibatch (s, s', a, r, done) staged in one launch; a copy moves 2x its "
                                         "algorithmic read bytes, so frac <= 0.5 for an unfused gather"}}
    roofline = {"kernel": "k_gather_bulk — TMA bulk gather of one minibatch", "bound": "hbm", "achieved": g_ach,
                "peak": peak, "unit": "GB/s", "frac": g_ach / peak, "peak_source": peak_src, "traffic": None,
                "launch_us": gather_us, "algorithmic_bytes_per_launch": ALG_BYTES_PER_TRANSITION_GATHER * B}
    if cfg.FUSED_CONV1 and learner._conv1_ready():
        # fused gather + conv_1 for online+target nets over s': reads B frame stacks, writes 2 x B x (20,20,32) fp32
        alg = B * (28224 + 2 * 400 * 32 * 4)
        out2 = torch.empty((2, B, 20, 20, 32), device=dev)
        nsf = store.field_view("next_state")
        c_us = time_graph(lambda ix: R.conv1_fused(nsf, ix, learner._pack2, relu=True, out=out2))
        c_ach = alg / (c_us * 1e-6) / 1e9
        ops = 2.0 * (B * 400) * 256 * 256        # useful MACs x2 incl. the 4 weight digits (N=256 columns)
        kernels["k_conv1_fused<2>"] = {"launch_us": c_us, "algorithmic_bytes_per_launch": alg, "achieved_GBs": c_ach,
                                       "frac": c_ach / peak, "int8_TOPS": ops / (c_us * 1e-6) / 1e12,
                                       "note": "reads 28 224 B per sampled s' directly from the replay payload "
                                               "(no staging copy) and writes conv_1 activations of both networks"}
        roofline = {"kernel": "k_conv1_fused<2> — fused TMA gather + im2col + tcgen05 conv_1 (online+target) of s'",
                    "bound": "hbm", "achieved": c_ach, "peak": peak, "unit": "GB/s", "frac": c_ach / peak,
                    "peak_source": peak_src, "traffic": None, "launch_us": c_us, "algorithmic_bytes_per_launch": alg,
                    "note": "algorithmic bytes = sampled frames read (SURVEY §8d: 28 224 B per frame stack) + the two "
                            "fp32 NHWC activation maps written; currently epilogue/issue-bound, not HBM-bound "
                            "(tensor pipe 21.6 % active, profiles/r01_conv1.md)"}
    if cfg.FUSED_CONV1 and learner._conv1_ready():
        # fused gather + conv_1 weight gradient: reads B frame stacks + dL/dy (B x 400 x 32 fp32), writes 8192 floats
        alg_w = B * (28224 + 400 * 32 * 4)
        gyw = torch.randn(B, 32, 20, 20, device=dev).contiguous(memory_format=torch.channels_last)
        sf = store.field_view("state")
        w_us = time_graph(lambda ix: R.conv1_wgrad(sf, ix, gyw))
        w_ach = alg_w / (w_us * 1e-6) / 1e9
        kernels["k_conv1_wgrad"] = {"launch_us": w_us, "algorithmic_bytes_per_launch": alg_w, "achieved_GBs": w_ach,
                                    "frac": w_ach / peak, "int8_TOPS": 2.0 * (B * 400) * 256 * 128 / (w_us * 1e-6) / 1e12,
                                    "note": "launch_us covers k_conv1_wgrad + k_conv1_wgrad_reduce; reads each sampled s "
                                            "and its dL/dy once (dL/dy twice: scale pre-scan), no fp32 staging of the frames"}
    if cfg.DENSE_3XTF32:
        # the dominant kernel by device time: the 3xTF32 GEMM of the fused 3136 -> 2x512 heads (forward shape)
        from distributed_rl_b200 import linear as LIN
        # the forward call of the step: the online network's two passes run as ONE M = 2B GEMM (BATCHED_ONLINE)
        batched = bool(cfg.BATCHED_ONLINE and cfg.PARALLEL_FORWARDS and cfg.FUSED_CONV1)
        tpeak = float(peaks.get("bf16_tflops", 1719.3))

        def time_gemm(Mg, Ng, Kg):
            xa = LIN.split_pack(torch.randn(Mg, Kg, device=dev), False, False)
            wb = LIN.split_pack(torch.randn(Ng, Kg, device=dev) * 0.02, False, True)
            og = torch.empty(Mg, Ng, device=dev)
            us = time_graph(lambda ix: LIN.gemm_packed(xa, wb, Mg, Ng, Kg, out=og))
            fl = 2.0 * Mg * Ng * Kg
            return us, fl, fl / (us * 1e-6) / 1e12

        Mg, Ng, Kg = (2 * B if batched else B), 1024, 3136
        g_us, alg_fl, t_ach = time_gemm(Mg, Ng, Kg)
        kernels["k_gemm_tf32x3"] = {"launch_us": g_us, "algorithmic_flops_per_launch": alg_fl, "achieved_TFLOPs": t_ach,
                                    "frac": t_ach / tpeak, "tf32_TFLOPs_executed": 3 * t_ach,
                                    "frac_of_tf32_peak_est": 3 * t_ach / (tpeak / 2), "shape_MNK": [Mg, Ng, Kg],
                                    "note": f"launch_us covers k_gemm_tf32x3 + k_splitk_reduce for x[{Mg}x{Kg}] @ W[{Ng}x{Kg}]^T "
                                            "(the step's forward call: Q(s) and Q_online(s') batched); algorithmic flops = the "
                                            "fp32 GEMM (2MNK); the kernel executes 3 TF32 products per term pair, and TF32 dense "
                                            "peak is half the measured bf16 peak"}
        if batched:
            u1, f1, a1 = time_gemm(B, Ng, Kg)
            kernels["k_gemm_tf32x3(M=B, target-net call)"] = {"launch_us": u1, "algorithmic_flops_per_launch": f1,
                                                              "achieved_TFLOPs": a1, "frac": a1 / tpeak, "shape_MNK": [B, Ng, Kg]}
        roofline = {"kernel": "k_gemm_tf32x3 — fp32-accurate dense heads as 3xTF32 tcgen05 GEMM (largest share of the step)",
                    "bound": "tensor", "achieved": t_ach, "peak": tpeak, "unit": "TFLOP/s", "frac": t_ach / tpeak,
                    "peak_source": "measured (MEASURED_PEAKS.json bf16_tflops, burst)" if peaks else "fallback 1719.3",
                    "traffic": None, "launch_us": g_us, "algorithmic_flops_per_launch": alg_fl, "shape_MNK": [Mg, Ng, Kg],
                    "note": "achieved counts the fp32 GEMM's 2MNK flops once; the tensor pipe executes 3x that in TF32 "
                            "(tf32_TFLOPs_executed), whose dense peak is bf16/2 — see kernels[k_gemm_tf32x3]"}
    # ---- the sum-tree kernels (the kernels north_star sets the HBM target on), SURVEY.md §8d bytes:
    #      sample 4*(log2N+2) = 88 B/draw @2^20, update 4 + 8*log2N = 164 B/update @2^20, bulk build 8N B ----
    lg = args.log2n
    b_sample, b_update = 4 * (lg + 2), 4 + 8 * lg

    def time_plain(fn, reps=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            for _ in range(reps):
                fn()
        gr.replay(); torch.cuda.synchronize()
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        t0.record(); gr.replay(); t1.record(); torch.cuda.synchronize()
        del gr
        return t0.elapsed_time(t1) * 1e3 / reps

    prio_backup = store.priorities().clone()
    rng_t = torch.Generator(device=dev); rng_t.manual_seed(77 + rank)
    sweep = {}
    for ns in (B, 8192, 65536, 1 << 20):
        oi = torch.empty(ns, dtype=torch.int64, device=dev); ow = torch.empty(ns, device=dev)
        us = time_plain(lambda: store.sample(ns, beta=cfg.BETA, want_prob=False, out=(oi, None, ow)), reps=10)
        sweep[str(ns)] = {"launch_us": us, "achieved_GBs": b_sample * ns / (us * 1e-6) / 1e9,
                          "frac": b_sample * ns / (us * 1e-6) / 1e9 / peak}
    s_us = sweep[str(B)]["launch_us"]
    kernels["k_tree_sample"] = {"launch_us": s_us, "algorithmic_bytes_per_launch": b_sample * B,
                                "achieved_GBs": sweep[str(B)]["achieved_GBs"], "frac": sweep[str(B)]["frac"],
                                "samples_per_launch_sweep": sweep,
                                "note": f"{b_sample} B per draw (SURVEY §8d); latency-bound at B={B}: ceil(log2N/4) dependent "
                                        "128-byte loads per draw (sparse radix-16 tree) + the IS-weight pow; the sweep shows "
                                        "the large-batch asymptote"}
    upd = {}
    for nu in (B, 65536):
        ui = torch.randint(0, N, (nu,), device=dev, generator=rng_t)
        uv = torch.rand(nu, device=dev, generator=rng_t) + 0.01
        us = time_plain(lambda: store.update(ui, uv), reps=10)
        upd[str(nu)] = {"launch_us": us, "achieved_GBs": b_update * nu / (us * 1e-6) / 1e9,
                        "frac": b_update * nu / (us * 1e-6) / 1e9 / peak}
    kernels["k_update_small"] = {"launch_us": upd[str(B)]["launch_us"], "algorithmic_bytes_per_launch": b_update * B,
                                 "achieved_GBs": upd[str(B)]["achieved_GBs"], "frac": upd[str(B)]["frac"],
                                 "note": f"{b_update} B per update (SURVEY §8d); one CTA, last-writer-wins, "
                                         "ceil(log2N/4) level barriers; latency-bound"}
    kernels["k_update_large(65536)"] = {"launch_us": upd["65536"]["launch_us"],
                                        "algorithmic_bytes_per_launch": b_update * 65536,
                                        "achieved_GBs": upd["65536"]["achieved_GBs"], "frac": upd["65536"]["frac"],
                                        "note": "tag + write + one launch per stored level (2 + ceil(log2N/4) launches)"}
    pb = prio_backup if prio_backup.numel() == N else prios
    bu = time_plain(lambda: store.build(pb), reps=10)
    kernels["k_build_leaves+top"] = {"launch_us": bu, "algorithmic_bytes_per_launch": 8 * N,
                                     "achieved_GBs": 8 * N / (bu * 1e-6) / 1e9, "frac": 8 * N / (bu * 1e-6) / 1e9 / peak,
                                     "note": "8N B algorithmic (4N leaf read + 4N internal write, SURVEY §8d); moves "
                                             "~8.8N (4N read, 4N fp32 leaf copy, 0.75N fp64 sums + fp32 mins)"}
    store.build(prio_backup); store.seed(1234 + rank, 10 ** 9)
    if args.log2n_build and rank == 0:
        # bulk build at a larger N (default 2^23, SURVEY §8d C5's total) on a scratch tree-only replay
        nb = 1 << args.log2n_build
        scratch = R.DeviceReplay(nb, fields=(), device=dev)
        pbig = torch.rand(nb, device=dev) + 0.01
        bu2 = time_plain(lambda: scratch.build(pbig), reps=10)
        kernels[f"k_build_leaves+top(2^{args.log2n_build})"] = {
            "launch_us": bu2, "algorithmic_bytes_per_launch": 8 * nb, "achieved_GBs": 8 * nb / (bu2 * 1e-6) / 1e9,
            "frac": 8 * nb / (bu2 * 1e-6) / 1e9 / peak}
        scratch.close(); del pbig
    roofline["kernels"] = kernels
    roofline["tree_sample_update"] = {
        "what": "k_tree_sample + k_update_small at the step's batch (the north-star sum-tree sample+update pair)",
        "algorithmic_bytes": (b_sample + b_update) * B, "us": s_us + upd[str(B)]["launch_us"],
        "achieved_GBs": (b_sample + b_update) * B / ((s_us + upd[str(B)]["launch_us"]) * 1e-6) / 1e9,
        "frac": (b_sample + b_update) * B / ((s_us + upd[str(B)]["launch_us"]) * 1e-6) / 1e9 / peak,
        "bound": "latency (dependent loads), not bandwidth: 129 KB per launch cannot occupy HBM"}
    prof = os.path.join(REPO, "profiles", "r02_traffic.json")
    if os.path.isfile(prof):
        try:
            tr = json.load(open(prof))
            key = next((k for k in ("k_gemm_tf32x3", "k_conv1_fused<2>", "k_gather_bulk") if k in kernels and k in tr),
                       None)
            roofline["traffic"] = tr.get(key) if key else None
            roofline["traffic_source"] = "profiles/r02_traffic.json (dram__bytes_read.sum + dram__bytes_write.sum of one " \
                                         "ncu --set full capture of this kernel, per launch; not re-measured in this run)"
        except Exception:
            pass

    # ---- e2e: public API, host buffers in, scalars out -----------------------------------
    from distributed_rl_b200.hostmem import pinned_like, pinned_empty   # pinned pages on the GPU's NUMA node
    pin = lambda t: pinned_like(t, dev)
    rng = np.random.default_rng(7 + rank)
    hs = pin(torch.from_numpy(rng.integers(0, 256, size=(B, 4, 84, 84), dtype=np.uint8)))
    hns = pin(torch.from_numpy(rng.integers(0, 256, size=(B, 4, 84, 84), dtype=np.uint8)))
    ha = pin(torch.from_numpy(rng.integers(0, 6, size=B).astype(np.int32)))
    hr = pin(torch.from_numpy(np.clip(rng.standard_normal(B), -1, 1).astype(np.float32)))
    hd = pin(torch.from_numpy((rng.random(B) < 0.02).astype(np.uint8)))
    hp = pin(torch.ones(B, dtype=torch.float32))
    h2d = sum(t.numel() * t.element_size() for t in (hs, hns, ha, hr, hd, hp))
    host_scal = [pinned_empty(3, torch.float32, dev) for _ in range(2)]
    d2h_stream = torch.cuda.Stream(dev)
    d2h_done = [torch.cuda.Event(), torch.cuda.Event()]
    step_done = torch.cuda.Event()
    seen = {"n": 0, "loss": 0.0}

    # Pipelined ingest: the copy of the NEXT 512 transitions runs on the ingest stream while the
    # current learner step computes; every step still moves its own 29 MB H2D inside the timed region.
    # Every step's scalars (loss, mean target, mean weight) are read back to pinned host memory on a
    # D2H stream and consumed by the host one step later, so the host never idles the GPU.
    learner.memory.ingest(hs, hns, ha, hr, hd, hp)

    def e2e_step(i=[0]):
        k = i[0] & 1
        if i[0] > 0:   # the previous step's 12-byte read must leave `scalars` before the graph rewrites it
            torch.cuda.current_stream(dev).wait_event(d2h_done[k ^ 1])
        # ONE C call: the batch copied during the previous step becomes sampleable, the slots of the next 512
        # transitions are retired and their H2D copy starts on the library's copy stream (async)
        learner.memory.ingest(hs, hns, ha, hr, hd, hp)
        o = learner.fused_step(use_graph=use_graph)
        step_done.record(torch.cuda.current_stream(dev))
        if i[0] > 0:                                                # consume the PREVIOUS step's result
            d2h_done[k ^ 1].synchronize()
            seen["n"] += 1; seen["loss"] = float(host_scal[k ^ 1][0])
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(step_done)
            host_scal[k].copy_(o["scalars"], non_blocking=True)     # D2H of this step's loss / mean target / mean w
            d2h_done[k].record(d2h_stream)
        i[0] += 1

    # Warm-up: the PCIe link reaches its full rate only after ~0.2 s of sustained traffic (tools/h2d_probe.py:
    # 25 -> 47 -> 55 GB/s over the first three 150-copy bursts), and it idles during the device-resident
    # region above, so the steady-state loop is entered with enough untimed steps to move ~5 GB first.
    # The host thread that drives the loop is bound to the GPU's NUMA node (numactl --cpunodebind in a
    # deployment): every step makes ~10 driver calls whose doorbell writes cross the socket interconnect otherwise.
    from distributed_rl_b200.hostmem import on_gpu_node
    with on_gpu_node(dev) as bound:
        for _ in range(max(3, args.warmup) + 170):
            e2e_step()
        barrier()
        k2 = max(200, args.e2e_steps)             # independent of --steps: >= 200 steps per segment
        segs = []
        for _ in range(3):
            s0 = torch.cuda.Event(enable_timing=True); s1 = torch.cuda.Event(enable_timing=True)
            s0.record()
            th0 = time.perf_counter()
            for _ in range(k2):
                e2e_step()
            host_ms = (time.perf_counter() - th0) * 1e3
            s1.record()
            d2h_done[0].synchronize(); d2h_done[1].synchronize()   # the last step's result has been read too
            barrier()
            ms2 = s0.elapsed_time(s1)
            if world > 1:
                t = torch.tensor([ms2], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms2 = float(t.item())
            segs.append((ms2, host_ms))
    segs.sort()
    ms2, host_ms = segs[1]                        # median segment
    e2e = {"value": B * world * k2 / (ms2 / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": 12, "steps": k2, "segments": 3,
           "segment_values": [B * world * k2 / (m / 1e3) for m, _ in segs],
           "h2d_GBs": h2d * k2 / (ms2 / 1e3) / 1e9, "host_ms_per_step": host_ms / k2, "ms_per_step": ms2 / k2,
           "host_thread_bound_to_gpu_numa_node": bool(bound),
           "what": "Replay.ingest (b2rl_replay_ingest_pipelined: 512 new transitions from pinned host, H2D on the library's "
                   "copy stream overlapping the step, published by the next call) + Learner.fused_step() + per-step D2H "
                   "of the step's scalars to pinned host memory (consumed by the host one step later); median of 3 segments"}

    # ---- CPU baseline (rank 0, N=1 only) --------------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        r = best_cpu_port(N, B, args.cpu_steps, 1)
        cpu = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": "port",
               "tried_threads_tr_per_s": r["tried_threads"], "host_cpus": os.cpu_count(),
               "sample": f"{r['cycles']} cycle(s) x {r['m']} train steps x batch {B} at N=2^{args.log2n} priorities "
                         f"(pool of 2048 pickled records), {r['seconds']:.1f} s of CPU work",
               "parts_s_per_cycle": r["parts"]}
        try:        # SURVEY §8d C1: the reference's own CPU-runnable case, flat PER store and SumTree store
            cpu["c1_reference_case"] = cpu_c1_legs(r["cores"])
        except Exception as e:  # noqa: BLE001 — a baseline leg must never take the bench line down
            cpu["c1_reference_case"] = {"error": repr(e)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms / args.steps, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": workload_config(args, world), "roofline": roofline, "cpu_baseline": cpu,
                "e2e": e2e, "gpu_launches": int(per_step_launches * args.steps), "clocks": clock_info,
                "cuda_graph": use_graph, "fused_gather_conv1": bool(cfg.FUSED_CONV1), "fused_optimizer": bool(cfg.FUSED_OPTIM), "tf32_matmul": bool(args.tf32_matmul), "dense_3xtf32": bool(cfg.DENSE_3XTF32), "fused_conv1_wgrad": not args.cudnn_conv1_wgrad, "fused_dueling_tail": bool(cfg.FUSED_DUELING_TAIL), "parallel_forwards": bool(cfg.PARALLEL_FORWARDS), "deferred_wgrad": bool(cfg.DEFERRED_WGRAD), "peer_allreduce": bool(getattr(learner, "peer_allreduce", False)), "peer_allreduce_heads": bool(getattr(learner, "peer_allreduce_heads", False)), "last_step": {"loss": scal[0], "mean_target": scal[1], "mean_weight": scal[2]}}
        print(json.dumps(line), flush=True)
    sys.stdout.flush()
    if world > 1:
        # Orderly teardown: a CUDA graph that holds NCCL kernels must be destroyed BEFORE its communicator,
        # and every rank must have drained its device before the process group goes away.
        learner._graph = None
        learner._static = None
        import gc
        gc.collect()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
