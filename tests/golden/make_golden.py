"""Generate the golden vectors in this directory by EXECUTING the unmodified
reference (/root/reference, build container only; see oracle/ref_harness.py).

    python tests/golden/make_golden.py            # all groups, one subprocess each
    python tests/golden/make_golden.py apex       # one group

The reference ships no tests or golden vectors (SURVEY.md §4), so these files
are what pins the oracle: inputs are synthetic and seeded here, outputs are
whatever the reference's own functions returned.

Groups
  tree    baseline/sumtree.py SumTree + baseline/utils.py PrioritizedMemory
          (arbitrary fp32 priorities, ragged N, duplicate-index updates) and
          baseline/PER.py PER.sample / update / max_weight + the IS-weight lines
          of APE_X/ReplayMemory.py:65-67 (dyadic priorities, SURVEY §7).
  apex    APE_X/Learner.py Learner.train   (Q-values captured by wrapping forward)
  r2d2    R2D2/Learner.py Learner.train    (MEM=40, SURVEY §8a-note 1)
  impala  IMPALA/Learner.py Learner.train  (V-trace internals captured at calLoss)
  dropin  run_learner.py's Learner binding + baseline/baseAgent.py Q-values on seeded weights
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, REPO)


def _dyadic(rng, n):
    """k * 2^-10 priorities whose total is a power of two <= 2^24 units, so that
    every partial sum is exact in fp32 AND fp64 under any association (the flat
    reference sampler accumulates in fp32: 24 significand bits)."""
    import numpy as np

    kmax = max(2, min(1024, (1 << 23) // n))
    k = rng.integers(1, kmax + 1, size=n).astype(np.int64)
    tot = int(k.sum())
    goal = 1 << (tot - 1).bit_length()
    # spread the remainder over the elements, keeping every k >= 1
    rem = goal - tot
    add = rem // n
    k += add
    k[: rem - add * n] += 1
    assert int(k.sum()) == goal and goal <= (1 << 24)
    return (k.astype(np.float64) * 2.0 ** -10).astype(np.float32)


def gen_tree():
    import pickle
    import numpy as np
    import torch
    from oracle import ref_harness as H

    H.enter_reference("ape_x.json")
    from baseline.sumtree import SumTree          # type: ignore
    from baseline.utils import PrioritizedMemory  # type: ignore
    from baseline.PER import PER                  # type: ignore

    out = {}
    # ---- SumTree: arbitrary priorities, several sizes incl. ragged ------------
    for tag, n, nsamp in (("pow2", 4096, 512), ("ragged", 3000, 512), ("tiny", 5, 64), ("one", 1, 8)):
        rng = np.random.default_rng(0xB200 + n)
        prios32 = ((np.abs(rng.standard_normal(n)).clip(max=1) + 1e-7) ** 0.6).astype(np.float32)
        t = SumTree()
        t.extend([float(p) for p in prios32])
        np.random.seed(1234 + n)
        st = np.random.get_state()
        ixs, vals = t.prioritized_sample(nsamp)
        np.random.set_state(st)
        u01 = np.random.random_sample(nsamp)  # uniform(0, hi) == hi * random_sample()
        out[f"st_{tag}_prios"] = prios32
        out[f"st_{tag}_u01"] = u01
        out[f"st_{tag}_idx"] = np.array(ixs, np.int64)
        out[f"st_{tag}_vals"] = np.array(vals, np.float64)
        out[f"st_{tag}_total"] = np.float64(t.root.value)
        # duplicate-index update through PrioritizedMemory.update_priorities
        if n >= 5:
            pm = PrioritizedMemory(n)
            pm.priorities = t
            nupd = min(1000, 4 * n)
            uidx = rng.integers(0, n, size=nupd).astype(np.int64)
            uidx[-3:] = uidx[0]  # forced duplicates, last writer must win
            uval = ((np.abs(rng.standard_normal(nupd)).clip(max=1) + 1e-7) ** 0.6).astype(np.float32)
            pm.update_priorities([int(i) for i in uidx], [float(v) for v in uval])
            np.random.seed(99 + n)
            st = np.random.get_state()
            ixs2, vals2 = t.prioritized_sample(nsamp)
            np.random.set_state(st)
            out[f"st_{tag}_upd_idx"] = uidx
            out[f"st_{tag}_upd_val"] = uval
            out[f"st_{tag}_u01_after"] = np.random.random_sample(nsamp)
            out[f"st_{tag}_idx_after"] = np.array(ixs2, np.int64)
            out[f"st_{tag}_total_after"] = np.float64(t.root.value)
            out[f"st_{tag}_leaves_after"] = np.array([t[i] for i in range(n)], np.float64)

    # ---- PER (flat store): dyadic priorities ---------------------------------
    for tag, n, nsamp in (("4k", 4096, 512), ("64k", 65536, 512)):
        rng = np.random.default_rng(0xB200 + 7 * n)
        prios32 = _dyadic(rng, n)
        per = PER(maxlen=n, max_value=1.0, beta=0.4)
        blobs = [pickle.dumps([i, float(p)]) for i, p in enumerate(prios32)]  # last field = priority
        per.push(blobs)
        assert per.priority.prior_torch.dtype == torch.float32   # torch.tensor(list of floats)
        torch.manual_seed(1234)
        _, s_prob, idx = per.sample(nsamp)
        torch.manual_seed(1234)
        u01 = torch.rand(nsamp, dtype=torch.float64).numpy()
        nlen = len(per)
        weight = (1 / (nlen * s_prob)) ** 0.4            # APE_X/ReplayMemory.py:66
        max_w = per.max_weight                           # baseline/PER.py:129-133
        weight = weight / max_w                          # APE_X/ReplayMemory.py:67
        out[f"per_{tag}_prios"] = prios32
        out[f"per_{tag}_u01"] = u01
        out[f"per_{tag}_idx"] = idx.numpy().astype(np.int64)
        out[f"per_{tag}_prob"] = s_prob.numpy().astype(np.float32)
        out[f"per_{tag}_weight"] = weight.numpy().astype(np.float32)
        out[f"per_{tag}_max_weight"] = np.float64(max_w)
        # update with duplicates, then sample again
        nupd = 1024
        uidx = rng.integers(0, n, size=nupd).astype(np.int64)
        uidx[-2:] = uidx[5]
        uval = (rng.integers(1, 1025, size=nupd).astype(np.float64) * 2.0 ** -10).astype(np.float32)
        per.update([torch.tensor(int(i)) for i in uidx], uval)  # list of 0-d tensors, as the learner passes
        out[f"per_{tag}_upd_idx"] = uidx
        out[f"per_{tag}_upd_val"] = uval
        out[f"per_{tag}_prios_after"] = per.priority.prior_torch.numpy().astype(np.float32)

    # ---- PER on arbitrary fp32 priorities: pins the flat replay rule only ------
    n, nsamp = 8192, 512
    rng = np.random.default_rng(0xB200 + 3)
    prios32 = ((np.abs(rng.standard_normal(n)).clip(max=1) + 1e-7) ** 0.6).astype(np.float32)
    per = PER(maxlen=n, max_value=1.0, beta=0.4)
    per.push([pickle.dumps([0, float(p)]) for p in prios32])
    torch.manual_seed(77)
    _, s_prob, idx = per.sample(nsamp)
    torch.manual_seed(77)
    out["per_arb_prios"] = prios32
    out["per_arb_u01"] = torch.rand(nsamp, dtype=torch.float64).numpy()
    out["per_arb_idx"] = idx.numpy().astype(np.int64)
    out["per_arb_prob"] = s_prob.numpy().astype(np.float32)
    out["per_arb_max_weight"] = np.float64(per.max_weight)
    np.savez_compressed(os.path.join(HERE, "tree.npz"), **out)
    print("tree.npz:", len(out), "arrays")


def gen_apex():
    import numpy as np
    import torch
    from oracle import ref_harness as H

    H.enter_reference("ape_x.json")
    import configuration as C  # type: ignore

    out = {}
    for case, B in (("b32", 32), ("b8", 8)):
        C.BATCHSIZE = B
        torch.manual_seed(0)
        l = H.bare_learner("APE_X")
        # make the target net differ from the online net
        with torch.no_grad():
            for p in l.target_model.getParameters():
                p.add_(0.01 * torch.randn_like(p))
        rng = np.random.default_rng(0xB200 + B)
        s = rng.integers(0, 256, size=(B, 4, 84, 84), dtype=np.uint8)
        ns = rng.integers(0, 256, size=(B, 4, 84, 84), dtype=np.uint8)
        a = np.array([int(x) for x in rng.integers(0, 6, size=B)], dtype=object)
        r = np.array([float(x) for x in np.clip(rng.standard_normal(B) * 2, -1.5, 1.5)], dtype=object)
        d = np.array([bool(x) for x in (rng.random(B) < 0.25)], dtype=object)
        w = torch.from_numpy(rng.uniform(0.2, 1.0, size=B).astype(np.float32))
        idx = torch.arange(B)
        calls = {"m": [], "t": []}
        om, ot = l.model.forward, l.target_model.forward

        def ft(x, _o=ot):
            o = _o(x); calls["t"].append(o[0]); return o

        l.target_model.forward = ft
        # first online forward is Q(s) (APE_X/Learner.py:78); keep its grad = dLoss/dQ(s,.)
        grads = {}

        def fm_hook(x, _o=om):
            o = _o(x)
            calls["m"].append(o[0])
            if len(calls["m"]) == 1:
                o[0].retain_grad()
                grads["q"] = o[0]
            return o

        l.model.forward = fm_hook
        info, prio, idx_out, mean_w = l.train([s, a, r, ns, d, w, idx])
        out[f"{case}_q_s"] = calls["m"][0].detach().numpy()
        out[f"{case}_qn_online"] = calls["m"][1].detach().numpy()
        out[f"{case}_qn_target"] = calls["t"][0].detach().numpy()
        out[f"{case}_grad_q"] = grads["q"].grad.numpy()
        out[f"{case}_action"] = a.astype(np.int64)
        out[f"{case}_reward"] = r.astype(np.float32)
        out[f"{case}_done"] = d.astype(np.bool_)
        out[f"{case}_weight"] = w.numpy()
        out[f"{case}_new_priority"] = np.asarray(prio, np.float32)
        out[f"{case}_mean_value"] = np.float32(info["mean_value"])
        out[f"{case}_mean_weight"] = np.float32(mean_w)
        out[f"{case}_gamma_n"] = np.float64(0.99 ** C.UNROLL_STEP)
        out[f"{case}_alpha"] = np.float64(C.ALPHA)
    np.savez_compressed(os.path.join(HERE, "apex.npz"), **out)
    print("apex.npz:", len(out), "arrays")


def gen_r2d2():
    import numpy as np
    import torch
    from oracle import ref_harness as H

    # MEM = T/2 is the only setting for which the shipped R2D2/Learner.py:111 runs.
    T, MEM, B = 16, 8, 4
    H.enter_reference("r2d2.json", {"FIXED_TRAJECTORY": T, "MEM": MEM, "BATCHSIZE": B})
    import configuration as C  # type: ignore

    out = {}
    for case, seed in (("s0", 0), ("s1", 1)):
        torch.manual_seed(seed)
        l = H.bare_learner("R2D2")
        with torch.no_grad():
            for p in l.target_model.getParameters():
                p.add_(0.02 * torch.randn_like(p))
        rng = np.random.default_rng(0xB200 + seed)
        s = rng.integers(0, 256, size=(B, T, 4, 84, 84), dtype=np.uint8)
        a = rng.integers(0, 6, size=(B, T)).astype(np.int32)
        r = (rng.standard_normal((B, T)) * (3.0 if seed else 1.0)).astype(np.float32)
        notdone = np.array([float(x) for x in (rng.random(B) > 0.3)])
        w = torch.from_numpy(rng.uniform(0.2, 1.0, size=B).astype(np.float32))
        h0 = torch.from_numpy(rng.standard_normal((1, B, 512)).astype(np.float32)) * 0.1
        h1 = torch.from_numpy(rng.standard_normal((1, B, 512)).astype(np.float32)) * 0.1
        idx = torch.arange(B)
        calls = {"m": [], "t": []}
        om, ot = l.model.forward, l.target_model.forward
        grads = {}

        def fm(x, _o=om):
            o = _o(x)
            calls["m"].append(o[0])
            if len(calls["m"]) == 2:  # 1st call is the burn-in (:101), 2nd the window (:121)
                o[0].retain_grad(); grads["q"] = o[0]
            return o

        def ft(x, _o=ot):
            o = _o(x); calls["t"].append(o[0]); return o

        l.model.forward, l.target_model.forward = fm, ft
        info, prio, idx_out = l.train([(h0, h1), s, a, r, notdone, w, idx])
        L = T - MEM
        out[f"{case}_q"] = calls["m"][1].detach().numpy().reshape(L, B, 6)
        out[f"{case}_q_target"] = calls["t"][1].detach().numpy().reshape(L, B, 6)
        out[f"{case}_grad_q"] = grads["q"].grad.numpy().reshape(L, B, 6)
        out[f"{case}_action"] = np.transpose(a, (1, 0))[MEM:-1].astype(np.int64)
        out[f"{case}_reward"] = np.transpose(r, (1, 0))[MEM:-1].astype(np.float32)
        out[f"{case}_notdone"] = notdone
        out[f"{case}_weight"] = w.numpy()
        out[f"{case}_new_priority"] = np.asarray(prio, np.float32)
        out[f"{case}_mean_value"] = np.float32(info["mean_value"])
    out["n_step"] = np.int64(C.UNROLL_STEP)
    out["gamma"] = np.float64(C.GAMMA)
    out["alpha"] = np.float64(C.ALPHA)
    # value rescaling functions on a grid
    from R2D2.Learner import value_transform, value_inv_transform  # type: ignore
    x = torch.linspace(-30, 30, 2001)
    out["h_x"] = x.numpy()
    out["h_y"] = value_transform(x).numpy()
    out["hinv_y"] = value_inv_transform(x).numpy()
    np.savez_compressed(os.path.join(HERE, "r2d2.npz"), **out)
    print("r2d2.npz:", len(out), "arrays")


def gen_impala():
    import numpy as np
    import torch
    from oracle import ref_harness as H

    B = 8
    H.enter_reference("impala.json", {"BATCHSIZE": B})
    import configuration as C  # type: ignore

    T = C.UNROLL_STEP
    out = {}
    for case, seed, cval, pval, lam in (("c1", 0, 1.0, 1.0, 1), ("c2", 1, 0.8, 1.3, 0.9)):
        C.C_VALUE, C.P_VALUE, C.C_LAMBDA = cval, pval, lam
        import IMPALA.Learner as IL  # type: ignore
        IL.C_LAMBDA = lam
        torch.manual_seed(seed)
        l = H.bare_learner("IMPALA")
        l.c_value = torch.tensor(cval).float(); l.p_value = torch.tensor(pval).float()
        rng = np.random.default_rng(0xB200 + 40 + seed)
        s = rng.integers(0, 256, size=(T + 1, B, 4 * 84 * 84), dtype=np.uint8)
        a = rng.integers(0, 6, size=(T, B)).astype(np.int64)
        mu = rng.uniform(0.05, 0.9, size=(T, B)).astype(np.float32)
        r = rng.standard_normal((T, B)).astype(np.float32)
        done = (rng.random(B) > 0.3).astype(np.float32)
        rec = {}
        ofw = l.forward

        def fw(state, actionBatch, _o=ofw):
            p, v = _o(state, actionBatch); rec["pi"] = p; rec["v"] = v; return p, v

        l.forward = fw
        omf = l.model.forward
        first = {}

        def mf(x, _o=omf):
            o = _o(x)
            if "boot" not in first:
                first["boot"] = o[0][:, -1:].detach().clone()
            return o

        l.model.forward = mf
        ocl = l.calLoss

        def cl(state, actionTarget, criticTarget, action, _o=ocl):
            rec["adv"] = actionTarget.clone(); rec["vt"] = criticTarget.clone()
            return _o(state, actionTarget, criticTarget, action)

        l.calLoss = cl
        l.train((s, a, mu, r, done), 0)
        out[f"{case}_pi_a"] = rec["pi"].detach().numpy().reshape(T, B)
        out[f"{case}_value"] = rec["v"].detach().numpy().reshape(T, B)
        out[f"{case}_mu_a"] = mu
        out[f"{case}_reward"] = r
        out[f"{case}_bootstrap"] = (first["boot"][:, 0] * torch.from_numpy(done)).numpy()
        out[f"{case}_vtarget"] = rec["vt"].numpy().reshape(T, B)
        out[f"{case}_advantage"] = rec["adv"].numpy().reshape(T, B)
        out[f"{case}_params"] = np.array([C.GAMMA, lam, cval, pval], np.float64)
    np.savez_compressed(os.path.join(HERE, "impala.npz"), **out)
    print("impala.npz:", len(out), "arrays")


def seeded_weights(shapes, seed):
    """Network weights that both the reference (here) and the GPU test can regenerate from a seed."""
    import numpy as np
    rng = np.random.default_rng(seed)
    out = []
    for shp in shapes:
        fan_in = int(np.prod(shp[1:]))
        out.append((rng.uniform(-1, 1, size=shp) / np.sqrt(fan_in)).astype(np.float32))
    return out


def gen_apex_e2e():
    """Whole reference Learner.train (CPU) — network forward x3, target, loss, backward, centered
    RMSprop — on seeded weights and a seeded minibatch; records what train returns plus a slice of
    every updated weight tensor.  The GPU test replays it through distributed_rl_b200.apex.Learner."""
    import numpy as np
    import torch
    from oracle import ref_harness as H

    H.enter_reference("ape_x.json")
    import configuration as C  # type: ignore

    B = 16
    C.BATCHSIZE = B
    l = H.bare_learner("APE_X")
    out = {}
    for tag, model, seed in (("online", l.model, 101), ("target", l.target_model, 202)):
        sd = model.state_dict()
        names = list(sd.keys())
        ws = seeded_weights([tuple(sd[k].shape) for k in names], seed)
        model.load_state_dict({k: torch.from_numpy(w) for k, w in zip(names, ws)})
        out[f"{tag}_names"] = np.array(names)
    rng = np.random.default_rng(0xB200 + 99)
    s = rng.integers(0, 256, size=(B, 4, 84, 84), dtype=np.uint8)
    ns = rng.integers(0, 256, size=(B, 4, 84, 84), dtype=np.uint8)
    a = np.array([int(x) for x in rng.integers(0, 6, size=B)], dtype=object)
    r = np.array([float(x) for x in np.clip(rng.standard_normal(B), -1, 1)], dtype=object)
    d = np.array([bool(x) for x in (rng.random(B) < 0.25)], dtype=object)
    w = torch.from_numpy(rng.uniform(0.2, 1.0, size=B).astype(np.float32))
    info, prio, idx, mean_w = l.train([s, a, r, ns, d, w, torch.arange(B)])
    out["new_priority"] = np.asarray(prio, np.float32)
    out["mean_value"] = np.float32(info["mean_value"])
    out["p_norm"] = np.float32(info["p_norm"])
    for k, v in l.model.state_dict().items():
        out["after_" + k] = v.reshape(-1)[:256].numpy().copy()
    out["batch"] = np.int64(B)
    np.savez_compressed(os.path.join(HERE, "apex_e2e.npz"), **out)
    print("apex_e2e.npz:", len(out), "arrays")


def _load_seeded(model, seed):
    import numpy as np
    import torch
    sd = model.state_dict()
    names = list(sd.keys())
    ws = seeded_weights([tuple(sd[k].shape) if sd[k].dim() > 1 else (sd[k].shape[0], 64) for k in names], seed)
    fixed = {}
    for k, w in zip(names, ws):
        fixed[k] = torch.from_numpy(w if sd[k].dim() > 1 else np.ascontiguousarray(w[:, 0]))
    model.load_state_dict(fixed)
    return names


def gen_r2d2_e2e():
    """Whole reference R2D2 Learner.train on the CPU (burn-in, LSTM, targets, clip 40, Adam), MEM = T/2."""
    import numpy as np
    import torch
    from oracle import ref_harness as H

    T, MEM, B = 16, 8, 4
    H.enter_reference("r2d2.json", {"FIXED_TRAJECTORY": T, "MEM": MEM, "BATCHSIZE": B})
    l = H.bare_learner("R2D2")
    out = {"online_names": np.array(_load_seeded(l.model, 303)), "target_names": np.array(_load_seeded(l.target_model, 404))}
    rng = np.random.default_rng(0xB200 + 77)
    s = rng.integers(0, 256, size=(B, T, 4, 84, 84), dtype=np.uint8)
    a = rng.integers(0, 6, size=(B, T)).astype(np.int32)
    r = rng.standard_normal((B, T)).astype(np.float32)
    notdone = np.array([float(x) for x in (rng.random(B) > 0.3)])
    w = torch.from_numpy(rng.uniform(0.2, 1.0, size=B).astype(np.float32))
    h0 = torch.from_numpy((rng.standard_normal((1, B, 512)) * 0.1).astype(np.float32))
    h1 = torch.from_numpy((rng.standard_normal((1, B, 512)) * 0.1).astype(np.float32))
    info, prio, idx = l.train([(h0, h1), s, a, r, notdone, w, torch.arange(B)])
    out["new_priority"] = np.asarray(prio, np.float32)
    out["mean_value"] = np.float32(info["mean_value"])
    out["p_norm"] = np.float32(info["p_norm"])
    for k, v in l.model.state_dict().items():
        out["after_" + k] = v.reshape(-1)[:256].numpy().copy()
    out["dims"] = np.array([T, MEM, B], np.int64)
    np.savez_compressed(os.path.join(HERE, "r2d2_e2e.npz"), **out)
    print("r2d2_e2e.npz:", len(out), "arrays")


def gen_impala_e2e():
    """Whole reference IMPALA Learner.train on the CPU (V-trace, losses, clip 40, RMSprop)."""
    import numpy as np
    import torch
    from oracle import ref_harness as H

    B = 8
    H.enter_reference("impala.json", {"BATCHSIZE": B})
    import configuration as C  # type: ignore
    T = C.UNROLL_STEP
    l = H.bare_learner("IMPALA")
    out = {"names": np.array(_load_seeded(l.model, 505))}
    rng = np.random.default_rng(0xB200 + 55)
    s = rng.integers(0, 256, size=(T + 1, B, 4 * 84 * 84), dtype=np.uint8)
    a = rng.integers(0, 6, size=(T, B)).astype(np.int64)
    mu = rng.uniform(0.05, 0.9, size=(T, B)).astype(np.float32)
    r = rng.standard_normal((T, B)).astype(np.float32)
    done = (rng.random(B) > 0.3).astype(np.float32)
    l.train((s, a, mu, r, done), 0)
    for k, v in l.model.state_dict().items():
        out["after_" + k] = v.reshape(-1)[:256].numpy().copy()
    out["dims"] = np.array([T, B], np.int64)
    np.savez_compressed(os.path.join(HERE, "impala_e2e.npz"), **out)
    print("impala_e2e.npz:", len(out), "arrays")


def gen_dropin():
    """What the drop-in tests compare with: the Learner class the reference's run_learner.py binds under the Ape-X
    cfg, and the reference baseAgent's parameter names, shapes and Q-values on seeded weights and a seeded input."""
    import runpy
    import numpy as np
    import torch
    from oracle import ref_harness as H

    H.enter_reference("ape_x.json")
    L = runpy.run_path(os.path.join(H.REFERENCE_ROOT, "run_learner.py"), run_name="not_main")["Learner"]
    import configuration as C  # type: ignore
    from baseline.baseAgent import baseAgent  # type: ignore

    net = baseAgent(C.MODEL)
    names = _load_seeded(net, 606)
    x = np.random.default_rng(0xB200 + 66).random((5, 4, 84, 84), dtype=np.float32)
    with torch.no_grad():
        q = net.forward([torch.from_numpy(x)])[0].numpy()
    out = {"run_learner_alg": np.array(C.ALG), "run_learner_class": np.array(f"{L.__module__}.{L.__qualname__}"),
           "agent_names": np.array(names),
           "agent_shapes": np.array(["x".join(map(str, v.shape)) for v in net.state_dict().values()]),
           "agent_q": q}
    np.savez_compressed(os.path.join(HERE, "dropin.npz"), **out)
    print("dropin.npz:", len(out), "arrays")


GROUPS = {"tree": gen_tree, "apex": gen_apex, "r2d2": gen_r2d2, "impala": gen_impala, "apex_e2e": gen_apex_e2e,
          "r2d2_e2e": gen_r2d2_e2e, "impala_e2e": gen_impala_e2e, "dropin": gen_dropin}

if __name__ == "__main__":
    want = sys.argv[1:] or list(GROUPS)
    if len(want) == 1 and os.environ.get("B2RL_GOLDEN_CHILD") == "1":
        GROUPS[want[0]]()
    else:
        env = dict(os.environ, B2RL_GOLDEN_CHILD="1")
        for g in want:  # one interpreter per group: `configuration` is process-global
            subprocess.run([sys.executable, os.path.abspath(__file__), g], check=True, env=env)
