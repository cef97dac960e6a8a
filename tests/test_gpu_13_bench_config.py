"""Parity AT THE BENCHMARKED CONFIGURATION (bench.py, BASELINE.json configs[1]): Ape-X, 2^20 slots, batch 512, the whole
step replayed as a CUDA graph, PyTorch's default library precision (TF32 convolutions) with cuDNN's heuristic, deterministic
algorithm choice — what bench.py's line is measured on, not a reduced stand-in."""
import numpy as np
import pytest

from oracle import oracle as O

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

LOG2N, B, STEPS = 20, 512, 50


def test_graph_replays_at_bench_config_match_the_oracle_step_by_step():
    """50 graph replays; after each, the step's indices / IS weights / new priorities are read back and checked
    against the numpy oracle that replays the SAME sequence: draws from the device Philox stream
    (`philox_u01(seed, counter)`) through the binary `SumTreeOracle` must give bit-identical indices, the IS weights
    must agree to 2 ulp, and after the oracle applies the GPU's priorities (last writer wins) the two trees must
    hold bit-identical leaves and roots at every step.  Then the target kernel is checked on the step's own Q."""
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    free, _ = torch.cuda.mem_get_info()
    if free < 70 << 30:
        pytest.skip("needs ~62 GB of free HBM (2^20 Ape-X slots)")
    from distributed_rl_b200 import apex, replay as R
    torch.backends.cudnn.benchmark = False             # the bench's library knobs (bench.py reproducible_cudnn)
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.allow_tf32 = True
    N = 1 << LOG2N
    cfg = apex.ApexConfig(BATCHSIZE=B, REPLAY_MEMORY_LEN=N, BUFFER_SIZE=0, LEARNER_DEVICE="cuda:0", CUDNN_BENCHMARK=False)
    torch.manual_seed(0)
    L = apex.Learner(cfg, connect=None, start_replay=False)
    st = L.memory.store
    st.fill_hash(N, seed=0xB200)
    g = torch.Generator(device="cuda"); g.manual_seed(0xB201)
    st.field_view("action").copy_(torch.randint(0, 6, (N,), device="cuda", generator=g, dtype=torch.int32))
    st.field_view("reward").copy_(torch.randn(N, device="cuda", generator=g).clamp_(-1, 1))
    st.field_view("done").copy_((torch.rand(N, device="cuda", generator=g) < 0.02).to(torch.uint8))
    prios = (torch.randn(N, device="cuda", generator=g).abs().clamp(max=1) + 1e-7) ** cfg.ALPHA
    st.build(prios)
    seed = 1234
    st.seed(seed, 0)
    tree = O.SumTreeOracle(N)
    tree.build(prios.cpu().numpy())
    assert st.stats(cfg.BETA).cpu().numpy()[0] == tree.total

    # the first call runs 3 eager warm-ups + capture (no execution) + 1 replay = 4 bodies; the oracle replays those too,
    # but their (idx, prio) are not observable -> start the bookkeeping after a rebuild of the tree
    L.fused_step(use_graph=True)
    torch.cuda.synchronize()
    st.build(prios)
    counter = 4 * B                                     # draws consumed so far; build() does not touch the RNG
    mism = 0
    for step in range(STEPS):
        out = L.fused_step(use_graph=True)
        torch.cuda.synchronize()
        idx = L._cur["idx"].cpu().numpy(); w = L._cur["w"].cpu().numpy(); prio = out["prio"].cpu().numpy()
        u = O.philox_u01(seed, counter, B)
        counter += B
        oidx, _ = tree.sample(u)
        np.testing.assert_array_equal(idx, oidx, err_msg=f"step {step}")                     # bit-exact draws
        ow, _, _ = O.is_weights(tree.sum[tree.cap + oidx].astype(np.float32), tree.total, tree.min_priority, N, cfg.BETA)
        np.testing.assert_allclose(w, ow, rtol=2.4e-7, err_msg=f"step {step}")
        a = st.field_view("action")[L._cur["idx"]].cpu().numpy()
        assert np.array_equal(L._cur["action"].cpu().numpy(), a)                             # scalars fetched by the draw
        tree.update(oidx, prio)                                                              # last writer wins
        root = st.stats(cfg.BETA).cpu().numpy()
        assert root[0] == tree.total and np.float32(root[1]) == tree.min_priority, step
        assert np.isfinite(prio).all() and (prio > 0).all()
    np.testing.assert_array_equal(st.priorities().cpu().numpy().astype(np.float64), tree.leaves())

    # target / TD / priority kernel on the step's OWN Q tensors (TF32 convolutions and all): capture them eagerly
    cap = {}
    orig = R.apex_target

    def spy(q, qo, qt, a, r, nd, ww, gamma_n, alpha, **kw):
        res = orig(q, qo, qt, a, r, nd, ww, gamma_n, alpha, **kw)
        cap.update(q=q, qo=qo, qt=qt, a=a, r=r, nd=nd, w=ww, out=res)
        return res

    R.apex_target = spy
    try:
        L._graph = None
        L.fused_step(use_graph=False)
        torch.cuda.synchronize()
    finally:
        R.apex_target = orig
    c = {k: v.cpu().numpy() for k, v in cap.items() if k != "out"}
    tgt, td, oprio, gq, info = O.apex_target(c["q"], c["qo"], c["qt"], c["a"], c["r"], c["nd"], c["w"], L.gamma_n, cfg.ALPHA)
    np.testing.assert_array_equal(cap["out"]["td"].cpu().numpy(), td)                        # fp32 op-by-op: bit-exact
    np.testing.assert_allclose(cap["out"]["prio"].cpu().numpy(), oprio, rtol=2.4e-7)
    np.testing.assert_allclose(cap["out"]["target"].cpu().numpy(), tgt, rtol=0, atol=1e-5)
    st.close()
