"""TEST INFRASTRUCTURE — loader for the UNMODIFIED reference (build container only).

Imports seungju-k1m/Distributed_RL from /root/reference (read-only, never copied)
so that `tests/golden/make_golden.py` can execute the reference's own functions
and record their outputs as golden vectors.  /root/reference does not exist on
GPU machines, so nothing under tests/ -m gpu, bench.py or smoke() may use
this module to load it; only the golden generator does.

What has to be shimmed for the reference to import under python 3.12 /
numpy 2.3 / torch 2.11 (SURVEY.md §8c):
  * `numpy.lib.arraysetops` (removed module, imported but unused at
    baseline/PER.py:3)                      -> alias exposing `isin`
  * `redis` (not installed)                 -> in-memory stub with the calls the
    learners make (APE_X/Learner.py:26,41-43,152-155; IMPALA/Learner.py:237-240)
  * `configuration.py:11` hard-codes ./cfg/ape_x.json and mkdirs ./log ./weight
    in the cwd (:16-32)                     -> run from a temp cwd holding a copy
    of the wanted cfg with LEARNER_DEVICE=cpu
"""
from __future__ import annotations

import json
import os
import sys
import tempfile
import types

REFERENCE_ROOT = os.environ.get("B2RL_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "baseline", "PER.py"))


class _Pipe:
    def __init__(self, store):
        self._s = store
        self._out = []

    def lrange(self, key, a, b):
        self._out.append(list(self._s.get(key, [])))

    def ltrim(self, key, a, b):
        self._s[key] = []

    def execute(self):
        out, self._out = self._out, []
        return out


class _StrictRedis:
    """In-memory stand-in for redis.StrictRedis (only what the learners call)."""

    def __init__(self, host=None, port=6379, **kw):
        self._s = {}

    def pipeline(self):
        return _Pipe(self._s)

    def set(self, k, v):
        self._s[k] = v

    def get(self, k):
        return self._s.get(k)

    def delete(self, *keys):
        for k in keys:
            self._s.pop(k, None)

    def rpush(self, k, v):
        self._s.setdefault(k, []).append(v)
        return len(self._s[k])

    def scan(self):
        return (0, list(self._s.keys()))


def install_shims() -> None:
    import numpy as np

    if "numpy.lib.arraysetops" not in sys.modules:
        m = types.ModuleType("numpy.lib.arraysetops")
        m.isin = np.isin
        sys.modules["numpy.lib.arraysetops"] = m
    if "redis" not in sys.modules:
        r = types.ModuleType("redis")
        r.StrictRedis = _StrictRedis
        r.Redis = _StrictRedis
        sys.modules["redis"] = r


def enter_reference(alg_cfg: str = "ape_x.json", overrides: dict | None = None) -> str:
    """chdir into a scratch cwd holding cfg/ape_x.json (= the requested cfg,
    LEARNER_DEVICE forced to cpu) and put the reference on sys.path.
    One algorithm per interpreter: `configuration` is a module of globals."""
    if not reference_available():
        raise RuntimeError(f"reference not found under {REFERENCE_ROOT}")
    install_shims()
    work = tempfile.mkdtemp(prefix="b2rl_ref_")
    os.makedirs(os.path.join(work, "cfg"))
    with open(os.path.join(REFERENCE_ROOT, "cfg", alg_cfg)) as f:
        cfg = json.load(f)
    cfg["LEARNER_DEVICE"] = "cpu"
    cfg["DEVICE"] = "cpu"
    if overrides:
        cfg.update(overrides)
    with open(os.path.join(work, "cfg", "ape_x.json"), "w") as f:
        json.dump(cfg, f)
    os.chdir(work)
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    return work


def bare_learner(alg: str):
    """Construct a reference Learner without its __init__ side effects
    (mkdir, Replay thread, SummaryWriter, Redis flush): object.__new__ +
    the two builder calls, as SURVEY.md §8c prescribes."""
    import torch

    if alg == "APE_X":
        from APE_X.Learner import Learner  # type: ignore

        l = object.__new__(Learner)
        l.device = torch.device("cpu")
        l.build_model()
        l.build_optim()
        return l
    if alg == "R2D2":
        import numpy as np
        import configuration as C  # type: ignore
        from R2D2.Learner import Learner  # type: ignore

        l = object.__new__(Learner)
        l.device = torch.device("cpu")
        l.build_model()
        l.build_optim()
        # R2D2/Learner.py:61-62
        l.action_idx = torch.tensor(
            [C.ACTION_SIZE * i for i in range(C.BATCHSIZE * (C.FIXED_TRAJECTORY - C.MEM))]
        )
        l.action_idx_np = np.array(
            [C.ACTION_SIZE * i for i in range(C.BATCHSIZE * (C.FIXED_TRAJECTORY - C.MEM - 1))]
        )
        return l
    if alg == "IMPALA":
        import configuration as C  # type: ignore
        from IMPALA.Learner import Learner  # type: ignore

        class _W:
            def add_scalar(self, *a, **k):
                pass

            def add_text(self, *a, **k):
                pass

        l = object.__new__(Learner)
        l.device = torch.device("cpu")
        l.buildModel()
        l.genOptim()
        l._connect = _StrictRedis()
        l.writer = _W()
        # IMPALA/Learner.py:49-52
        l.c_value = torch.tensor(C.C_VALUE).float()
        l.p_value = torch.tensor(C.P_VALUE).float()
        l.div = torch.tensor(255).float()
        return l
    raise ValueError(alg)
