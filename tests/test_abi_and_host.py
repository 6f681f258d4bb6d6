"""CPU-side checks: the C-ABI library loads and exports every symbol the header
declares (no compute without a GPU), the product fails loudly without CUDA, host
logic (layout arithmetic, error mapping), and — where facebookresearch/Pearl is
available (tests/_pearl.py) — that the plugins subclass Pearl's own base classes."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

from _pearl import PEARL_ROOT
from conftest import ROOT

HEADER = os.path.join(ROOT, "include", "pearl_b200.h")


def declared_symbols():
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(prl_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from pearl_b200 import _lib, build
    build.build()
    lib = ctypes.CDLL(_lib.LIB_PATH)
    names = declared_symbols()
    assert len(names) >= 30
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/pearl_b200.h but not exported"
    # and the ctypes table binds exactly the declared set
    assert sorted(_lib.EXPORTS) == names
    assert _lib.load().prl_abi_version() == 1


def test_layout_arithmetic_is_host_only():
    from pearl_b200 import _lib
    lib = _lib.load()
    d = _lib.BufDesc(1_000_000, 128, 1, 16, _lib.PRL_BUF_DISCRETE)
    lay = _lib.BufLayout()
    assert lib.prl_buf_layout_of(ctypes.byref(d), ctypes.byref(lay)) == 0
    assert lay.record_words * 4 == 1040 and lay.storage_bytes == 1_040_000_000
    assert (lay.off_state, lay.off_next_state, lay.off_action, lay.off_reward, lay.off_flags) == (0, 128, 256, 257, 258)
    d = _lib.BufDesc(10, 6, 1, 5, _lib.PRL_BUF_DISCRETE | _lib.PRL_BUF_DYNAMIC_ACTIONS)
    assert lib.prl_buf_layout_of(ctypes.byref(d), ctypes.byref(lay)) == 0
    assert lay.off_next_state == 8 and lay.record_words % 4 == 0 and lay.off_avail == 19
    d = _lib.BufDesc(10, 376, 17, 0, _lib.PRL_BUF_CONTINUOUS)
    assert lib.prl_buf_layout_of(ctypes.byref(d), ctypes.byref(lay)) == 0
    assert lay.act_words == 17 and lay.record_words * 4 >= 3082
    bad = _lib.BufDesc(0, 4, 1, 2, _lib.PRL_BUF_DISCRETE)
    assert lib.prl_buf_layout_of(ctypes.byref(bad), ctypes.byref(lay)) == _lib.PRL_EINVAL
    with pytest.raises(ValueError):
        _lib.check(lib.prl_buf_layout_of(ctypes.byref(bad), ctypes.byref(lay)))
    assert "capacity" in _lib.last_error()


def test_param_count_matches_torch_module():
    from pearl_b200 import _lib
    lib = _lib.load()
    cfg = _lib.DqnCfg(obs_dim=128, n_actions=16, hidden1=64, hidden2=64, target_update_freq=10, max_batch=256,
                      max_rounds=16)
    assert lib.prl_dqn_param_count(ctypes.byref(cfg)) == 13505
    assert lib.prl_dqn_workspace_bytes(ctypes.byref(cfg)) > 0


def test_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import pearl_b200
    with pytest.raises(RuntimeError):
        pearl_b200.B200ReplayBuffer(16)
    from pearl_b200 import _lib
    assert _lib.load().prl_init(0) != 0  # no device -> error code, never a silent CPU path


def test_product_never_imports_the_oracle():
    """The oracle is a checker: nothing under pearl_b200/ may import, include, load or execute it
    (comments may cite it as the specification)."""
    bad = re.compile(r"^\s*(from|import)\s+oracle\b|#\s*include\s*[\"<][^\">]*oracle|liboracle|CDLL\([^)]*oracle|"
                     r"(subprocess|os\.system|exec|__import__)[^\n]*oracle", re.M)
    for dirpath, _, files in os.walk(os.path.join(ROOT, "pearl_b200")):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not bad.search(src), f"{f} uses the oracle"


@pytest.mark.skipif(PEARL_ROOT is None, reason="facebookresearch/Pearl is not available")
def test_plugins_subclass_pearl_when_available():
    code = (
        "import sys; sys.path[:0]=[%r, %r, %r]\n"
        "import pearl_b200\n"
        "from pearl.replay_buffers.replay_buffer import ReplayBuffer\n"
        "from pearl.policy_learners.sequential_decision_making.deep_q_learning import DeepQLearning\n"
        "from pearl.policy_learners.sequential_decision_making.double_dqn import DoubleDQN\n"
        "from pearl.policy_learners.policy_learner import PolicyLearner\n"
        "assert pearl_b200.HAVE_PEARL\n"
        "assert issubclass(pearl_b200.B200ReplayBuffer, ReplayBuffer)\n"
        "assert issubclass(pearl_b200.B200DeepQLearning, DeepQLearning)\n"
        "assert issubclass(pearl_b200.B200DoubleDQN, DoubleDQN) and issubclass(pearl_b200.B200DoubleDQN, PolicyLearner)\n"
        "from pearl.policy_learners.sequential_decision_making.soft_actor_critic_continuous import ContinuousSoftActorCritic\n"
        "from pearl.policy_learners.sequential_decision_making.ppo import ProximalPolicyOptimization\n"
        "from pearl.policy_learners.sequential_decision_making.td3 import TD3\n"
        "from pearl.policy_learners.sequential_decision_making.ddpg import DeepDeterministicPolicyGradient\n"
        "assert issubclass(pearl_b200.B200ContinuousSoftActorCritic, ContinuousSoftActorCritic)\n"
        "assert issubclass(pearl_b200.B200ProximalPolicyOptimization, ProximalPolicyOptimization)\n"
        "assert issubclass(pearl_b200.B200TD3, TD3) and issubclass(pearl_b200.B200DeepDeterministicPolicyGradient, DeepDeterministicPolicyGradient)\n"
        "assert not issubclass(pearl_b200.B200DeepDeterministicPolicyGradient, TD3)\n"
        "import torch\n"
        "from pearl.utils.instantiations.spaces.box_action import BoxActionSpace\n"
        "l = pearl_b200.B200ContinuousSoftActorCritic(state_dim=6, action_space=BoxActionSpace(-torch.ones(2), torch.ones(2)),\n"
        "        actor_hidden_dims=[32, 32], critic_hidden_dims=[32, 32], seed=3)\n"
        "class Buf:\n"
        "    def __len__(self): return 4\n"
        "try:\n"
        "    l.learn(Buf()); raise SystemExit('a CPU learner must not learn')\n"
        "except RuntimeError as e:\n"
        "    assert 'no CPU path' in str(e)\n"
        "from pearl.replay_buffers.transition import TransitionBatch\n"
        "assert pearl_b200.TransitionBatch is TransitionBatch\n"
        "print('ok')\n" % (os.path.join(ROOT, "oracle", "stubs"), PEARL_ROOT, ROOT))
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env)
    assert out.returncode == 0 and "ok" in out.stdout, out.stderr[-2000:]


@pytest.mark.skipif(PEARL_ROOT is None, reason="facebookresearch/Pearl is not available")
def test_actor_critic_plugins_bind_reference_modules_to_flat_vectors():
    """Host logic of pearl_b200/actor_critic.py against a stand-in learner (tests/actor_critic_host_worker.py): constructor
    arguments, parameters / AdamW state as views, step counts, SAC's entropy block, checkpoint import into a fresh and into an
    already bound learner, refusal of unsupported optimizers and network shapes."""
    env = dict(os.environ, PYTHONDONTWRITEBYTECODE="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "actor_critic_host_worker.py"), PEARL_ROOT],
                         capture_output=True, text=True, env=env, timeout=600)
    assert out.returncode == 0 and "ACTOR_CRITIC_HOST_OK" in out.stdout, (out.stdout[-1500:], out.stderr[-4000:])


def test_ctypes_signatures_match_the_header_arity():
    """Every ctypes binding takes exactly as many arguments as the C declaration (a mismatch would corrupt the call
    silently); pointer / integer / floating classes are compared as well."""
    from pearl_b200 import _lib
    src = open(HEADER).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"typedef struct[^;{]*\{.*?\}[^;]*;", "", src, flags=re.S)
    decls = dict(re.findall(r"\b(prl_[a-z0-9_]+)\s*\(([^;{]*?)\)\s*;", src, flags=re.S))
    assert set(decls) == set(_lib.EXPORTS)

    def kind(c_param: str) -> str:
        p = " ".join(c_param.split())
        if "*" in p or "[" in p:          # arrays decay to pointers
            return "ptr"
        base = p.rsplit(" ", 1)[0] if " " in p else p
        return "float" if base in ("float", "double") else "int"

    def ckind(t) -> str:
        if t in (ctypes.c_float, ctypes.c_double):
            return "float"
        if t in (ctypes.c_int, ctypes.c_int32, ctypes.c_int64, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_uint):
            return "int"
        return "ptr"
    for name, params in decls.items():
        plist = [] if params.strip() in ("", "void") else [p for p in params.split(",")]
        _, argtypes = _lib._SIGNATURES[name]
        assert len(plist) == len(argtypes), f"{name}: header has {len(plist)} parameters, ctypes table {len(argtypes)}"
        for i, (cp, at) in enumerate(zip(plist, argtypes)):
            assert kind(cp) == ckind(at), f"{name} argument {i}: `{' '.join(cp.split())}` bound as {at}"
