"""Discrete SAC on the GPU (pearl_b200/dsac.py, csrc/dsac.cu) against (a) the recordings of the reference
(tests/golden/dsac_small.npz with the entropy coefficient tuned, dsac_fixed.npz with it fixed: two learn() calls with one
ExponentialLR step of the actor learning rate between them) and (b) oracle/dsac_oracle.py at Pearl's SAC_method shape
(CartPole: obs 4, 2 actions, [64, 64], batch 32) and at a stress shape (obs 128, 16 actions, [256, 256], batch 256,
1e5-transition ring).  Tolerance: elementwise 1e-4 (tests/_tol.py)."""
import os
import random

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from oracle.dsac_oracle import OracleDiscreteSAC
from oracle.pearl_oracle import flat

pytestmark = pytest.mark.gpu

from _tol import close as _close, close_params as _close_params  # noqa: E402


def _fill(buf, st, ac, rw, ns, term, A):
    n = st.shape[0]
    buf.push_batch(torch.from_numpy(st), torch.from_numpy(ac).to(torch.int32), torch.from_numpy(rw), torch.from_numpy(ns),
                   torch.from_numpy(term), torch.zeros(n, dtype=torch.bool), max_number_actions=A)


def _data(n, obs, A, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    q8 = lambda x: (np.rint(x * 256) / 256).astype(np.float32)  # noqa: E731
    st, ns, rw = q8(rng.standard_normal((n, obs))), q8(rng.standard_normal((n, obs))), q8(rng.standard_normal(n))
    return st, rng.integers(0, A, size=n).astype(np.int64), rw, ns, rng.random(n) < 0.05


@pytest.mark.parametrize("name", ["dsac_small", "dsac_fixed"])
def test_dsac_matches_reference_recording(name):
    """Both learn() calls of the recording; the second at the learning rate the reference's reset() scheduled, set through
    prl_dsac_set_lr on the live handle."""
    import pearl_b200
    fx = np.load(os.path.join(GOLDEN, f"{name}.npz"))
    R, B, n, A, autotune = int(fx["rounds"]), int(fx["batch"]), int(fx["n"]), int(fx["n_act"]), bool(fx["autotune"])
    buf = pearl_b200.B200ReplayBuffer(n)
    _fill(buf, fx["state"], fx["action"], fx["reward"], fx["next_state"], fx["terminated"], A)
    lrs = fx["actor_lr_call"]
    pl = pearl_b200.B200SoftActorCritic(
        state_dim=int(fx["obs"]), n_actions=A, actor_hidden_dims=[32, 32], critic_hidden_dims=[32, 32], training_rounds=R,
        batch_size=B, actor_learning_rate=float(lrs[0]), critic_learning_rate=float(fx["critic_lr"]),
        critic_soft_update_tau=float(fx["tau"]), discount_factor=float(fx["gamma"]), entropy_coef=float(fx["entropy_coef"]),
        entropy_autotune=autotune)
    if autotune:
        assert np.float32(pl.target_entropy) == fx["target_entropy"]
    pl.load_parameters(fx["init_actor"], fx["init_q1"], fx["init_q2"], fx["init_q1t"], fx["init_q2t"])
    seed = int(fx["seed"])
    random.seed(seed)                                   # the state the recording sampled from
    pc = pl.critic_params.numel() // 2
    handle = None
    for call in (1, 2):
        if call == 2:
            pl.set_learning_rates(float(lrs[1]), float(fx["critic_lr"]))
        trace = {}
        rep = pl.learn(buf, trace=trace)
        assert trace["idx"].tolist() == fx["idx"][(call - 1) * R:call * R].tolist()      # bit-exact sampling
        if handle is None:
            handle = pl._handle.value
        assert pl._handle.value == handle                                                  # no re-creation for the new rate
        _close(rep["actor_loss"], fx[f"actor_loss{call}"], f"call {call}: actor_loss")
        _close(rep["critic_loss"], fx[f"critic_loss{call}"], f"call {call}: critic_loss")
        assert ("entropy_coef" in rep) == autotune
        if autotune:
            _close(rep["entropy_coef"], fx[f"entropy_loss{call}"], f"call {call}: entropy loss")
            _close(pl._log_entropy[:1].cpu().numpy(), fx[f"after{call}_log_entropy"], f"call {call}: log_alpha")
        _close([pl.entropy_coef], [float(fx[f"after{call}_entropy_coef"])], f"call {call}: alpha")
        _close(pl.actor_params.cpu().numpy(), fx[f"after{call}_actor"], f"call {call}: actor")
        _close(pl.critic_params[:pc].cpu().numpy(), fx[f"after{call}_q1"], f"call {call}: q1")
        _close(pl.critic_params[pc:].cpu().numpy(), fx[f"after{call}_q2"], f"call {call}: q2")
        _close(pl.critic_target_params[:pc].cpu().numpy(), fx[f"after{call}_q1t"], f"call {call}: q1 target")
        _close(pl.critic_target_params[pc:].cpu().numpy(), fx[f"after{call}_q2t"], f"call {call}: q2 target")
    assert pl.adam_step() == 2 * R
    # the python RNG advanced exactly as 2R calls of random.sample would have
    after = random.getstate()
    random.seed(seed)
    for _ in range(2 * R):
        random.sample(range(n), B)
    assert random.getstate() == after


def _adam_flat(opt, params, key):
    return torch.cat([opt.state[p][key].reshape(-1) for p in params])


def _sync_from_oracle(pl, orc):
    """Copy the oracle's parameters and optimizer states into the GPU learner (both have taken the same number of steps)."""
    pl.load_parameters(flat(orc.actor), flat(orc.q[0]), flat(orc.q[1]), flat(orc.qt[0]), flat(orc.qt[1]))
    ap = list(orc.actor.parameters())
    cp = list(orc.q[0].parameters()) + list(orc.q[1].parameters())
    for i, key in enumerate(("exp_avg", "exp_avg_sq", "max_exp_avg_sq")):
        pl._actor_state[i].copy_(_adam_flat(orc.opt_actor, ap, key))
        pl._critic_state[i].copy_(_adam_flat(orc.opt_critic, cp, key))
    if orc.autotune:
        st = orc.opt_alpha.state[orc.log_alpha]
        pl._log_entropy[:3].copy_(torch.stack([orc.log_alpha.detach()[0], st["exp_avg"][0], st["exp_avg_sq"][0]]))
        pl._entropy_coef.copy_(orc.alpha.reshape(1))


def _setup(obs, A, hidden, B, n, R, autotune, lr=(3e-4, 5e-4), seed=3):
    import pearl_b200
    torch.manual_seed(seed)
    torch.set_num_threads(4)
    st, ac, rw, ns, term = _data(n, obs, A, seed)
    orc = OracleDiscreteSAC(obs, A, (hidden, hidden), (hidden, hidden), actor_lr=lr[0], critic_lr=lr[1], gamma=0.99, tau=0.005,
                            entropy_coef=0.2, autotune=autotune)
    for m in [orc.actor] + orc.q:                          # xavier + 0.01 biases like the reference
        for mod in m.modules():
            if isinstance(mod, torch.nn.Linear):
                torch.nn.init.xavier_uniform_(mod.weight)
                mod.bias.data.fill_(0.01)
    for i in range(2):
        orc.qt[i].load_state_dict(orc.q[i].state_dict())
    buf = pearl_b200.B200ReplayBuffer(n)
    _fill(buf, st, ac, rw, ns, term, A)
    pl = pearl_b200.B200SoftActorCritic(
        state_dim=obs, n_actions=A, actor_hidden_dims=[hidden, hidden], critic_hidden_dims=[hidden, hidden], training_rounds=R,
        batch_size=B, actor_learning_rate=lr[0], critic_learning_rate=lr[1], critic_soft_update_tau=0.005, discount_factor=0.99,
        entropy_coef=0.2, entropy_autotune=autotune)
    pl.load_parameters(flat(orc.actor), flat(orc.q[0]), flat(orc.q[1]))

    def oracle_round(idx):
        t = lambda x: torch.from_numpy(x[idx])  # noqa: E731
        return orc.learn_batch(dict(state=t(st), action=t(ac), reward=t(rw), next_state=t(ns), terminated=t(term)))
    return pl, orc, buf, oracle_round


def _check_params(pl, orc, lr, rounds):
    pc = pl.critic_params.numel() // 2
    _close_params(pl.actor_params.cpu().numpy(), flat(orc.actor).numpy(), "actor", lr, rounds)
    _close_params(pl.critic_params[:pc].cpu().numpy(), flat(orc.q[0]).numpy(), "q1", lr, rounds)
    _close_params(pl.critic_params[pc:].cpu().numpy(), flat(orc.q[1]).numpy(), "q2", lr, rounds)
    _close_params(pl.critic_target_params[:pc].cpu().numpy(), flat(orc.qt[0]).numpy(), "q1 target", lr, rounds)
    _close_params(pl.critic_target_params[pc:].cpu().numpy(), flat(orc.qt[1]).numpy(), "q2 target", lr, rounds)
    _close([pl.entropy_coef], [float(orc.alpha)], "entropy coefficient")


@pytest.mark.parametrize("obs,A,hidden,B,n,autotune,graph,resync", [
    (4, 2, 64, 32, 2000, True, True, False),             # SAC_method (CartPole) shape
    (4, 2, 64, 32, 2000, False, False, False),
    (128, 16, 256, 256, 100_000, True, True, True),      # stress shape
    (128, 16, 256, 256, 100_000, False, False, True),
])
def test_dsac_against_oracle(obs, A, hidden, B, n, autotune, graph, resync):
    """CUDA-graph replay and plain launches, entropy autotune on and off.  The stress shape is checked step by step from a
    state re-synchronised with the oracle after every round: AdamW's FIRST step moves every element by exactly
    lr * sign(gradient), so an element whose gradient is zero to within fp32 summation noise can step the other way and then
    perturb its neighbours over the following rounds of an unsynchronised run (tests/test_sac.py documents the measurement)."""
    R = 5
    lr = (3e-4, 5e-4)
    pl, orc, buf, oracle_round = _setup(obs, A, hidden, B, n, R, autotune, lr)
    pl.use_cuda_graph = graph
    random.seed(77)
    if resync:
        pl._training_rounds = 1
        for r in range(R):
            trace = {}
            rep = pl.learn(buf, trace=trace)
            out = oracle_round(trace["idx"][0].tolist())
            _close(rep["actor_loss"], [out["actor_loss"]], "actor_loss")
            _close(rep["critic_loss"], [out["critic_loss"]], "critic_loss")
            if autotune:
                _close(rep["entropy_coef"], [out["entropy_coef"]], "entropy loss")
            _check_params(pl, orc, max(lr), 1)
            _sync_from_oracle(pl, orc)
        return
    trace = {}
    rep = pl.learn(buf, trace=trace)
    random.seed(77)
    outs = []
    for r in range(R):
        idx = random.sample(range(n), B)
        assert idx == trace["idx"][r].tolist()
        outs.append(oracle_round(idx))
    for k in rep:
        _close(rep[k], [o[k] for o in outs], k)
    _check_params(pl, orc, max(lr), R)


def test_dsac_learning_rate_change_keeps_the_handle():
    """New actor and critic learning rates between learn() calls reach the replayed round (no re-capture, same handle) and
    match the oracle stepping at the same rates."""
    R = 3
    lr = (3e-4, 5e-4)
    pl, orc, buf, oracle_round = _setup(4, 2, 64, 32, 2000, R, True, lr)
    random.seed(5)
    for call, (la, lc) in enumerate([lr, (lr[0] * 0.99, lr[1] * 0.5), (lr[0] * 0.99 * 0.99, lr[1] * 0.5)]):
        if call:
            handle = pl._handle.value
            pl.set_learning_rates(la, lc)
            orc.set_actor_lr(la)
            orc.set_critic_lr(lc)
        st = random.getstate()
        trace = {}
        rep = pl.learn(buf, trace=trace)
        if call:
            assert pl._handle.value == handle
        after = random.getstate()
        random.setstate(st)
        outs = [oracle_round(random.sample(range(2000), 32)) for _ in range(R)]
        assert random.getstate() == after
        for k in rep:
            _close(rep[k], [o[k] for o in outs], f"call {call}: {k}")
        _check_params(pl, orc, max(lr), R * (call + 1))
    assert pl.adam_step() == 3 * R


def test_dsac_refuses_unsupported_buffers():
    """prl_dsac_learn refuses (PRL_EINVAL, no device work: the buffer's sampler state is untouched) a continuous-action
    buffer, a buffer with per-transition action sets, a sharded buffer and mismatched dimensions."""
    import pearl_b200
    from pearl_b200 import _lib
    from pearl_b200.replay_buffer import _stream_ptr
    pl = pearl_b200.B200SoftActorCritic(state_dim=4, n_actions=3, actor_hidden_dims=[8, 8], critic_hidden_dims=[8, 8],
                                        training_rounds=1, batch_size=4)
    assert pl.learn(pearl_b200.B200ReplayBuffer(16)) == {}          # empty buffer: nothing to do (policy_learner.py:171-173)
    pl._bind(4)
    g = torch.Generator().manual_seed(0)

    def discrete(obs=4, A=3, ids=None, cnt=None):
        b = pearl_b200.B200ReplayBuffer(32, rng="device")
        b.push_batch(torch.randn(20, obs, generator=g), torch.randint(0, A, (20,), generator=g).to(torch.int32), torch.randn(20),
                     torch.randn(20, obs, generator=g), torch.zeros(20, dtype=torch.bool), torch.zeros(20, dtype=torch.bool),
                     next_available_ids=ids, next_available_count=cnt, max_number_actions=A)
        return b
    cont = pearl_b200.B200ReplayBuffer(32, rng="device")
    cont.is_action_continuous = True
    cont.push_batch(torch.randn(20, 4), torch.randn(20, 3), torch.randn(20), torch.randn(20, 4), torch.zeros(20, dtype=torch.bool),
                    torch.zeros(20, dtype=torch.bool))
    dyn = discrete(ids=torch.zeros(20, 3, dtype=torch.uint8), cnt=torch.ones(20, dtype=torch.int32))
    sharded = pearl_b200.B200ReplayBuffer(32, rng="device")
    sharded.push_batch_sharded(0, 2, torch.randn(40, 4), torch.randint(0, 3, (40,)).to(torch.int32), torch.randn(40), torch.randn(40, 4),
                               torch.zeros(40, dtype=torch.bool), torch.zeros(40, dtype=torch.bool), max_number_actions=3)
    out = torch.zeros((3, 1), dtype=torch.float32, device=pl._device)
    for what, b in [("continuous", cont), ("dynamic action sets", dyn), ("sharded", sharded), ("obs mismatch", discrete(obs=5)),
                    ("n_actions mismatch", discrete(A=4))]:
        before = b.get_rng_state()
        rc = pl._lib.prl_dsac_learn(pl._handle, b.handle, 1, 4, _lib.ptr(out[0]), _lib.ptr(out[1]), _lib.ptr(out[2]), None,
                                    _stream_ptr(pl._device))
        assert rc == _lib.PRL_EINVAL, (what, rc)
        assert np.array_equal(b.get_rng_state(), before), what
        assert not out.any(), what
    assert pl.adam_step() == 0
    with pytest.raises(ValueError):
        pl.learn(cont)
    with pytest.raises(ValueError):
        pl.learn(dyn)
    ok = discrete()
    assert len(pl.learn(ok)["actor_loss"]) == 1
    with pytest.raises(NotImplementedError):
        pearl_b200.B200SoftActorCritic(state_dim=4, n_actions=3, actor_hidden_dims=[8], critic_hidden_dims=[8, 8])
    with pytest.raises(ValueError):
        pearl_b200.B200SoftActorCritic(state_dim=4, actor_hidden_dims=[8, 8], critic_hidden_dims=[8, 8])


@pytest.mark.parametrize("graph", [True, False])
def test_dsac_is_deterministic(graph):
    """Two learners with the same seed, buffer contents and index stream are bit-identical (fixed summation orders)."""
    import pearl_b200
    st, ac, rw, ns, term = _data(5000, 128, 16, 11)
    runs = []
    for _ in range(2):
        buf = pearl_b200.B200ReplayBuffer(5000)
        _fill(buf, st, ac, rw, ns, term, 16)
        pl = pearl_b200.B200SoftActorCritic(state_dim=128, n_actions=16, actor_hidden_dims=[256, 256], critic_hidden_dims=[256, 256],
                                            training_rounds=4, batch_size=256, actor_learning_rate=3e-4, critic_learning_rate=3e-4,
                                            seed=21)
        pl.use_cuda_graph = graph
        random.seed(8)
        rep = pl.learn(buf)
        runs.append((rep, pl.actor_params.cpu(), pl.critic_params.cpu(), pl.critic_target_params.cpu(), pl._log_entropy.cpu()))
    (r1, *t1), (r2, *t2) = runs
    assert r1 == r2
    assert all(torch.equal(a, b) for a, b in zip(t1, t2))
