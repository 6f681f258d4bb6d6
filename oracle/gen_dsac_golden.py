#!/usr/bin/env python
"""Generate the discrete soft actor-critic fixtures tests/golden/dsac_small.npz (entropy coefficient tuned) and
dsac_fixed.npz (fixed coefficient) by RUNNING THE REFERENCE.

TEST INFRASTRUCTURE, like oracle/gen_golden.py, whose environment (the reference on sys.path with the test-only stubs of
oracle/stubs/) and helpers it reuses.  It cannot run where the reference is absent; its outputs are committed.

    PYTHONDONTWRITEBYTECODE=1 python oracle/gen_dsac_golden.py

Running it again gives identical arrays (seeded data quantised to a 1/256 grid, seeded torch and CPython RNGs, one thread).
"""
from __future__ import annotations

import os
import random
import sys

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from oracle.gen_golden import (GOLDEN, BasicReplayBuffer, DiscreteActionSpace,  # noqa: E402
                               OneHotActionTensorRepresentationModule, PearlAgent)


def gen_dsac_golden(name="dsac_small", *, autotune=True, entropy_coef=0.2, seed=43):
    """Discrete SAC: PearlAgent(SoftActorCritic, BasicReplayBuffer, OneHotActionTensorRepresentationModule(A)).learn(), then
    agent.reset() (one ExponentialLR step of the actor learning rate, soft_actor_critic.py:147-149) and a second learn().
    A discrete SAC step draws no random numbers: the sampled indices pin every float of both calls."""
    from pearl.policy_learners.sequential_decision_making.soft_actor_critic import SoftActorCritic
    torch.manual_seed(seed)
    random.seed(seed)
    torch.set_num_threads(1)
    obs, A, n, B, rounds = 11, 5, 300, 64, 6
    space = DiscreteActionSpace(actions=list(torch.arange(A).view(-1, 1)))
    hp = dict(actor_lr=3e-4, critic_lr=5e-4, tau=0.05, gamma=0.98)
    pl = SoftActorCritic(state_dim=obs, action_space=space, actor_hidden_dims=[32, 32], critic_hidden_dims=[32, 32],
                         training_rounds=rounds, batch_size=B, actor_learning_rate=hp["actor_lr"], critic_learning_rate=hp["critic_lr"],
                         critic_soft_update_tau=hp["tau"], discount_factor=hp["gamma"], entropy_coef=entropy_coef,
                         entropy_autotune=autotune, action_representation_module=OneHotActionTensorRepresentationModule(A))
    buf = BasicReplayBuffer(n)
    agent = PearlAgent(policy_learner=pl, replay_buffer=buf, device_id=-1)
    rng = np.random.Generator(np.random.PCG64(seed + 100))
    q8 = lambda x: (np.rint(x * 256) / 256).astype(np.float32)  # noqa: E731
    st, ns, rw = q8(rng.standard_normal((n, obs))), q8(rng.standard_normal((n, obs))), q8(rng.standard_normal(n))
    ac = rng.integers(0, A, size=n).astype(np.int64)
    term = rng.random(n) < 0.05
    for i in range(n):
        buf.push(state=torch.from_numpy(st[i]), action=torch.tensor(int(ac[i])), reward=float(rw[i]), terminated=bool(term[i]),
                 truncated=False, curr_available_actions=space, next_state=torch.from_numpy(ns[i]), next_available_actions=space,
                 max_number_actions=A)
    fl = lambda m: np.concatenate([p.detach().numpy().ravel() for p in m.parameters()])  # noqa: E731

    def nets(tag):
        return {f"{tag}_actor": fl(pl._actor), f"{tag}_q1": fl(pl._critic._critic_1), f"{tag}_q2": fl(pl._critic._critic_2),
                f"{tag}_q1t": fl(pl._critic_target._critic_1), f"{tag}_q2t": fl(pl._critic_target._critic_2)}

    def entropy_state(tag):
        if not autotune:
            return {f"{tag}_entropy_coef": np.float32(float(pl._entropy_coef))}
        s = pl._entropy_optimizer.state[pl._log_entropy]
        return {f"{tag}_log_entropy": pl._log_entropy.detach().numpy().copy(), f"{tag}_entropy_exp_avg": s["exp_avg"].numpy().copy(),
                f"{tag}_entropy_exp_avg_sq": s["exp_avg_sq"].numpy().copy(), f"{tag}_entropy_coef": np.float32(float(pl._entropy_coef))}

    idxs = []
    orig_sample = buf.sample

    def sample_spy(k):
        pos = {id(t): j for j, t in enumerate(buf.memory)}
        stt = random.getstate()
        idxs.append([pos[id(t)] for t in random.sample(buf.memory, k)])
        random.setstate(stt)
        return orig_sample(k)
    buf.sample = sample_spy
    out = dict(obs=obs, n_act=A, n=n, batch=B, rounds=rounds, seed=seed, autotune=autotune, entropy_coef=entropy_coef, **hp,
               state=st, next_state=ns, reward=rw, action=ac, terminated=term,
               target_entropy=np.float32(float(pl._target_entropy)) if autotune else np.float32(0.0), **nets("init"))
    lrs = []
    for call in (1, 2):
        if call == 2:
            agent.reset(torch.from_numpy(st[0]), space)                  # one scheduler step of the actor learning rate
        lrs.append(float(pl._actor_optimizer.param_groups[0]["lr"]))
        rep = agent.learn()
        out[f"actor_loss{call}"] = np.asarray(rep["actor_loss"])
        out[f"critic_loss{call}"] = np.asarray(rep["critic_loss"])
        if autotune:
            out[f"entropy_loss{call}"] = np.asarray([float(x.detach()) for x in rep["entropy_coef"]])
        out.update(nets(f"after{call}"))
        out.update(entropy_state(f"after{call}"))
    assert len(idxs) == 2 * rounds and lrs[1] == lrs[0] * 0.99
    out.update(idx=np.asarray(idxs, dtype=np.int32), actor_lr_call=np.asarray(lrs, dtype=np.float64))
    np.savez_compressed(os.path.join(GOLDEN, f"{name}.npz"), **out)
    print(f"{name}.npz: actor_loss", out["actor_loss1"][:2], "critic_loss", out["critic_loss1"][:2])



if __name__ == "__main__":
    os.makedirs(GOLDEN, exist_ok=True)
    gen_dsac_golden("dsac_small")
    gen_dsac_golden("dsac_fixed", autotune=False, entropy_coef=0.1, seed=44)
