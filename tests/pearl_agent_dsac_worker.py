"""Worker of tests/test_pearl_agent_dsac_gpu.py: B200SoftActorCritic as a SUBCLASS of the reference's discrete SoftActorCritic
(pearl_b200/actor_critic.py), (1) against the stand-alone CUDA learner it wraps, bit for bit, over two learn() calls with a
reset() (one ExponentialLR step of the actor learning rate) between them, (2) under the reference's own PearlAgent facade
(pearl/pearl_agent.py:55-330: reset -> act -> observe -> learn) with the C handle surviving every reset, (3) through a
checkpoint round trip of `agent.state_dict()` (actor_critic_base.py:411-428) after which both agents continue identically.
The numerics against recordings of the reference are tests/test_dsac.py; this file is about the plugin boundary.  Test
infrastructure: needs facebookresearch/Pearl on sys.path (argv[1] = its root) plus the test-only gymnasium / matplotlib stubs."""
import io
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.dont_write_bytecode = True
sys.path[:0] = [os.path.join(ROOT, "oracle", "stubs"), sys.argv[1], ROOT]

import torch  # noqa: E402

import pearl_b200  # noqa: E402
from pearl_b200 import actor_critic as ac  # noqa: E402
from pearl.action_representation_modules.one_hot_action_representation_module import OneHotActionTensorRepresentationModule  # noqa: E402
from pearl.api.action_result import ActionResult  # noqa: E402
from pearl.pearl_agent import PearlAgent  # noqa: E402
from pearl.policy_learners.sequential_decision_making.soft_actor_critic import SoftActorCritic  # noqa: E402
from pearl.utils.instantiations.spaces.discrete_action import DiscreteActionSpace  # noqa: E402

assert pearl_b200.HAVE_PEARL and ac.HAVE_REFERENCE
OBS, NACT, CAP, B, ROUNDS, STEPS = 10, 4, 400, 32, 3, 48
DEV = torch.device("cuda", 0)


def space():
    return DiscreteActionSpace([torch.tensor([i]) for i in range(NACT)], seed=5)


def make_learner(seed=7, **kw):
    return pearl_b200.B200SoftActorCritic(state_dim=OBS, action_space=space(), actor_hidden_dims=[64, 64], critic_hidden_dims=[64, 64],
                                          training_rounds=ROUNDS, batch_size=B, actor_learning_rate=3e-4, critic_learning_rate=5e-4,
                                          action_representation_module=OneHotActionTensorRepresentationModule(NACT), seed=seed, **kw)


def make_buffer(n, seed):
    g = torch.Generator().manual_seed(seed)
    buf = pearl_b200.B200ReplayBuffer(CAP, rng="python")
    buf.push_batch(torch.randn((n, OBS), generator=g), torch.randint(0, NACT, (n,), generator=g).to(torch.int32), torch.randn(n, generator=g),
                   torch.randn((n, OBS), generator=g), torch.rand(n, generator=g) < 0.1, torch.zeros(n, dtype=torch.bool),
                   max_number_actions=NACT)
    return buf


def flat(module):
    return torch.cat([p.detach().reshape(-1).float().cpu() for p in module.parameters()])


def wrapped_vs_core(autotune):
    """The reference-backed plugin == the CUDA learner it wraps: same initial parameters, same replay contents, same index
    stream (CPython's global `random`, re-seeded) -> identical reports and parameters, twice in a row (the second call
    continues the optimizers from the first, at the actor learning rate the plugin's reset() scheduled)."""
    learner = make_learner(entropy_autotune=autotune, entropy_coef=0.05).to(DEV)
    assert issubclass(type(learner), SoftActorCritic)
    init = {n: flat(getattr(learner, n)) for n in ("_actor", "_critic", "_critic_target")}
    core = ac.DsacCore(state_dim=OBS, n_actions=NACT, actor_hidden_dims=[64, 64], critic_hidden_dims=[64, 64], training_rounds=ROUNDS,
                       batch_size=B, actor_learning_rate=3e-4, critic_learning_rate=5e-4, entropy_autotune=autotune, entropy_coef=0.05,
                       device=DEV)
    pc = init["_critic"].numel() // 2
    core.load_parameters(init["_actor"], init["_critic"][:pc], init["_critic"][pc:], init["_critic_target"][:pc], init["_critic_target"][pc:])
    buf = make_buffer(200, seed=31)
    handle = None
    for call in range(2):
        if call:
            learner.reset(space())                                        # ExponentialLR(0.99) of the actor optimizer
            lr = learner._actor_optimizer.param_groups[0]["lr"]
            assert lr == 3e-4 * 0.99
            core.set_learning_rates(lr, 5e-4)
        random.seed(100 + call); ra = learner.learn(buf)
        random.seed(100 + call); rb = core.learn(buf)
        handle = handle or learner._b200._handle.value
        assert learner._b200._handle.value == handle, "the learning-rate change re-created the C handle"
        assert ra.keys() == rb.keys() and ("entropy_coef" in ra) == autotune, (list(ra), list(rb))
        for k in ra:
            assert ra[k] == rb[k], (f"wrapped vs core, call {call}: {k}", ra[k], rb[k])
        assert len(ra["actor_loss"]) == ROUNDS and all(x == x for v in ra.values() for x in v)
    assert learner._b200._actor_learning_rate == 3e-4 * 0.99
    assert torch.equal(flat(learner._actor), core.actor_params.cpu())
    assert torch.equal(flat(learner._critic), core.critic_params.cpu())
    assert torch.equal(flat(learner._critic_target), core.critic_target_params.cpu())
    assert float(learner._entropy_coef) == core.entropy_coef
    # the torch optimizers show the live AdamW / Adam state (views) and the step counts
    for opt, mod, state in ((learner._actor_optimizer, learner._actor, learner._b200._actor_state),
                            (learner._critic_optimizer, learner._critic, learner._b200._critic_state)):
        st = opt.state[next(mod.parameters())]
        assert st["exp_avg"].data_ptr() == state[0].data_ptr() and st["max_exp_avg_sq"].data_ptr() == state[2].data_ptr()
        assert float(st["exp_avg"].abs().sum()) > 0 and int(st["step"]) == 2 * ROUNDS
    if autotune:
        st = learner._entropy_optimizer.state[learner._log_entropy]
        assert st["exp_avg"].data_ptr() == learner._b200._log_entropy[1:2].data_ptr() and int(st["step"]) == 2 * ROUNDS
        assert float(learner._log_entropy) == float(core._log_entropy[0]) and float(st["exp_avg_sq"]) == float(core._log_entropy[2])
        assert learner._entropy_coef.shape == (1,)
    try:
        learner.learn_batch(None)
        raise AssertionError("learn_batch should not silently fall back to the torch path")
    except NotImplementedError:
        pass


def make_agent(seed=7):
    return PearlAgent(policy_learner=make_learner(seed), replay_buffer=pearl_b200.B200ReplayBuffer(CAP, rng="python"), device_id=0)


def drive(agent, steps, seed):
    g = torch.Generator().manual_seed(seed)
    obs, rew, done = torch.randn((steps + 1, OBS), generator=g), torch.randn(steps, generator=g), torch.rand(steps, generator=g) < 0.08
    agent.reset(obs[0], space())
    reports, handles, resets = [], set(), 1
    for t in range(steps):
        a = torch.as_tensor(agent.act(exploit=False))
        assert 0 <= int(a.reshape(-1)[0]) < NACT
        agent.observe(ActionResult(observation=obs[t + 1], reward=float(rew[t]), terminated=bool(done[t]), truncated=False))
        rep = agent.learn()
        if rep:
            reports.append(rep)
            handles.add(agent.policy_learner._b200._handle.value)
        if bool(done[t]):
            agent.reset(obs[t + 1], space())
            resets += 1
    return reports, handles, resets


def under_pearl_agent():
    random.seed(1); torch.manual_seed(1)
    agent = make_agent()
    pl = agent.policy_learner
    before = flat(pl._actor)
    reports, handles, resets = drive(agent, STEPS, seed=3)
    assert reports and all(set(r) == {"actor_loss", "critic_loss", "entropy_coef"} for r in reports)
    assert all(x == x and abs(x) < 1e6 for r in reports for v in r.values() for x in v), reports[-1]
    assert resets >= 3 and len(handles) == 1, (resets, handles)       # the C handle survived every scheduler step
    lr = pl._actor_optimizer.param_groups[0]["lr"]
    assert lr < 3e-4 and pl._b200._actor_learning_rate == lr
    assert not torch.equal(flat(pl._actor), before), "the actor did not move"
    assert next(pl._actor.parameters()).data_ptr() == pl._b200.actor_params.data_ptr()      # act() reads what the kernels write
    # ---- checkpoint round trip through the agent's own state_dict
    blob = io.BytesIO()
    torch.save(agent.state_dict(), blob)
    blob.seek(0)
    other = make_agent(seed=11)
    other.load_state_dict(torch.load(blob, weights_only=False))
    assert agent.compare(other) == "", agent.compare(other)[:600]
    # both continue identically: same replay contents and index stream; the optimizers continue from the restored step
    buf = make_buffer(150, seed=77)
    other.policy_learner._training_steps = pl._training_steps
    other.policy_learner._ensure_core()
    # the reference does not checkpoint `_entropy_optimizer` (actor_critic_base.py:411-418): carry its Adam state over
    other.policy_learner._b200._log_entropy[1:].copy_(pl._b200._log_entropy[1:])
    random.seed(9); r1 = pl.learn(buf)
    random.seed(9); r2 = other.policy_learner.learn(buf)
    for k in r1:
        assert r1[k] == r2[k], (f"continuation after the checkpoint: {k}", r1[k], r2[k])
    assert agent.compare(other) == "", agent.compare(other)[:600]
    return len(reports), resets


for autotune in (True, False):
    wrapped_vs_core(autotune)
n, resets = under_pearl_agent()
print(f"dsac: subclass of SoftActorCritic; wrapped learner == stand-alone CUDA learner over two calls with a scheduler step "
      f"(reports and parameters identical, AdamW / Adam state seen through the torch optimizers); PearlAgent: {STEPS} env steps, "
      f"{n} learn() reports, {resets} resets on one C handle; checkpoint round trip: compare() == '' and identical continuation")
print("PEARL_AGENT_DSAC_OK")
