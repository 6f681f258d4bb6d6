"""Actor-critic plugins that SUBCLASS the reference classes (SURVEY.md §8 rows a1 / a14-a16, f3):

    B200ContinuousSoftActorCritic   (ContinuousSoftActorCritic, soft_actor_critic_continuous.py:42-231)
    B200SoftActorCritic             (SoftActorCritic, soft_actor_critic.py:48-286; discrete actions)
    B200ProximalPolicyOptimization  (ProximalPolicyOptimization, ppo.py:96-293)
    B200TD3 / B200DeepDeterministicPolicyGradient  (td3.py:43-202, ddpg.py:41-157)

When facebookresearch/Pearl is importable these are the reference classes with `learn()` replaced: the reference
constructor runs unchanged (same arguments, same networks, same optimizers, same exploration module), so
`pearl.pearl_agent.PearlAgent` accepts them as they are, `act()` / `reset()` / `compare()` / `state_dict()` are the
reference's own code.  On the first `learn()` (after PearlAgent moved the learner to its CUDA device) the parameters of
`_actor`, `_critic` (and their targets) are re-pointed at views into the flat fp32 vectors of the CUDA learner
(`pearl_b200.sac / dsac / ppo / td3`), and `optimizer.state` at views into its flat AdamW vectors: the kernels and torch see the
same memory, nothing is copied per call, `get_extra_state` / `set_extra_state` (actor_critic_base.py:411-428) checkpoint
the live state, and a state loaded with `load_state_dict` is picked up on the next `learn()`.

When Pearl is not installed (the GPU test box) the same public names are the stand-alone CUDA learners, which take the
same keyword arguments.  Nothing here computes anything; there is no CPU path."""
from __future__ import annotations

import ctypes as C
from typing import Any

import torch

from .dsac import B200SoftActorCritic as DsacCore
from .ppo import B200ProximalPolicyOptimization as PpoCore
from .sac import B200ContinuousSoftActorCritic as SacCore
from .td3 import B200DeepDeterministicPolicyGradient as DdpgCore
from .td3 import B200TD3 as Td3Core

try:  # pragma: no cover - depends on the environment
    from pearl.policy_learners.sequential_decision_making.ddpg import DeepDeterministicPolicyGradient as _RefDDPG
    from pearl.policy_learners.sequential_decision_making.ppo import ProximalPolicyOptimization as _RefPPO
    from pearl.policy_learners.sequential_decision_making.soft_actor_critic import SoftActorCritic as _RefDSAC
    from pearl.policy_learners.sequential_decision_making.soft_actor_critic_continuous import (
        ContinuousSoftActorCritic as _RefSAC,
    )
    from pearl.policy_learners.sequential_decision_making.td3 import TD3 as _RefTD3

    HAVE_REFERENCE = True
except Exception:  # ModuleNotFoundError (pearl or gymnasium missing)
    HAVE_REFERENCE = False


def _adamw_lr(opt: torch.optim.Optimizer, what: str) -> float:
    """The CUDA learners implement torch.optim.AdamW(amsgrad=True) with torch's default betas / eps / weight decay
    (what the reference constructs, actor_critic_base.py:157-166, 200-209)."""
    g = opt.param_groups[0] if isinstance(opt, torch.optim.AdamW) and len(opt.param_groups) == 1 else None
    if (g is None or not g.get("amsgrad", False) or g.get("maximize", False) or tuple(g["betas"]) != (0.9, 0.999)
            or float(g["eps"]) != 1e-8 or float(g["weight_decay"]) != 0.01):
        raise NotImplementedError(f"{what}: the fused update implements torch.optim.AdamW(amsgrad=True) with default "
                                  "betas / eps / weight_decay in one parameter group")
    return float(g["lr"])


def _shapes(module: torch.nn.Module) -> list:
    return [tuple(p.shape) for p in module.parameters()]


def _adopt(module: torch.nn.Module, flat: torch.Tensor) -> None:
    """Copy the module's parameters into `flat` (torch's parameters() order) and re-point them at views of it."""
    off = 0
    for p in module.parameters():
        n = p.numel()
        if off + n > flat.numel():
            break
        flat[off:off + n].copy_(p.detach().reshape(-1).to(device=flat.device, dtype=torch.float32))
        p.data = flat[off:off + n].view(p.shape)
        off += n
    if off != flat.numel() or off != sum(p.numel() for p in module.parameters()):
        raise NotImplementedError(f"{type(module).__name__}: parameter layout is not the one the CUDA learner is built for")


def _is_adopted(module: torch.nn.Module, flat: torch.Tensor) -> bool:
    return next(module.parameters()).data_ptr() == flat.data_ptr()


def _bind_optimizer(opt: torch.optim.Optimizer, module: torch.nn.Module, state3: list, step: int) -> int:
    """Make `opt.state` views into the flat AdamW vectors.  State that is already there and is NOT ours (built by torch,
    or just loaded from a checkpoint) is imported first; returns the AdamW step count to continue from."""
    params = list(module.parameters())
    st = opt.state
    if all(p in st and "exp_avg" in st[p] for p in params) and st[params[0]]["exp_avg"].data_ptr() != state3[0].data_ptr():
        dev = state3[0].device
        cat = lambda key: torch.cat([st[p][key].detach().reshape(-1).to(dev, torch.float32) for p in params])  # noqa: E731
        state3[0].copy_(cat("exp_avg"))
        state3[1].copy_(cat("exp_avg_sq"))
        state3[2].copy_(cat("max_exp_avg_sq") if all("max_exp_avg_sq" in st[p] for p in params) else cat("exp_avg_sq"))
        step = int(float(st[params[0]]["step"]))
    off = 0
    for p in params:
        n = p.numel()
        st[p] = dict(step=torch.tensor(float(step), dtype=torch.float32), exp_avg=state3[0][off:off + n].view(p.shape),
                     exp_avg_sq=state3[1][off:off + n].view(p.shape), max_exp_avg_sq=state3[2][off:off + n].view(p.shape))
        off += n
    return step


def _is_bound(opt: torch.optim.Optimizer, module: torch.nn.Module, state3: list) -> bool:
    p0 = next(module.parameters())
    return p0 in opt.state and "exp_avg" in opt.state[p0] and opt.state[p0]["exp_avg"].data_ptr() == state3[0].data_ptr()


def _set_steps(opt: torch.optim.Optimizer, step: int) -> None:
    for s in opt.state.values():
        if "step" in s:
            s["step"].fill_(float(step))


class _B200ActorCriticMixin:
    """In front of a reference ActorCriticBase subclass.  Subclasses say how to build the CUDA learner from the
    reference object (`_make_core`) and which (module, flat vector) / (optimizer, module, AdamW vectors) pairs exist."""

    def __init__(self, *args: Any, max_rounds_per_call: int = 1024, seed: int | None = None, **kwargs: Any) -> None:
        super().__init__(*args, **kwargs)
        self._b200_opts = dict(max_rounds_per_call=max_rounds_per_call, seed=seed)
        self._b200 = None

    # ---- per algorithm
    def _make_core(self, device: torch.device):
        raise NotImplementedError

    def _module_pairs(self, core) -> list:      # [(module, flat vector)]
        raise NotImplementedError

    def _optimizer_triples(self, core) -> list:  # [(optimizer, module, [exp_avg, exp_avg_sq, max_exp_avg_sq])]
        return [(self._actor_optimizer, self._actor, core._actor_state), (self._critic_optimizer, self._critic, core._critic_state)]

    def _core_steps(self, core) -> tuple:        # AdamW step counts (actor, critic) the CUDA learner is at
        raise NotImplementedError

    def _restart_core(self, core, steps: tuple) -> None:   # drop the C handle; the next learn() re-creates it at `steps`
        raise NotImplementedError

    def _bind_extras(self, core) -> None:   # idempotent: runs on every learn()
        pass

    # ---- binding
    def _device_of_parameters(self) -> torch.device:
        dev = next(self._actor.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError(f"{type(self).__name__}: parameters are on {dev}; move the learner to a CUDA device "
                               "(PearlAgent(device_id=0) does this) - pearl_b200 has no CPU path")
        return dev

    def _ensure_core(self):
        dev = self._device_of_parameters()
        core = self._b200
        if core is None or core._device != dev:
            core = self._make_core(dev)
            self._b200 = core
        pairs = self._module_pairs(core)
        if not all(_is_adopted(m, flat) for m, flat in pairs):
            for m, flat in pairs:
                _adopt(m, flat)
        self._bind_extras(core)
        # learning rates changed since the CUDA learner was configured (a scheduler, or the user editing param_groups): the C
        # handle is re-created with the new rates at the current AdamW step counts (moments and parameters live in our vectors)
        lrs = (_adamw_lr(self._actor_optimizer, "actor optimizer"), _adamw_lr(self._critic_optimizer, "critic optimizer"))
        if lrs != (core._actor_learning_rate, core._critic_learning_rate):
            steps = self._core_steps(core)
            core._actor_learning_rate, core._critic_learning_rate = lrs
            self._restart_core(core, steps)
        triples = self._optimizer_triples(core)
        if not all(_is_bound(o, m, s3) for o, m, s3 in triples):
            cur = self._core_steps(core)
            steps = tuple(_bind_optimizer(o, m, s3, c) for (o, m, s3), c in zip(triples, cur))
            if steps != cur:
                self._restart_core(core, steps)
        return core

    # ---- PolicyLearner.learn (policy_learner.py:162-204)
    def learn(self, replay_buffer) -> dict:
        if len(replay_buffer) == 0:
            return {}
        core = self._ensure_core()
        core._training_rounds, core._batch_size = int(self._training_rounds), int(self._batch_size)
        core._training_steps = int(self._training_steps)
        report = core.learn(replay_buffer)
        self._training_steps = int(core._training_steps)
        for (opt, _, _), step in zip(self._optimizer_triples(core), self._core_steps(core)):
            _set_steps(opt, step)
        self._after_learn(core)
        return report

    def _after_learn(self, core) -> None:
        pass

    def learn_batch(self, batch) -> dict:
        raise NotImplementedError(f"{type(self).__name__} trains from a B200ReplayBuffer through learn(); a step on a "
                                  "caller-supplied batch is not part of the CUDA learner")


def _mlp3(shapes: list, what: str) -> tuple:
    """(in, h1, h2, out) of a two-hidden-layer MLP from its parameter shapes [W1, b1, W2, b2, W3, b3, ...]."""
    if len(shapes) < 6 or any(len(s) != (2 if i % 2 == 0 else 1) for i, s in enumerate(shapes)):
        raise NotImplementedError(f"{what}: the CUDA learners are built for MLPs with two hidden layers")
    (h1, din), (h2, h1b), (out, h2b) = shapes[0], shapes[2], shapes[4]
    if h1b != h1 or h2b != h2:
        raise NotImplementedError(f"{what}: unexpected layer shapes {shapes}")
    return din, h1, h2, out


if HAVE_REFERENCE:

    class B200ContinuousSoftActorCritic(_B200ActorCriticMixin, _RefSAC):
        """Drop-in for `pearl...soft_actor_critic_continuous.ContinuousSoftActorCritic`."""

        def _make_core(self, device):
            sa, sc = _shapes(self._actor), _shapes(self._critic)
            if len(sa) != 8 or len(sc) != 12:
                raise NotImplementedError("the CUDA SAC learner is built for GaussianActorNetwork + TwinCritic(VanillaQValueNetwork) "
                                          "with two hidden layers each")
            obs, h1, h2, act = _mlp3(sa, "actor")
            dq, c1, c2, one = _mlp3(sc[:6], "critic")
            if sa[6] != (act, h2) or dq != obs + act or one != 1 or sc[6:] != sc[:6]:
                raise NotImplementedError("unexpected SAC network shapes")
            space = getattr(self._actor, "_action_space", None) or self._action_space   # the box the actor scales its output to
            return SacCore(state_dim=obs, actor_hidden_dims=[h1, h2], critic_hidden_dims=[c1, c2],
                           actor_learning_rate=_adamw_lr(self._actor_optimizer, "actor optimizer"),
                           critic_learning_rate=_adamw_lr(self._critic_optimizer, "critic optimizer"),
                           critic_soft_update_tau=float(self._critic_soft_update_tau), discount_factor=float(self._discount_factor),
                           training_rounds=int(self._training_rounds), batch_size=int(self._batch_size),
                           entropy_coef=float(self._entropy_coef), entropy_autotune=bool(self._entropy_autotune),
                           low=space.low, high=space.high, device=device, **self._b200_opts)

        def _module_pairs(self, core):
            return [(self._actor, core.actor_params), (self._critic, core.critic_params), (self._critic_target, core.critic_target_params)]

        def _core_steps(self, core):
            s = int(core._lib.prl_sac_adam_step(core._handle)) if core._handle.value else int(core._adam_step)
            return (s, s)

        def _restart_core(self, core, steps):
            if steps[0] != steps[1]:
                raise NotImplementedError("SAC steps its actor and critics once per round: one AdamW step count")
            if core._handle.value:
                core._lib.prl_sac_destroy(core._handle)
                core._handle = C.c_void_p(0)
            core._adam_step = int(steps[0])

        def _bind_extras(self, core):
            """Entropy coefficient: `_log_entropy` (Parameter) and its AdamW state are the 4 floats of the CUDA learner's
            log-entropy block, `_entropy_coef` (buffer, shape kept) a view of its coefficient.  A state loaded into the
            entropy optimizer since the last call is imported."""
            coef = core._entropy_coef
            if self._entropy_coef.data_ptr() != coef.data_ptr():
                coef.copy_(self._entropy_coef.detach().reshape(1).to(coef))
                self._entropy_coef = coef.view(self._entropy_coef.shape)
            if not self._entropy_autotune:
                return
            blk, p, st = core._log_entropy, self._log_entropy, self._entropy_optimizer.state
            if p.data_ptr() != blk.data_ptr():
                _adamw_lr(self._entropy_optimizer, "entropy optimizer")
                blk[0:1].copy_(p.detach().reshape(1).to(blk))
                p.data = blk[0:1]
            if p in st and "exp_avg" in st[p] and st[p]["exp_avg"].data_ptr() == blk[1:2].data_ptr():
                return
            if p in st and "exp_avg" in st[p]:
                blk[1:2].copy_(st[p]["exp_avg"].reshape(1))
                blk[2:3].copy_(st[p]["exp_avg_sq"].reshape(1))
                blk[3:4].copy_(st[p].get("max_exp_avg_sq", st[p]["exp_avg_sq"]).reshape(1))
            st[p] = dict(step=torch.tensor(float(self._core_steps(core)[0])), exp_avg=blk[1:2], exp_avg_sq=blk[2:3],
                         max_exp_avg_sq=blk[3:4])

        def _after_learn(self, core):
            if self._entropy_autotune:
                _set_steps(self._entropy_optimizer, self._core_steps(core)[0])

    def _entropy_adam_lr(opt: torch.optim.Optimizer) -> float:
        """The CUDA learner's entropy step is torch.optim.Adam(eps=1e-4) with default betas, no weight decay, no amsgrad
        (what SoftActorCritic constructs, soft_actor_critic.py:126-133)."""
        g = opt.param_groups[0] if type(opt) is torch.optim.Adam and len(opt.param_groups) == 1 else None
        if (g is None or g.get("amsgrad", False) or g.get("maximize", False) or tuple(g["betas"]) != (0.9, 0.999)
                or float(g["eps"]) != 1e-4 or float(g["weight_decay"]) != 0.0):
            raise NotImplementedError("entropy optimizer: the CUDA learner implements torch.optim.Adam(eps=1e-4, betas=(0.9, 0.999), "
                                      "weight_decay=0, amsgrad=False) in one parameter group")
        return float(g["lr"])

    class B200SoftActorCritic(_B200ActorCriticMixin, _RefDSAC):
        """Drop-in for `pearl...soft_actor_critic.SoftActorCritic` (discrete actions, fixed action space).  `reset()` steps the
        reference's ExponentialLR of the actor every episode; the new rate reaches the CUDA learner through prl_dsac_set_lr
        without re-creating its handle or re-capturing its round."""

        def _make_core(self, device):
            from pearl.action_representation_modules.one_hot_action_representation_module import (
                OneHotActionTensorRepresentationModule,
            )
            from pearl.neural_networks.sequential_decision_making.actor_networks import VanillaActorNetwork
            from pearl.neural_networks.sequential_decision_making.q_value_networks import VanillaQValueNetwork
            from pearl.neural_networks.sequential_decision_making.twin_critic import TwinCritic
            critic = self._critic
            if (type(self._actor) is not VanillaActorNetwork or not isinstance(critic, TwinCritic)
                    or not all(type(c) is VanillaQValueNetwork for c in (critic._critic_1, critic._critic_2))):
                raise NotImplementedError("the CUDA discrete SAC learner is built for VanillaActorNetwork + TwinCritic(VanillaQValueNetwork)")
            sa, sc = _shapes(self._actor), _shapes(critic)
            if len(sa) != 6 or len(sc) != 12:
                raise NotImplementedError("the CUDA discrete SAC learner is built for two hidden layers in the actor and in each critic")
            obs, h1, h2, n_act = _mlp3(sa, "actor")
            dq, c1, c2, one = _mlp3(sc[:6], "critic")
            arm = self.action_representation_module
            if (not isinstance(arm, OneHotActionTensorRepresentationModule) or int(arm.max_number_actions) != n_act
                    or dq != obs + n_act or one != 1 or sc[6:] != sc[:6]):
                raise NotImplementedError("the CUDA discrete SAC learner needs a one-hot action representation of the actor's "
                                          "n_actions and critics over state || one-hot action")
            hsm = getattr(self, "_history_summarization_module", None)
            if hsm is not None and any(True for _ in hsm.parameters()):
                raise NotImplementedError("the CUDA discrete SAC learner takes states as they are: a history summarization "
                                          "module with parameters (e.g. LSTM) is not supported")
            core = DsacCore(state_dim=obs, n_actions=n_act, actor_hidden_dims=[h1, h2], critic_hidden_dims=[c1, c2],
                            actor_learning_rate=_adamw_lr(self._actor_optimizer, "actor optimizer"),
                            critic_learning_rate=_adamw_lr(self._critic_optimizer, "critic optimizer"),
                            critic_soft_update_tau=float(self._critic_soft_update_tau), discount_factor=float(self._discount_factor),
                            training_rounds=int(self._training_rounds), batch_size=int(self._batch_size),
                            entropy_coef=float(self._entropy_coef), entropy_autotune=bool(self._entropy_autotune),
                            device=device, **self._b200_opts)
            if self._entropy_autotune:
                core._target_entropy = float(self._target_entropy)
                core._entropy_learning_rate = _entropy_adam_lr(self._entropy_optimizer)
            return core

        def _module_pairs(self, core):
            return [(self._actor, core.actor_params), (self._critic, core.critic_params), (self._critic_target, core.critic_target_params)]

        def _core_steps(self, core):
            s = core.adam_step()
            return (s, s)

        def _restart_core(self, core, steps):
            if steps[0] != steps[1]:
                raise NotImplementedError("discrete SAC steps its actor and critics once per round: one AdamW step count")
            if core._handle.value and tuple(steps) == self._core_steps(core):
                # only the learning rates changed (ExponentialLR at every reset()): keep the handle and its captured round
                core.set_learning_rates(core._actor_learning_rate, core._critic_learning_rate)
                return
            core._release()
            core._adam_step = int(steps[0])

        def _bind_extras(self, core):
            """Entropy coefficient: `_log_entropy` (Parameter) and its Adam state are views of the CUDA learner's log-entropy
            block, `_entropy_coef` (buffer, shape kept) a view of its coefficient.  A state loaded into the entropy optimizer
            since the last call is imported."""
            coef = core._entropy_coef
            if self._entropy_coef.data_ptr() != coef.data_ptr():
                coef.copy_(self._entropy_coef.detach().reshape(1).to(coef))
                self._entropy_coef = coef.view(self._entropy_coef.shape)
            if not self._entropy_autotune:
                return
            lr = _entropy_adam_lr(self._entropy_optimizer)
            if lr != core._entropy_learning_rate:        # part of the handle's configuration
                core._entropy_learning_rate = lr
                core._release()
            blk, p, st = core._log_entropy, self._log_entropy, self._entropy_optimizer.state
            if p.data_ptr() != blk.data_ptr():
                blk[0:1].copy_(p.detach().reshape(1).to(blk))
                p.data = blk[0:1]
            if p in st and "exp_avg" in st[p] and st[p]["exp_avg"].data_ptr() == blk[1:2].data_ptr():
                return
            if p in st and "exp_avg" in st[p]:
                blk[1:2].copy_(st[p]["exp_avg"].reshape(1))
                blk[2:3].copy_(st[p]["exp_avg_sq"].reshape(1))
            st[p] = dict(step=torch.tensor(float(self._core_steps(core)[0])), exp_avg=blk[1:2], exp_avg_sq=blk[2:3])

        def _after_learn(self, core):
            if self._entropy_autotune:
                _set_steps(self._entropy_optimizer, self._core_steps(core)[0])

    class B200ProximalPolicyOptimization(_B200ActorCriticMixin, _RefPPO):
        """Drop-in for `pearl...ppo.ProximalPolicyOptimization` (discrete actions, as the reference's `_actor_loss`)."""

        def _make_core(self, device):
            sa, sc = _shapes(self._actor), _shapes(self._critic)
            if len(sa) != 6 or len(sc) != 6:
                raise NotImplementedError("the CUDA PPO learner is built for VanillaActorNetwork + VanillaValueNetwork with two hidden layers")
            obs, h1, h2, n_act = _mlp3(sa, "actor")
            oc, c1, c2, one = _mlp3(sc, "critic")
            if oc != obs or one != 1:
                raise NotImplementedError("unexpected PPO network shapes")
            return PpoCore(state_dim=obs, n_actions=n_act, actor_hidden_dims=[h1, h2], critic_hidden_dims=[c1, c2],
                           actor_learning_rate=_adamw_lr(self._actor_optimizer, "actor optimizer"),
                           critic_learning_rate=_adamw_lr(self._critic_optimizer, "critic optimizer"),
                           discount_factor=float(self._discount_factor), training_rounds=int(self._training_rounds),
                           batch_size=int(self._batch_size), epsilon=float(self._epsilon),
                           trace_decay_param=float(self._trace_decay_param), entropy_bonus_scaling=float(self._entropy_bonus_scaling),
                           device=device, **self._b200_opts)

        def _module_pairs(self, core):
            return [(self._actor, core.actor_params), (self._critic, core.critic_params)]

        def _core_steps(self, core):
            s = int(core._lib.prl_ppo_adam_step(core._handle)) if core._handle.value else int(core._adam_step)
            return (s, s)

        def _restart_core(self, core, steps):
            if steps[0] != steps[1]:
                raise NotImplementedError("PPO steps actor and critic once per round: one AdamW step count")
            if core._handle.value:
                core._lib.prl_ppo_destroy(core._handle)
                core._handle = C.c_void_p(0)
            core._adam_step = int(steps[0])

        def preprocess_replay_buffer(self, replay_buffer, process_group=None):
            """ppo.py:201-293 on the GPU; `learn()` calls it itself (as the reference's `learn` does)."""
            core = self._ensure_core()
            core._batch_size = int(self._batch_size)
            return core.preprocess_replay_buffer(replay_buffer, process_group=process_group)

    class _DeterministicMixin(_B200ActorCriticMixin):
        _core_cls = Td3Core

        def _core_kwargs(self) -> dict:
            return {}

        def _make_core(self, device):
            sa, sc = _shapes(self._actor), _shapes(self._critic)
            if len(sa) != 6 or len(sc) != 12:
                raise NotImplementedError("the CUDA TD3 / DDPG learner is built for VanillaContinuousActorNetwork + "
                                          "TwinCritic(VanillaQValueNetwork) with two hidden layers each")
            obs, h1, h2, act = _mlp3(sa, "actor")
            dq, c1, c2, one = _mlp3(sc[:6], "critic")
            if dq != obs + act or one != 1 or sc[6:] != sc[:6]:
                raise NotImplementedError("unexpected TD3 / DDPG network shapes")
            space = getattr(self._actor, "_action_space", None) or self._action_space   # the box the actor scales its output to
            return self._core_cls(state_dim=obs, actor_hidden_dims=[h1, h2], critic_hidden_dims=[c1, c2],
                                  actor_learning_rate=_adamw_lr(self._actor_optimizer, "actor optimizer"),
                                  critic_learning_rate=_adamw_lr(self._critic_optimizer, "critic optimizer"),
                                  actor_soft_update_tau=float(self._actor_soft_update_tau),
                                  critic_soft_update_tau=float(self._critic_soft_update_tau), discount_factor=float(self._discount_factor),
                                  training_rounds=int(self._training_rounds), batch_size=int(self._batch_size),
                                  low=space.low, high=space.high, device=device, **self._core_kwargs(), **self._b200_opts)

        def _module_pairs(self, core):
            return [(self._actor, core.actor_params), (self._actor_target, core.actor_target_params),
                    (self._critic, core.critic_params), (self._critic_target, core.critic_target_params)]

        def _core_steps(self, core):
            if core._handle.value:
                return (int(core._lib.prl_td3_actor_adam_step(core._handle)), int(core._lib.prl_td3_critic_adam_step(core._handle)))
            return tuple(int(x) for x in core._adam_steps)

        def _restart_core(self, core, steps):
            if core._handle.value:
                core._lib.prl_td3_destroy(core._handle)
                core._handle = C.c_void_p(0)
            core._adam_steps = (int(steps[0]), int(steps[1]))

    class B200TD3(_DeterministicMixin, _RefTD3):
        """Drop-in for `pearl...td3.TD3`."""

        def _core_kwargs(self):
            return dict(actor_update_freq=int(self._actor_update_freq), actor_update_noise=float(self._actor_update_noise),
                        actor_update_noise_clip=float(self._actor_update_noise_clip))

    class B200DeepDeterministicPolicyGradient(_DeterministicMixin, _RefDDPG):
        """Drop-in for `pearl...ddpg.DeepDeterministicPolicyGradient`."""
        _core_cls = DdpgCore

else:
    B200ContinuousSoftActorCritic = SacCore
    B200SoftActorCritic = DsacCore
    B200ProximalPolicyOptimization = PpoCore
    B200TD3 = Td3Core
    B200DeepDeterministicPolicyGradient = DdpgCore
