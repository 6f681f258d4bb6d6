"""B200SoftActorCritic — the learner side of Pearl's discrete SoftActorCritic
(pearl/policy_learners/sequential_decision_making/soft_actor_critic.py:48-286 on top of actor_critic_base.py:309-366) on a
B200: `learn(replay_buffer)` runs `training_rounds` x (sample -> actor step -> critic step -> soft target update ->
entropy-coefficient step) on the GPU through `prl_dsac_learn` (include/pearl_b200.h).  Same constructor argument names and
the same reporting keys as the reference (`actor_loss`, `critic_loss`, `entropy_coef`).  A discrete SAC step takes
expectations over the softmax policy and draws no random numbers, so the sampled indices pin every float.  PyTorch holds
the flat parameter vectors; no math happens in Python.  No CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Iterable, Optional

import torch

from . import _lib
from .replay_buffer import B200ReplayBuffer, _stream_ptr


class B200SoftActorCritic:
    def __init__(self, action_space: Any = None, state_dim: Optional[int] = None, actor_hidden_dims: Optional[Iterable[int]] = None,
                 critic_hidden_dims: Optional[Iterable[int]] = None, actor_learning_rate: float = 1e-4,
                 critic_learning_rate: float = 1e-4, critic_soft_update_tau: float = 0.005, discount_factor: float = 0.99,
                 training_rounds: int = 100, batch_size: int = 128, entropy_coef: float = 0.2, entropy_autotune: bool = True,
                 target_entropy_scale: float = 0.89, *, n_actions: Optional[int] = None,
                 device: Optional[torch.device | str | int] = None, max_rounds_per_call: int = 1024, seed: Optional[int] = None) -> None:
        self._device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if self._device.index is None:
            self._device = torch.device("cuda", torch.cuda.current_device())
        self._lib = _lib.init(self._device.index)
        actor_hidden_dims, critic_hidden_dims = list(actor_hidden_dims or []), list(critic_hidden_dims or [])
        if len(actor_hidden_dims) != 2 or len(critic_hidden_dims) != 2:
            raise NotImplementedError("the CUDA discrete SAC learner is built for two hidden layers in the actor and in each critic")
        if state_dim is None:
            raise ValueError("state_dim is required")
        if n_actions is None:
            if action_space is None or not hasattr(action_space, "n"):
                raise ValueError("discrete SAC needs a discrete action space (`action_space.n`) or n_actions")
            n_actions = action_space.n
        self._state_dim, self._n_actions = int(state_dim), int(n_actions)
        self._actor_hidden_dims, self._critic_hidden_dims = actor_hidden_dims, critic_hidden_dims
        self._actor_learning_rate, self._critic_learning_rate = float(actor_learning_rate), float(critic_learning_rate)
        self._entropy_learning_rate = float(critic_learning_rate)          # soft_actor_critic.py:126-133
        self._critic_soft_update_tau, self._discount_factor = float(critic_soft_update_tau), float(discount_factor)
        self._training_rounds, self._batch_size = int(training_rounds), int(batch_size)
        self._entropy_autotune = bool(entropy_autotune)
        # -scale * log(1 / n) in fp32, as the reference evaluates it (soft_actor_critic.py:139-142)
        self._target_entropy = float(-target_entropy_scale * torch.log(1.0 / torch.tensor(self._n_actions)))
        self._max_rounds = max(int(max_rounds_per_call), 1)
        self._training_steps = 0
        self.use_cuda_graph = True       # False: plain stream launches (profilers)
        self._handle = C.c_void_p(0)
        self._bound_batch = 0
        self._gen = torch.Generator(device=self._device)
        if seed is not None:
            self._gen.manual_seed(int(seed))
        cfg = self._cfg(1)
        pa, pc = int(self._lib.prl_dsac_actor_param_count(C.byref(cfg))), int(self._lib.prl_dsac_critic_param_count(C.byref(cfg)))
        dev, f32 = self._device, torch.float32
        self.actor_params = torch.empty(pa, dtype=f32, device=dev)
        self.critic_params = torch.empty(2 * pc, dtype=f32, device=dev)
        self._init_like_reference()
        self.critic_target_params = self.critic_params.clone()
        self._actor_state = [torch.zeros(pa, dtype=f32, device=dev) for _ in range(3)]      # exp_avg, exp_avg_sq, max_exp_avg_sq
        self._critic_state = [torch.zeros(2 * pc, dtype=f32, device=dev) for _ in range(3)]
        self._log_entropy = torch.zeros(4, dtype=f32, device=dev)                              # value, Adam exp_avg, exp_avg_sq, unused
        self._entropy_coef = torch.full((1,), 1.0 if entropy_autotune else float(entropy_coef), dtype=f32, device=dev)
        self._adam_step = 0

    # ------------------------------------------------------------------ parameters
    def _cfg(self, max_batch: int) -> _lib.DsacCfg:
        return _lib.DsacCfg(self._state_dim, self._n_actions, self._actor_hidden_dims[0], self._actor_hidden_dims[1],
                            self._critic_hidden_dims[0], self._critic_hidden_dims[1], int(self._entropy_autotune), max_batch,
                            self._max_rounds, self._actor_learning_rate, self._critic_learning_rate, self._entropy_learning_rate,
                            0.9, 0.999, 1e-8, 0.01, self._discount_factor, self._critic_soft_update_tau, self._target_entropy, 1e-4)

    def _actor_shapes(self):
        O, A, (h1, h2) = self._state_dim, self._n_actions, self._actor_hidden_dims
        return [(h1, O), (h1,), (h2, h1), (h2,), (A, h2), (A,)]

    def _critic_shapes(self):
        D, (c1, c2) = self._state_dim + self._n_actions, self._critic_hidden_dims
        return [(c1, D), (c1,), (c2, c1), (c2,), (1, c2), (1,)]

    def _init_like_reference(self) -> None:
        """Xavier-uniform weights, biases 0.01 (neural_networks/common/utils.py:201-205, applied to the actor at
        actor_critic_base.py:154 and to both critics at twin_critic.py:36-60)."""
        def fill(vec, shapes):
            off = 0
            for shp in shapes:
                if len(shp) == 2:
                    n = shp[0] * shp[1]
                    bound = (6.0 / (shp[0] + shp[1])) ** 0.5
                    vec[off:off + n].uniform_(-bound, bound, generator=self._gen)
                else:
                    n = shp[0]
                    vec[off:off + n].fill_(0.01)
                off += n
            assert off == vec.numel()
        fill(self.actor_params, self._actor_shapes())
        pc = self.critic_params.numel() // 2
        fill(self.critic_params[:pc], self._critic_shapes())
        fill(self.critic_params[pc:], self._critic_shapes())

    def load_parameters(self, actor, q1, q2, q1_target=None, q2_target=None) -> None:
        """Flat fp32 vectors in `torch.nn.Module.parameters()` order of the reference networks (actor: VanillaActorNetwork;
        critics: VanillaQValueNetwork over state || one-hot action)."""
        t = lambda x: torch.as_tensor(x, dtype=torch.float32).reshape(-1).to(self._device)  # noqa: E731
        pc = self.critic_params.numel() // 2
        self.actor_params.copy_(t(actor))
        self.critic_params[:pc].copy_(t(q1))
        self.critic_params[pc:].copy_(t(q2))
        self.critic_target_params[:pc].copy_(t(q1 if q1_target is None else q1_target))
        self.critic_target_params[pc:].copy_(t(q2 if q2_target is None else q2_target))

    def set_learning_rates(self, actor_learning_rate: float, critic_learning_rate: float) -> None:
        """New AdamW learning rates from the next learn() on (the reference's ExponentialLR steps the actor's at every
        reset()); the C handle and its captured round are kept."""
        self._actor_learning_rate, self._critic_learning_rate = float(actor_learning_rate), float(critic_learning_rate)
        if self._handle.value:
            _lib.check(self._lib.prl_dsac_set_lr(self._handle, self._actor_learning_rate, self._critic_learning_rate))

    @property
    def entropy_coef(self) -> float:
        return float(self._entropy_coef.item())

    @property
    def target_entropy(self) -> float:
        return self._target_entropy

    @property
    def batch_size(self) -> int:
        return self._batch_size

    @property
    def training_rounds(self) -> int:
        return self._training_rounds

    def adam_step(self) -> int:
        """Optimizer steps taken so far (the actor, critic and entropy optimizers step once per round)."""
        return int(self._lib.prl_dsac_adam_step(self._handle)) if self._handle.value else int(self._adam_step)

    def _release(self) -> None:
        """Drop the C handle (keeping the step count); the next learn() re-creates it from the Python-side settings."""
        if self._handle.value:
            self._adam_step = int(self._lib.prl_dsac_adam_step(self._handle))
            self._lib.prl_dsac_destroy(self._handle)
            self._handle = C.c_void_p(0)

    def __del__(self):
        try:
            if getattr(self, "_handle", None) and self._handle.value:
                self._lib.prl_dsac_destroy(self._handle)
                self._handle = C.c_void_p(0)
        except Exception:
            pass

    def _bind(self, need_batch: int) -> None:
        if self._handle.value and need_batch <= self._bound_batch:
            return
        self._release()
        cfg = self._cfg(max(need_batch, self._batch_size if self._batch_size > 0 else need_batch))
        nbytes = int(self._lib.prl_dsac_workspace_bytes(C.byref(cfg)))
        self._workspace = torch.empty(nbytes, dtype=torch.uint8, device=self._device)
        h = C.c_void_p(0)
        p = _lib.ptr
        with torch.cuda.device(self._device):
            _lib.check(self._lib.prl_dsac_create(
                C.byref(h), C.byref(cfg), p(self.actor_params), p(self._actor_state[0]), p(self._actor_state[1]),
                p(self._actor_state[2]), p(self.critic_params), p(self._critic_state[0]), p(self._critic_state[1]),
                p(self._critic_state[2]), p(self.critic_target_params), p(self._log_entropy), p(self._entropy_coef),
                self._adam_step, p(self._workspace)))
        self._handle, self._bound_batch = h, cfg.max_batch

    # ------------------------------------------------------------------ PolicyLearner.learn (policy_learner.py:162-204)
    def learn(self, replay_buffer: B200ReplayBuffer, trace: Optional[dict] = None) -> dict:
        if not isinstance(replay_buffer, B200ReplayBuffer):
            raise TypeError("B200SoftActorCritic learns from a B200ReplayBuffer (GPU-resident ring)")
        if len(replay_buffer) == 0:
            return {}
        if replay_buffer.is_action_continuous:
            raise ValueError("discrete SAC needs a replay buffer with is_action_continuous=False")
        B = len(replay_buffer) if (self._batch_size == -1 or len(replay_buffer) < self._batch_size) else self._batch_size
        self._bind(B)
        R, dev = self._training_rounds, self._device
        report = {"actor_loss": [], "critic_loss": []}
        if self._entropy_autotune:
            report["entropy_coef"] = []
        idx_all = []
        done = 0
        while done < R:
            r = min(self._max_rounds, R - done)
            out = torch.empty((3, r), dtype=torch.float32, device=dev)
            idx = torch.empty((r, B), dtype=torch.int32, device=dev) if trace is not None else None
            replay_buffer._rng_push()
            with torch.cuda.device(dev):
                _lib.check(self._lib.prl_dsac_set_graph(self._handle, int(self.use_cuda_graph)))
                _lib.check(self._lib.prl_dsac_learn(self._handle, replay_buffer.handle, r, B, _lib.ptr(out[0]), _lib.ptr(out[1]),
                                                    _lib.ptr(out[2]), _lib.ptr(idx) if idx is not None else None, _stream_ptr(dev)))
            replay_buffer._rng_pull()
            host = out.cpu()
            report["actor_loss"] += host[0].tolist()
            report["critic_loss"] += host[1].tolist()
            if self._entropy_autotune:
                report["entropy_coef"] += host[2].tolist()
            if idx is not None:
                idx_all.append(idx.cpu())
            done += r
        self._training_steps += R
        if trace is not None:
            trace["idx"] = torch.cat(idx_all)
        return report
