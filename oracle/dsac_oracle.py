"""oracle/dsac_oracle.py — CPU restatement of discrete Soft Actor-Critic's `learn_batch`
(TEST INFRASTRUCTURE ONLY; eager PyTorch fp32 like the reference).

Restated reference sites (paths relative to /root/reference/pearl):
  policy_learners/sequential_decision_making/actor_critic_base.py:309-366   actor step, then critic step, soft target update
  policy_learners/sequential_decision_making/soft_actor_critic.py:137-149   target entropy, entropy Adam(eps=1e-4), reset()
  policy_learners/sequential_decision_making/soft_actor_critic.py:151-178   entropy-coefficient step after the two steps
  policy_learners/sequential_decision_making/soft_actor_critic.py:180-286   critic target (expectation over the policy), actor loss
  neural_networks/sequential_decision_making/actor_networks.py:107-153     VanillaActorNetwork (softmax head)
  neural_networks/sequential_decision_making/twin_critic.py:75-91, q_value_networks.py:152-174  twin VanillaQValueNetwork
  utils/functional_utils/learning/critic_utils.py:103-122,170-203          twin loss, target update
A discrete SAC step draws no random numbers: the batch indices pin every float.  Every action is available (the fixed
action space of a BasicReplayBuffer), so the reference's unavailable-action masks are all False and are not restated.
Parity pinned by tests/golden/dsac_small.npz and dsac_fixed.npz (oracle/gen_dsac_golden.py).
"""
from __future__ import annotations

import torch

from .pearl_oracle import _mlp, flat, load_flat  # noqa: F401


class OracleDiscreteSAC:
    def __init__(self, obs, n_actions, actor_hidden, critic_hidden, *, actor_lr=1e-4, critic_lr=1e-4, gamma=0.99, tau=0.005,
                 entropy_coef=0.2, autotune=True, target_entropy_scale=0.89, init=None):
        self.obs, self.A, self.gamma, self.tau, self.autotune = obs, n_actions, gamma, tau, autotune
        self.actor = _mlp([obs] + list(actor_hidden) + [n_actions])
        self.q = [_mlp([obs + n_actions] + list(critic_hidden) + [1]) for _ in range(2)]
        self.qt = [_mlp([obs + n_actions] + list(critic_hidden) + [1]) for _ in range(2)]
        if init is not None:
            load_flat(self.actor, init["actor"])
            for i in range(2):
                load_flat(self.q[i], init[f"q{i + 1}"])
                load_flat(self.qt[i], init[f"q{i + 1}t"])
        self.opt_actor = torch.optim.AdamW(self.actor.parameters(), lr=actor_lr, amsgrad=True)
        self.opt_critic = torch.optim.AdamW(list(self.q[0].parameters()) + list(self.q[1].parameters()), lr=critic_lr, amsgrad=True)
        self.log_alpha = torch.nn.Parameter(torch.zeros(1))
        self.opt_alpha = torch.optim.Adam([self.log_alpha], lr=critic_lr, eps=1e-4)
        self.alpha = torch.exp(self.log_alpha).detach() if autotune else torch.tensor(entropy_coef)
        self.target_entropy = -target_entropy_scale * torch.log(1.0 / torch.tensor(n_actions))

    def set_actor_lr(self, lr: float) -> None:
        self.opt_actor.param_groups[0]["lr"] = lr

    def set_critic_lr(self, lr: float) -> None:
        self.opt_critic.param_groups[0]["lr"] = lr

    def scheduler_step(self) -> None:
        """SoftActorCritic.reset: ExponentialLR(actor optimizer, gamma=0.99).step()."""
        self.set_actor_lr(self.opt_actor.param_groups[0]["lr"] * 0.99)

    def policy(self, s):
        return torch.softmax(self.actor(s), dim=-1)

    def q_all(self, nets, s):
        """Q(s, a) for every action a: the state paired with each one-hot row (get_q_values with [B, A, A] actions)."""
        B = s.shape[0]
        x = torch.cat([s.unsqueeze(1).expand(B, self.A, self.obs), torch.eye(self.A).expand(B, self.A, self.A)], dim=-1)
        return [net(x).squeeze(-1) for net in nets]

    def learn_batch(self, b):
        s, a, r, s2, term = b["state"], b["action"], b["reward"], b["next_state"], b["terminated"]
        onehot = torch.nn.functional.one_hot(a.long().reshape(-1), self.A).float()
        # ---- actor step (the critics' values only)
        with torch.no_grad():
            q1, q2 = self.q_all(self.q, s)
            q = torch.minimum(q1, q2)
        p = self.policy(s)
        logp = torch.log(p + 1e-8)
        actor_loss = (p * (self.alpha * logp - q)).mean()
        self.opt_actor.zero_grad()
        actor_loss.backward()
        self.opt_actor.step()
        # ---- critic step with the UPDATED actor
        self.opt_critic.zero_grad()
        with torch.no_grad():
            qt1, qt2 = self.q_all(self.qt, s2)
            p2 = self.policy(s2)
            v = ((torch.minimum(qt1, qt2) - self.alpha * torch.log(p2 + 1e-8)) * p2).sum(dim=1)
            y = (v * self.gamma * (1 - term.float())) + r
        x = torch.cat([s, onehot], dim=-1)
        mse = torch.nn.MSELoss()
        critic_loss = (mse(self.q[0](x).view(-1), y) + mse(self.q[1](x).view(-1), y)) / 2.0
        critic_loss.backward()
        self.opt_critic.step()
        with torch.no_grad():
            for i in range(2):
                for pt, pp in zip(self.qt[i].parameters(), self.q[i].parameters()):
                    pt.copy_(self.tau * pp + (1.0 - self.tau) * pt)
        out = {"actor_loss": actor_loss.item(), "critic_loss": critic_loss.item()}
        # ---- entropy coefficient (pre-update policy of the actor step)
        if self.autotune:
            entropy = -(p.detach() * logp.detach()).sum(1).mean()
            ent_loss = torch.exp(self.log_alpha) * (entropy - self.target_entropy).detach()
            self.opt_alpha.zero_grad()
            ent_loss.backward()
            self.opt_alpha.step()
            self.alpha = torch.exp(self.log_alpha).detach()
            out["entropy_coef"] = float(ent_loss.detach())
        return out
