"""ORACLE (test infrastructure, never imported by the product path).

CPU restatement of ``MATD3.learn / learn_individual / soft_update`` (agilerl/algorithms/matd3.py:630-846) in plain
functional torch-fp32, driven from reference ``state_dict``s, with the networks and forward functions of
``oracle.maddpg`` (MATD3 builds the same actors and centralised critics as MADDPG, two critic sets instead of one).
Pinned bit-exactly against the unmodified reference executed through ``oracle/refshim`` by
``tests/golden/make_golden_matd3.py`` (fixture ``matd3_vector.npz``).

Quirks kept literally: next actions of every agent come from the target actors BEFORE any update of this call, with
no target-policy smoothing noise; min(Q'1, Q'2); NaN rewards -> 0, NaN dones -> 1 (then ``uint8``); critic_loss =
MSE(Q1, y) + MSE(Q2, y), one backward, both critic Adam steps on every call; ``learn_counter[agent] += 1`` and, when it
is a multiple of ``policy_freq``, the actor step through the UPDATED critic_1; the soft updates of every target after
all agents, on the condition evaluated with the LAST agent's counter; ``None`` as the actor loss of other calls.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .maddpg import MlpSpec, _leaf, actor_forward, critic_forward


class OracleMATD3:
    def __init__(self, agent_ids, a_specs: dict, c_head: MlpSpec, actor_sds: dict, actor_target_sds: dict, critic_1_sds: dict,
                 critic_target_1_sds: dict, critic_2_sds: dict, critic_target_2_sds: dict, *, gamma=0.95, tau=0.01, lr_actor=1e-3,
                 lr_critic=1e-2, policy_freq: int = 2):
        self.agent_ids, self.a_specs, self.c_head = list(agent_ids), a_specs, c_head
        cp = lambda sds: {a: {k: v.clone() for k, v in sds[a].items()} for a in agent_ids}
        self.actors = {a: _leaf(actor_sds[a]) for a in agent_ids}
        self.critics_1 = {a: _leaf(critic_1_sds[a]) for a in agent_ids}
        self.critics_2 = {a: _leaf(critic_2_sds[a]) for a in agent_ids}
        self.actor_targets, self.critic_targets_1, self.critic_targets_2 = cp(actor_target_sds), cp(critic_target_1_sds), cp(critic_target_2_sds)
        self.gamma, self.tau, self.policy_freq = gamma, tau, policy_freq
        self.learn_counter = dict.fromkeys(agent_ids, 0)
        self.opt_actor = {a: torch.optim.Adam(list(self.actors[a].values()), lr=lr_actor) for a in agent_ids}
        self.opt_critic_1 = {a: torch.optim.Adam(list(self.critics_1[a].values()), lr=lr_critic) for a in agent_ids}
        self.opt_critic_2 = {a: torch.optim.Adam(list(self.critics_2[a].values()), lr=lr_critic) for a in agent_ids}
        self.last_grads: dict = {}

    def _soft(self, net, target):
        with torch.no_grad():
            for k in net:
                target[k].copy_(self.tau * net[k].data + (1.0 - self.tau) * target[k])

    def learn(self, experiences):
        """matd3.py:630-694.  ``experiences`` = (states, actions, rewards, next_states, dones), dicts by agent id.
        ``last_grads`` holds this call's gradients (critic_1 / critic_2 always, actor on policy calls)."""
        states, actions, rewards, next_states, dones = experiences
        rewards, dones = dict(rewards), dict(dones)
        ids = self.agent_ids
        with torch.no_grad():
            next_actions = [actor_forward(self.actor_targets[a], self.a_specs[a], next_states[a]) for a in ids]
        stacked_actions = torch.cat([actions[a] for a in ids], dim=1)
        stacked_next_actions = torch.cat(next_actions, dim=1)
        obs_list, next_obs_list = [states[a] for a in ids], [next_states[a] for a in ids]
        self.last_grads = {}
        out = {}
        for a in ids:                                                     # learn_individual :696-831
            q1 = critic_forward(self.critics_1[a], self.c_head, obs_list, stacked_actions)
            q2 = critic_forward(self.critics_2[a], self.c_head, obs_list, stacked_actions)
            with torch.no_grad():
                qn1 = critic_forward(self.critic_targets_1[a], self.c_head, next_obs_list, stacked_next_actions)
                qn2 = critic_forward(self.critic_targets_2[a], self.c_head, next_obs_list, stacked_next_actions)
            q_next = torch.min(qn1, qn2)
            r = torch.where(torch.isnan(rewards[a]), torch.full_like(rewards[a], 0), rewards[a]).to(torch.float32)
            d = torch.where(torch.isnan(dones[a]), torch.full_like(dones[a], 1), dones[a]).to(torch.uint8)
            rewards[a], dones[a] = r, d
            y = r + (1 - d) * self.gamma * q_next
            critic_loss = F.mse_loss(q1, y) + F.mse_loss(q2, y)
            self.opt_critic_1[a].zero_grad()
            self.opt_critic_2[a].zero_grad()
            critic_loss.backward()
            self.last_grads.update({f"critic_1/{a}/{k}": v.grad.detach().clone() for k, v in self.critics_1[a].items()})
            self.last_grads.update({f"critic_2/{a}/{k}": v.grad.detach().clone() for k, v in self.critics_2[a].items()})
            self.opt_critic_1[a].step()
            self.opt_critic_2[a].step()
            actor_loss = None
            action = actor_forward(self.actors[a], self.a_specs[a], states[a])
            detached = dict(actions)
            detached[a] = action
            self.learn_counter[a] += 1
            if self.learn_counter[a] % self.policy_freq == 0:
                stacked_detached = torch.cat([detached[b] for b in ids], dim=1)
                actor_loss = -critic_forward(self.critics_1[a], self.c_head, obs_list, stacked_detached).mean()
                self.opt_actor[a].zero_grad()
                actor_loss.backward()
                self.last_grads.update({f"actor/{a}/{k}": v.grad.detach().clone() for k, v in self.actors[a].items()})
                self.opt_actor[a].step()
            out[a] = (actor_loss.item() if actor_loss is not None else None, critic_loss.item())
        if self.learn_counter[ids[-1]] % self.policy_freq == 0:           # :682, the loop variable left at the last agent
            for a in ids:
                self._soft(self.actors[a], self.actor_targets[a])
                self._soft(self.critics_1[a], self.critic_targets_1[a])
                self._soft(self.critics_2[a], self.critic_targets_2[a])
        return out
