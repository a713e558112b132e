"""``MATD3`` — drop-in for agilerl/algorithms/matd3.py on the CUDA path: MADDPG with twin centralised critics and delayed
policy updates, for vector (1-D ``Box``) observations and continuous (``Box``) actions.

Same constructor (matd3.py:107-183: MADDPG's parameters plus ``policy_freq``) and attributes (``critics_1, critics_2,
critic_targets_1, critic_targets_2, critic_1_optimizers, critic_2_optimizers``; ``learn_counter`` is ``{agent_id: int}``).
``learn`` (matd3.py:630-831) is ONE ``b2rl_maddpg_learn`` call with ``twin = 1``: every agent's next action from the target
actors (no target-policy smoothing noise), then per agent Q1, Q2, Q'1, Q'2, y = r + (1 - d) gamma min(Q'1, Q'2),
critic_loss = MSE(Q1, y) + MSE(Q2, y) and both critic Adam steps; only on every ``policy_freq``-th call the actor step
through the updated critic_1 and the soft update of every target (``critic_only = 0``).  Other calls return ``None`` as
the actor loss.  The critic optimisers step on every call and the actor optimisers on policy calls only, so the two
carry separate Adam step counts (and bias corrections).

Acting, noise, ``test``, replay interplay, captured graphs (one per step kind and batch size), checkpoints and cross-rank
moves are MADDPG's (algorithms/maddpg.py).

``agilerl_b200.install()`` does not bind ``agilerl.algorithms.MATD3`` to this class: code written against the reference
(its own test suite among it) also builds MATD3 members with discrete (Gumbel-softmax) actors, which this package does not
implement, so the alias would turn working reference code into errors.  Import it from ``agilerl_b200.algorithms``."""
from __future__ import annotations

import ctypes
from typing import Any

from .. import _lib
from .core.registry import HyperparameterConfig
from .maddpg import MADDPG, _LearnPlan


class MATD3(MADDPG):
    _CRITIC_SETS = (("critics_1", "critic_targets_1", "critic_1_optimizers"),
                    ("critics_2", "critic_targets_2", "critic_2_optimizers"))

    def __init__(self, observation_spaces, action_spaces, agent_ids: list[str] | None = None, O_U_noise: bool = True,
                 expl_noise: float = 0.1, vect_noise_dim: int = 1, mean_noise: float = 0.0, theta: float = 0.15,
                 dt: float = 1e-2, index: int = 0, hp_config: HyperparameterConfig | None = None, policy_freq: int = 2,
                 net_config: dict[str, Any] | None = None, batch_size: int = 64, lr_actor: float = 0.001,
                 lr_critic: float = 0.01, learn_step: int = 5, gamma: float = 0.95, tau: float = 0.01,
                 normalize_images: bool = True, mut: str | None = None, actor_networks=None, critic_networks=None,
                 device: str = "cuda", accelerator: Any | None = None, torch_compiler: str | None = None, wrap: bool = True) -> None:
        assert isinstance(policy_freq, int), "Policy frequency must be an integer."
        assert policy_freq > 0, "Policy frequency must be greater than zero."
        super().__init__(observation_spaces, action_spaces, agent_ids=agent_ids, O_U_noise=O_U_noise, expl_noise=expl_noise,
                         vect_noise_dim=vect_noise_dim, mean_noise=mean_noise, theta=theta, dt=dt, index=index,
                         hp_config=hp_config, net_config=net_config, batch_size=batch_size, lr_actor=lr_actor,
                         lr_critic=lr_critic, learn_step=learn_step, gamma=gamma, tau=tau, mut=mut,
                         normalize_images=normalize_images, actor_networks=actor_networks, critic_networks=critic_networks,
                         device=device, accelerator=accelerator, torch_compiler=torch_compiler, wrap=wrap)
        self.policy_freq = policy_freq
        self.learn_counter = dict.fromkeys(self.agent_ids, 0)          # matd3.py:182

    def _init_kwargs(self) -> dict:
        kw = super()._init_kwargs()
        kw["policy_freq"] = self.policy_freq
        return kw

    # -- step kinds (matd3.py:682, :814-815) ----------------------------------------------------------------------
    def _next_critic_only(self) -> bool:
        counts = {c % self.policy_freq for c in self.learn_counter.values()}
        if len(counts) != 1:
            # the reference decides the actor step per agent and the soft updates by the last agent: one call cannot
            # mix both kinds on the CUDA path
            raise NotImplementedError("MATD3 agents whose learn_counter differ modulo policy_freq are not supported on the CUDA path")
        return (self.learn_counter[self.agent_ids[-1]] + 1) % self.policy_freq != 0

    def _advance(self) -> bool:
        critic_only = self._next_critic_only()
        for a in self.agent_ids:
            self.learn_counter[a] += 1
        for _, _, opt in self._CRITIC_SETS:
            for o in getattr(self, opt).values():
                o.step += 1
        if not critic_only:
            for o in self.actor_optimizers.values():
                o.step += 1
        return critic_only

    def _launch(self, plan: _LearnPlan, graph, critic_only: bool, stream: int) -> None:
        """Two pairs of bias corrections: the critics' (every call) and, on a policy call, the actors'."""
        c_step = next(iter(self.critic_1_optimizers.values())).step
        plan.state_host.bias_correction1, plan.state_host.bias_correction2 = 1.0 - 0.9 ** c_step, 1.0 - 0.999 ** c_step
        hosts, devs = [ctypes.addressof(plan.state_host)], [plan.state_dev.data_ptr()]
        if not critic_only:
            a_step = next(iter(self.actor_optimizers.values())).step
            plan.actor_state_host.bias_correction1 = 1.0 - 0.9 ** a_step
            plan.actor_state_host.bias_correction2 = 1.0 - 0.999 ** a_step
            hosts.append(ctypes.addressof(plan.actor_state_host))
            devs.append(plan.actor_state_dev.data_ptr())
        n = len(hosts)
        hv = (ctypes.c_void_p * n)(*hosts)
        dv = (ctypes.c_void_p * n)(*devs)
        _lib.check(self._lib.b2rl_graph_launch_states(graph, hv, dv, n, stream))
