"""``MADDPG`` — drop-in for agilerl/algorithms/maddpg.py:39-800 on the CUDA path (SURVEY 8f-4, BASELINE configs[4]:
4 agents x 18-dim observations, shared replay), for vector (1-D ``Box``) observations and continuous (``Box``) actions.

Same constructor (maddpg.py:103-131) and attributes (``agent_ids, n_agents, possible_observation_spaces,
possible_action_spaces, action_dims, actors, actor_targets, critics, critic_targets, actor_optimizers,
critic_optimizers, batch_size, lr_actor, lr_critic, learn_step, gamma, tau, mut, O_U_noise, expl_noise, mean_noise,
current_noise ...``); ``learn(experiences) -> {agent_id: (actor_loss, critic_loss)}`` (:571-628), ``get_action(obs,
infos) -> (processed, raw)`` (:428-532), ``action_noise`` / ``reset_action_noise``, ``soft_update``, ``clone``.
The body of ``learn`` — every agent's target action, centralised critic TD step, actor step through the updated critic
and all soft updates — is ONE C call, ``b2rl_maddpg_learn`` (csrc/maddpg.cuh).

The batch may be the reference's tuple of ``{agent_id: tensor}`` dicts or what ``MultiAgentReplayBuffer.sample``
returns here (dicts carrying the already concatenated ``[B, sum]`` matrices: no ``torch.cat`` on the way in).

Not implemented (raises): image / Dict sub-observations, discrete (Gumbel-softmax) actors, custom networks,
``accelerator``, architecture mutations of the sub-networks.  ``env_defined_actions`` in the info dicts are honoured like the
reference's (maddpg.py:518-529)."""
from __future__ import annotations

import copy
import ctypes
import os
from collections import OrderedDict
from typing import Any

import numpy as np
import torch

from .. import _lib
from ..compat import spaces
from ..networks.actors import DeterministicActor, MultiInputContinuousQNetwork
from .core.base import EvolvableAlgorithm
from .core.registry import HyperparameterConfig, NetworkGroup, OptimizerConfig
from .td3 import _AdamState


_GRAPH = os.environ.get("B2RL_MADDPG_GRAPH", "1") != "0"      # CUDA-graph replay of learn() (0: always eager)
_FAN = os.environ.get("B2RL_MADDPG_STREAMS", "1") != "0"      # the agents' steps on one side stream each (0: serial)


class _LearnPlan:
    """Static batch buffers + the captured graph of one ``b2rl_maddpg_learn`` call for a batch size: ~130 dependent
    launches (four concurrent per-agent chains) replayed as ONE graph launch.  What changes between steps — Adam's bias
    corrections — lives in a ``b2rl_step_state`` on the device, rewritten by the graph's first node from the host's
    double arithmetic, so a replay is bit-identical to the eager call (tests/test_maddpg_gpu.py).

    ``graphs`` holds one graph per step kind (``critic_only``): MADDPG only ever has the full step (``graph``); MATD3 also
    captures its critic-only call, and its full step writes a second state block for the actors (``actor_state_*``), whose
    optimisers have stepped fewer times than the critics'."""

    def __init__(self, agent, B: int):
        dev, n = agent._dev, agent.n_agents
        SO, SA = sum(agent.obs_dims.values()), sum(agent.action_dims.values())
        mk = lambda w: torch.zeros((B, w), dtype=torch.float32, device=dev)
        self.obs, self.action, self.reward, self.next_obs, self.done = mk(SO), mk(SA), mk(n), mk(SO), mk(n)
        self.out = torch.zeros((n, 2), dtype=torch.float32, device=dev)
        self.state_host = _lib.StepState()
        self.state_ref = ctypes.byref(self.state_host)
        self.state_dev = torch.zeros(ctypes.sizeof(_lib.StepState), dtype=torch.uint8, device=dev)
        self.actor_state_host = _lib.StepState()
        self.actor_state_dev = torch.zeros(ctypes.sizeof(_lib.StepState), dtype=torch.uint8, device=dev)
        self.graphs: dict = {}
        self._fields = [self.obs, self.action, self.reward, self.next_obs, self.done]

    def fields(self):
        """The static buffers in the replay's field order (obs, action, reward, next_obs, done)."""
        return self._fields

    @property
    def graph(self):
        """The captured full step (actor and critic updates, soft updates)."""
        return self.graphs.get(False)

    def destroy(self) -> None:
        for g in self.graphs.values():
            _lib.load().b2rl_graph_destroy(g)
        self.graphs = {}


class _AgentOptimizers(OrderedDict):
    """{agent_id: Adam state}; ``.optimizer`` is the mapping itself — the reference's ``OptimizerWrapper`` over a
    ``ModuleDict`` exposes its per-agent optimisers under that name (optimizer_wrapper.py)."""

    @property
    def optimizer(self):
        return self


def concatenate_spaces(space_list) -> spaces.Box:
    """utils/algo_utils.py concatenate_spaces for 1-D Boxes."""
    low = np.concatenate([np.asarray(s.low, np.float32).reshape(-1) for s in space_list])
    high = np.concatenate([np.asarray(s.high, np.float32).reshape(-1) for s in space_list])
    return spaces.Box(low, high, (int(low.shape[0]),), np.float32)


class MADDPG(EvolvableAlgorithm):
    # (networks, targets, optimisers) of each centralised critic set; MATD3 has two
    _CRITIC_SETS = (("critics", "critic_targets", "critic_optimizers"),)

    def __init__(self, observation_spaces, action_spaces, agent_ids: list[str] | None = None, O_U_noise: bool = True,
                 expl_noise: float = 0.1, vect_noise_dim: int = 1, mean_noise: float = 0.0, theta: float = 0.15,
                 dt: float = 1e-2, index: int = 0, hp_config: HyperparameterConfig | None = None,
                 net_config: dict[str, Any] | None = None, batch_size: int = 64, lr_actor: float = 0.001,
                 lr_critic: float = 0.01, learn_step: int = 5, gamma: float = 0.95, tau: float = 0.01, mut: str | None = None,
                 normalize_images: bool = True, actor_networks=None, critic_networks=None, device: str = "cuda",
                 accelerator: Any | None = None, torch_compiler: str | None = None, wrap: bool = True) -> None:
        super().__init__(index, hp_config, device, accelerator, torch_compiler, name=type(self).__name__)
        if isinstance(observation_spaces, (spaces.Dict, dict)):
            agent_ids = list(observation_spaces.keys()) if agent_ids is None else agent_ids
            observation_spaces = [observation_spaces[a] for a in agent_ids]
        if isinstance(action_spaces, (spaces.Dict, dict)):
            action_spaces = [action_spaces[a] for a in agent_ids]
        assert agent_ids is not None, "Agent IDs must be specified if observation spaces are passed as a list."
        assert len(agent_ids) == len(observation_spaces) == len(action_spaces), \
            "Number of agent IDs must match number of observation and action spaces."
        assert learn_step >= 1, "Learn step must be greater than or equal to one."
        assert isinstance(learn_step, int), "Learn step rate must be an integer."
        assert isinstance(batch_size, int), "Batch size must be an integer."
        assert batch_size >= 1, "Batch size must be greater than or equal to one."
        assert isinstance(lr_actor, float), "Actor learning rate must be a float."
        assert lr_actor > 0, "Actor learning rate must be greater than zero."
        assert isinstance(lr_critic, float), "Critic learning rate must be a float."
        assert lr_critic > 0, "Critic learning rate must be greater than zero."
        assert isinstance(gamma, float), "Gamma must be a float."
        assert isinstance(tau, float), "Tau must be a float."
        assert tau > 0, "Tau must be greater than zero."
        assert isinstance(wrap, bool), "Wrap models flag must be boolean value True or False."
        if actor_networks is not None or critic_networks is not None:
            raise NotImplementedError("custom actor / critic networks are not implemented for MADDPG on the CUDA path")
        if len(agent_ids) > _lib.B2RL_MAX_AGENTS:
            raise NotImplementedError(f"at most {_lib.B2RL_MAX_AGENTS} agents per MADDPG instance on the CUDA path")
        for a, osp, asp in zip(agent_ids, observation_spaces, action_spaces):
            if not (isinstance(osp, spaces.Box) and len(osp.shape) == 1):
                raise NotImplementedError(f"{a}: only 1-D Box observations are implemented for MADDPG on the CUDA path")
            if not (isinstance(asp, spaces.Box) and len(asp.shape) == 1):
                raise NotImplementedError(f"{a}: only continuous (1-D Box) actions are implemented for MADDPG on the CUDA path")
        self.agent_ids, self.n_agents = list(agent_ids), len(agent_ids)
        self.observation_spaces, self.action_spaces = list(observation_spaces), list(action_spaces)
        self.possible_observation_spaces = OrderedDict(zip(self.agent_ids, observation_spaces))
        self.possible_action_spaces = OrderedDict(zip(self.agent_ids, action_spaces))
        self.observation_space = spaces.Dict(self.possible_observation_spaces)
        self.action_space = spaces.Dict(self.possible_action_spaces)
        self.action_dims = {a: int(s.shape[0]) for a, s in self.possible_action_spaces.items()}
        self.obs_dims = {a: int(s.shape[0]) for a, s in self.possible_observation_spaces.items()}
        self.normalize_images = normalize_images
        self.batch_size, self.lr_actor, self.lr_critic, self.learn_step = batch_size, lr_actor, lr_critic, learn_step
        self.gamma, self.tau, self.mut, self.net_config = gamma, tau, mut, net_config
        self.learn_counter = 0
        self.O_U_noise, self.vect_noise_dim, self.theta, self.dt, self.sqdt = O_U_noise, vect_noise_dim, theta, dt, dt ** 0.5
        mk = lambda v: v if isinstance(v, dict) else {a: v * torch.ones(vect_noise_dim, d) for a, d in self.action_dims.items()}
        self.sample_gaussian = {a: torch.zeros(vect_noise_dim, d) for a, d in self.action_dims.items()}
        self.expl_noise, self.mean_noise = mk(expl_noise), mk(mean_noise)
        self.current_noise = {a: torch.zeros(vect_noise_dim, d) for a, d in self.action_dims.items()}

        # networks (maddpg.py:272-350): per-agent actors; every critic sees all observations and all actions
        net_config = {} if net_config is None else copy.deepcopy(net_config)
        if any(k in net_config for k in self.agent_ids):
            raise NotImplementedError("per-agent net_config dictionaries are not implemented on the CUDA path")
        actor_cfg = dict(net_config)
        head_config = actor_cfg.get("head_config")
        if head_config is None:
            head_config = dict(hidden_size=[64])
        head_config = {k: v for k, v in head_config.items() if k != "output_activation"}
        actor_cfg["head_config"] = head_config
        latent_dim = int(actor_cfg.get("latent_dim", 32))
        critic_head = copy.deepcopy(head_config)
        all_act = concatenate_spaces(self.action_spaces)
        mk_a = lambda a: DeterministicActor(self.possible_observation_spaces[a], self.possible_action_spaces[a],
                                            device=self.device, **copy.deepcopy(actor_cfg))
        mk_c = lambda: MultiInputContinuousQNetwork(self.observation_space, all_act, latent_dim=latent_dim,
                                                    head_config=critic_head, device=self.device)
        self.actors = OrderedDict((a, mk_a(a)) for a in self.agent_ids)
        for net, _, _ in self._CRITIC_SETS:
            setattr(self, net, OrderedDict((a, mk_c()) for a in self.agent_ids))
        self.actor_targets = OrderedDict((a, mk_a(a)) for a in self.agent_ids)
        for _, tgt, _ in self._CRITIC_SETS:
            setattr(self, tgt, OrderedDict((a, mk_c()) for a in self.agent_ids))
        for a in self.agent_ids:
            self.actors[a].encoder.disable_mutations()                                   # maddpg.py:324-326
            self.actor_targets[a].load_state_dict(self.actors[a].state_dict())
            for net, tgt, _ in self._CRITIC_SETS:
                getattr(self, tgt)[a].load_state_dict(getattr(self, net)[a].state_dict())
        self.register_network_group(NetworkGroup(eval_network="actors", shared_networks="actor_targets", policy=True))
        for net, tgt, _ in self._CRITIC_SETS:
            self.register_network_group(NetworkGroup(eval_network=net, shared_networks=tgt))
        self.registry.register_optimizer(OptimizerConfig(name="actor_optimizers", networks=["actors"], lr="lr_actor"))
        for net, _, opt in self._CRITIC_SETS:
            self.registry.register_optimizer(OptimizerConfig(name=opt, networks=[net], lr="lr_critic"))
        self._bind_engine()

    # -- engine state ------------------------------------------------------------------------------------
    def _bind_engine(self, keep: dict | None = None) -> None:
        self.actor_optimizers = _AgentOptimizers((a, _AdamState(self.actors[a], self.lr_actor)) for a in self.agent_ids)
        for net, _, opt in self._CRITIC_SETS:
            setattr(self, opt, _AgentOptimizers((a, _AdamState(getattr(self, net)[a], self.lr_critic)) for a in self.agent_ids))
        if keep:
            for name in self._opt_names():
                for a in self.agent_ids:
                    getattr(self, name)[a].load_state_dict(keep[name][a])
        n = self.n_agents
        critics = getattr(self, self._CRITIC_SETS[0][0])        # every critic set shares one architecture (one layer table)
        self._actor_descs = (ctypes.POINTER(_lib.NetDesc) * n)(*[ctypes.pointer(self.actors[a].layout.desc) for a in self.agent_ids])
        self._critic_descs = (ctypes.POINTER(_lib.NetDesc) * n)(*[ctypes.pointer(critics[a].layout.desc) for a in self.agent_ids])
        self._ws: dict = {}
        self._all_opts = [o for name in self._opt_names() for o in getattr(self, name).values()]
        self._lib = _lib.load()
        self._drop_plans()
        if "use_graph" not in self.__dict__:
            self.use_graph, self.concurrent_agents = _GRAPH, _FAN

    def _drop_plans(self) -> None:
        for plan in self.__dict__.get("_plans", {}).values():
            plan.destroy()
        self._plans: dict = {}

    def __del__(self):
        try:
            self._drop_plans()
        except Exception:  # noqa: BLE001 - interpreter shutdown
            pass

    def _opt_names(self) -> list:
        return ["actor_optimizers"] + [opt for _, _, opt in self._CRITIC_SETS]

    def _net_names(self) -> list:
        """Every network set, each evaluation network followed by its target."""
        return ["actors", "actor_targets"] + [x for net, tgt, _ in self._CRITIC_SETS for x in (net, tgt)]

    def _opt_state(self) -> dict:
        return {name: {a: o.state_dict() for a, o in getattr(self, name).items()} for name in self._opt_names()}

    def reinit_optimizers(self, optimizer=None) -> None:
        self._bind_engine()

    def __setattr__(self, name, value):
        object.__setattr__(self, name, value)
        if name == "lr_actor":
            for o in self.__dict__.get("actor_optimizers", {}).values():
                o.lr = value
        if name == "lr_critic":
            for _, _, opt in self._CRITIC_SETS:
                for o in self.__dict__.get(opt, {}).values():
                    o.lr = value
        if name in ("lr_actor", "lr_critic", "gamma", "tau", "policy_freq", "concurrent_agents") and self.__dict__.get("_plans"):
            self._drop_plans()                     # these scalars are baked into a captured call

    def clone(self, index: int | None = None, wrap: bool = True):
        """core/base.py:855-917: same constructor arguments, then networks, optimiser state and the run-time attributes."""
        kw = self._init_kwargs()
        kw["index"] = self.index if index is None else index
        kw["device"] = self.device
        c = type(self)(**kw)
        for a in self.agent_ids:
            for name in self._net_names():
                getattr(c, name)[a].buffers.copy_from(getattr(self, name)[a].buffers)
        c._bind_engine(keep=self._opt_state())
        c.use_graph, c.concurrent_agents = self.use_graph, self.concurrent_agents
        c.expl_noise = {a: v.clone() for a, v in self.expl_noise.items()}
        c.mean_noise = {a: v.clone() for a, v in self.mean_noise.items()}
        c.current_noise = {a: v.clone() for a, v in self.current_noise.items()}
        c.scores, c.fitness, c.steps = list(self.scores), list(self.fitness), list(self.steps)
        c.learn_counter = copy.deepcopy(self.learn_counter)
        return c

    # -- cross-rank move (population sharding: hpo/tournament.py::_select_sharded broadcasts a winner from its owner) ------
    def _init_kwargs(self) -> dict:
        return dict(observation_spaces=self.observation_spaces, action_spaces=self.action_spaces, agent_ids=list(self.agent_ids),
                    O_U_noise=self.O_U_noise, vect_noise_dim=self.vect_noise_dim, theta=self.theta, dt=self.dt,
                    hp_config=copy.deepcopy(self.registry.hp_config), net_config=copy.deepcopy(self.net_config),
                    batch_size=self.batch_size, lr_actor=self.lr_actor, lr_critic=self.lr_critic, learn_step=self.learn_step,
                    gamma=self.gamma, tau=self.tau, mut=self.mut, normalize_images=self.normalize_images)

    def _state_tensors(self) -> list:
        out = []
        for a in self.agent_ids:
            out += [getattr(self, name)[a].buffers.params for name in self._net_names()]
            for name in self._opt_names():
                o = getattr(self, name)[a]
                out += [o.exp_avg, o.exp_avg_sq]
        return out

    def _restore_steps(self, attrs: dict) -> None:
        """Adam step counts from ``export_state``'s attributes: per optimiser set where recorded, else the one count."""
        steps = attrs.get("opt_steps", {})
        for name in self._opt_names():
            for o in getattr(self, name).values():
                o.step = steps.get(name, attrs["opt_step"])

    def export_state(self):
        """-> (picklable description, [device tensors]): every network's flat parameter buffer and both Adam moments of
        every optimiser, 8 tensors per agent for MADDPG (≈ 0.5 MB for config 5), 12 for MATD3."""
        meta = {"init": self._init_kwargs(),
                "attrs": {"scores": list(self.scores), "fitness": list(self.fitness), "steps": list(self.steps), "index": self.index,
                          "learn_counter": copy.deepcopy(self.learn_counter), "opt_step": self._all_opts[-1].step,
                          "opt_steps": {name: next(iter(getattr(self, name).values())).step for name in self._opt_names()},
                          "expl_noise": self.expl_noise, "mean_noise": self.mean_noise, "current_noise": self.current_noise}}
        return meta, self._state_tensors()

    @classmethod
    def from_state(cls, meta, tensors, like):
        agent = cls(device=like.device, **meta["init"])
        for dst, src in zip(agent._state_tensors(), tensors):
            dst.copy_(src)
        a = meta["attrs"]
        agent.scores, agent.fitness, agent.steps, agent.index = a["scores"], a["fitness"], a["steps"], a["index"]
        agent.learn_counter = copy.deepcopy(a["learn_counter"])
        agent._restore_steps(a)
        agent.expl_noise, agent.mean_noise, agent.current_noise = a["expl_noise"], a["mean_noise"], a["current_noise"]
        return agent

    # -- checkpoints (core/base.py:919-1049 reduced to what this learner owns) ---------------------------------------
    def save_checkpoint(self, path: str) -> None:
        meta, tensors = self.export_state()
        torch.save({"algo": self.algo, "meta": meta, "tensors": [t.detach().cpu() for t in tensors]}, path)

    def load_checkpoint(self, path: str) -> None:
        """Restore networks, targets, Adam moments / step counts, hyper-parameters and run-time attributes into THIS
        member (same agents and network shapes; a mismatch raises)."""
        ckpt = torch.load(path, map_location="cpu", weights_only=False)
        meta, tensors = ckpt["meta"], ckpt["tensors"]
        init = meta["init"]
        if list(init["agent_ids"]) != self.agent_ids:
            raise ValueError(f"checkpoint holds agents {init['agent_ids']}, this member {self.agent_ids}")
        mine = self._state_tensors()
        if len(mine) != len(tensors) or any(tuple(a.shape) != tuple(b.shape) for a, b in zip(mine, tensors)):
            raise ValueError("checkpoint networks do not fit this member's architecture")
        for k in ("batch_size", "lr_actor", "lr_critic", "learn_step", "gamma", "tau", "mut", "policy_freq"):
            if k in init:
                setattr(self, k, init[k])
        if init.get("hp_config") is not None:
            self.hp_config = self.registry.hp_config = init["hp_config"]
        for dst, src in zip(mine, tensors):
            dst.copy_(src)
        a = meta["attrs"]
        self.scores, self.fitness, self.steps, self.index = a["scores"], a["fitness"], a["steps"], a["index"]
        self.learn_counter = copy.deepcopy(a["learn_counter"])
        self._restore_steps(a)
        self.expl_noise, self.mean_noise, self.current_noise = a["expl_noise"], a["mean_noise"], a["current_noise"]

    @classmethod
    def load(cls, path: str, device: str = "cuda", accelerator=None):
        """core/base.py ``EvolvableAlgorithm.load``: build the member from the checkpoint alone."""
        ckpt = torch.load(path, map_location="cpu", weights_only=False)

        class _Like:
            pass
        like = _Like()
        like.device = device
        return cls.from_state(ckpt["meta"], ckpt["tensors"], like)

    # -- acting (maddpg.py:428-558) ------------------------------------------------------------------------
    def preprocess_observation(self, observation: dict) -> dict:
        out = {}
        for a in self.agent_ids:
            o = observation[a]
            if not isinstance(o, torch.Tensor):
                o = torch.as_tensor(np.asarray(o))
            o = o.to(self._dev, dtype=torch.float32)
            out[a] = o.unsqueeze(0) if o.ndim == 1 else o
        return out

    @staticmethod
    def _key_in_nested_dict(nested: dict, target: str) -> bool:
        """utils/algo_utils.py:490-507, literally: only the FIRST nested dict met is searched."""
        for k, v in nested.items():
            if k == target:
                return True
            if isinstance(v, dict):
                return MADDPG._key_in_nested_dict(v, target)
        return False

    def extract_agent_masks(self, infos: dict | None = None):
        """core/base.py:1544-1603 for continuous actions: ``env_defined_actions`` per agent (NaN where the agent acts itself)
        and the boolean masks of the entries the environment dictates."""
        if (infos is None or not self._key_in_nested_dict(infos, "env_defined_actions")
                or all(not info for agent, info in infos.items() if agent in self.agent_ids)):
            return None, None
        env_defined = {agent: (info.get("env_defined_actions", None) if isinstance(info, dict) else None)
                       for agent, info in infos.items() if agent in self.agent_ids}
        masks = {}
        for agent_id, val in list(env_defined.items()):
            if val is None:                                   # environment not vectorised: this agent acts itself
                val = np.full(self.action_dims[agent_id], np.nan)
                env_defined[agent_id] = val
            if isinstance(val, (int, float)):
                val = np.array([val])
                env_defined[agent_id] = val
            masks[agent_id] = np.where(np.isnan(env_defined[agent_id]), 0, 1).astype(bool)
        return env_defined, masks

    @staticmethod
    def _reconcile_shapes(reference: np.ndarray, other: np.ndarray):
        """utils/algo_utils.py:1790-1819, continuous branch."""
        if reference.shape == other.shape:
            return reference, other
        if np.prod(other.shape) == np.prod(reference.shape):
            if other.ndim < reference.ndim:
                other = np.expand_dims(other, 0)
            else:
                reference = np.expand_dims(reference, 0)
        return reference, np.broadcast_to(other, reference.shape)

    def get_action(self, obs: dict, infos: dict | None = None, *args, **kwargs):
        assert not self._key_in_nested_dict(obs, "action_mask"), \
            "AgileRL requires action masks to be defined in the information dictionary."
        env_defined_actions, agent_masks = self.extract_agent_masks(infos)
        states = self.preprocess_observation(obs)
        processed, raw = OrderedDict(), OrderedDict()
        action_dict, actor = {}, None
        for a in self.agent_ids:
            actor = self.actors[a]
            actions = actor(states[a]).cpu()
            if self.training:
                actions = torch.clamp(actions + self.action_noise(a), -1.0, 1.0)
            action_dict[a] = actions
        for a in self.agent_ids:
            # kept quirk (maddpg.py:504-511): the rescaling loop reads ``actor`` — the variable the loop above left pointing
            # at the LAST agent's network — so every agent's action is rescaled to the last agent's bounds (and agents
            # whose action widths differ from the last one's raise, as in the reference)
            processed[a] = DeterministicActor.rescale_action(action_dict[a], actor.action_low, actor.action_high,
                                                             actor.output_activation).numpy()
            raw[a] = action_dict[a].numpy()
        if env_defined_actions is not None:
            # maddpg.py:518-529 -> algo_utils.py:1822-1852: the environment's actions overwrite the PROCESSED actions where it
            # defines them, and (kept quirk) that same dict is what comes back as the "raw" actions too
            for a in self.agent_ids:
                action, override = self._reconcile_shapes(processed[a], np.asarray(env_defined_actions[a]))
                action, mask = self._reconcile_shapes(action, agent_masks[a])
                action[mask] = override[mask]
                processed[a] = action
            raw = processed
        return processed, raw

    def action_noise(self, agent_id: str) -> torch.Tensor:
        """maddpg.py:534-558 (torch's global CPU generator)."""
        if self.O_U_noise:
            noise = (self.current_noise[agent_id] + self.theta * (self.mean_noise[agent_id] - self.current_noise[agent_id]) * self.dt
                     + self.expl_noise[agent_id] * self.sqdt * self.sample_gaussian[agent_id].normal_())
            self.current_noise[agent_id] = noise
        else:
            torch.normal(self.mean_noise[agent_id], self.expl_noise[agent_id], out=self.sample_gaussian[agent_id])
            noise = self.sample_gaussian[agent_id]
        return noise

    def reset_action_noise(self, indices) -> None:
        for a in self.agent_ids:
            for idx in indices:
                self.current_noise[a][idx, :] = 0

    # -- learning ------------------------------------------------------------------------------------------
    def _workspace(self, B: int) -> torch.Tensor:
        ws = self._ws.get(B)
        if ws is None:
            need = ctypes.c_size_t(0)
            actors, critics = ctypes.cast(self._actor_descs, ctypes.c_void_p), ctypes.cast(self._critic_descs, ctypes.c_void_p)
            if len(self._CRITIC_SETS) == 2:            # a twin call also holds the critic_2 passes
                cfg = _lib.MaddpgCfg()
                cfg.batch, cfg.n_agents, cfg.twin = B, self.n_agents, 1
                _lib.check(_lib.load().b2rl_maddpg_workspace_bytes_cfg(actors, critics, ctypes.byref(cfg), ctypes.byref(need)))
            else:
                _lib.check(_lib.load().b2rl_maddpg_workspace_bytes(actors, critics, self.n_agents, B, ctypes.byref(need)))
            ws = self._ws[B] = torch.empty(need.value, dtype=torch.uint8, device=self._dev)
        return ws

    def _packed(self, field, width: int) -> torch.Tensor:
        """[B, sum] float32 matrix of a field: the replay's packed gather if it rides along, else the reference's
        ``torch.cat(list(field.values()), dim=1)`` in agent order."""
        m = getattr(field, "packed", None)
        if m is None:
            m = torch.cat([field[a].to(self._dev, dtype=torch.float32).reshape(field[a].shape[0], -1) for a in self.agent_ids], dim=1)
        if m.dtype != torch.float32 or m.device != self._dev or not m.is_contiguous():
            m = m.to(self._dev, dtype=torch.float32).contiguous()
        assert m.ndim == 2 and m.shape[1] == width, f"expected [B, {width}], got {tuple(m.shape)}"
        return m

    def learn(self, experiences) -> dict:
        """maddpg.py:571-628.  Returns ``{agent_id: (actor_loss, critic_loss)}`` as Python floats (MATD3: ``None`` for the
        actor loss of a call without an actor step)."""
        critic_only = self._next_critic_only()
        out = self.learn_device(experiences)
        host = out.tolist()
        return {a: (None if critic_only else host[i][0], host[i][1]) for i, a in enumerate(self.agent_ids)}

    # -- step kinds: MADDPG steps every optimiser and soft-updates every target on every call ------------------------
    def _next_critic_only(self) -> bool:
        """Whether the NEXT learn call updates the critics only (no actor step, no soft update)."""
        return False

    def _advance(self) -> bool:
        """Count the learn call about to run: optimiser step counts and ``learn_counter``.  -> its step kind."""
        for o in self._all_opts:
            o.step += 1
        self.learn_counter += 1
        return False

    def _bias_corrections(self, cfg) -> None:
        a_step = max(next(iter(self.actor_optimizers.values())).step, 1)
        c_step = max(next(iter(getattr(self, self._CRITIC_SETS[0][2]).values())).step, 1)
        cfg.bc1_actor, cfg.bc2_actor = 1.0 - 0.9 ** a_step, 1.0 - 0.999 ** a_step
        cfg.bc1_critic, cfg.bc2_critic = 1.0 - 0.9 ** c_step, 1.0 - 0.999 ** c_step

    def batch_buffers(self, B: int) -> list:
        """The static ``[B, sum]`` matrices a captured learn call reads, in the replay's field order (obs, action, reward,
        next_obs, done): ``MultiAgentReplayBuffer.sample_device(B, out=agent.batch_buffers(B))`` gathers straight into
        them and ``learn_device`` then replays the graph without copying the batch."""
        return self._plan(B).fields()

    def _plan(self, B: int) -> _LearnPlan:
        plan = self._plans.get(B)
        if plan is None:
            plan = self._plans[B] = _LearnPlan(self, B)
        return plan

    def _call_args(self, B, obs, next_obs, act, rew, done, out, state_dev=None, critic_only=False, actor_state_dev=None):
        n = self.n_agents
        cfg = _lib.MaddpgCfg()
        cfg.batch, cfg.n_agents, cfg.serial = B, n, int(not self.concurrent_agents)
        cfg.gamma, cfg.tau = float(self.gamma), float(self.tau)
        cfg.lr_actor, cfg.lr_critic, cfg.beta1, cfg.beta2, cfg.adam_eps = float(self.lr_actor), float(self.lr_critic), 0.9, 0.999, 1e-8
        cfg.twin, cfg.critic_only = int(len(self._CRITIC_SETS) == 2), int(critic_only)
        self._bias_corrections(cfg)
        bufs = _lib.MaddpgBufs()
        for i, a in enumerate(self.agent_ids):
            ao = self.actor_optimizers[a]
            bufs.actor[i], bufs.actor_target[i] = self.actors[a].buffers.params.data_ptr(), self.actor_targets[a].buffers.params.data_ptr()
            bufs.actor_grads[i], bufs.actor_m[i], bufs.actor_v[i] = ao.grads.data_ptr(), ao.exp_avg.data_ptr(), ao.exp_avg_sq.data_ptr()
            for k, (net, tgt, opt) in enumerate(self._CRITIC_SETS):
                co = getattr(self, opt)[a]
                pre = "critic" if k == 0 else "critic2"
                getattr(bufs, pre)[i] = getattr(self, net)[a].buffers.params.data_ptr()
                getattr(bufs, pre + "_target")[i] = getattr(self, tgt)[a].buffers.params.data_ptr()
                getattr(bufs, pre + "_grads")[i], getattr(bufs, pre + "_m")[i] = co.grads.data_ptr(), co.exp_avg.data_ptr()
                getattr(bufs, pre + "_v")[i] = co.exp_avg_sq.data_ptr()
        bufs.obs, bufs.next_obs, bufs.action = obs.data_ptr(), next_obs.data_ptr(), act.data_ptr()
        bufs.reward, bufs.done = rew.data_ptr(), done.data_ptr()
        bufs.losses = out.data_ptr()
        ws = self._workspace(B)
        bufs.workspace, bufs.workspace_bytes = ws.data_ptr(), ws.numel()
        bufs.step_state = state_dev.data_ptr() if state_dev is not None else None
        bufs.actor_step_state = actor_state_dev.data_ptr() if actor_state_dev is not None else None
        return cfg, bufs

    def _capture(self, plan: _LearnPlan, B: int, critic_only: bool = False) -> None:
        lib = _lib.load()
        # separate actor bias corrections: only a twin (MATD3) full step, whose actors lag the critics
        actor_state = plan.actor_state_dev if (len(self._CRITIC_SETS) == 2 and not critic_only) else None
        cfg, bufs = self._call_args(B, plan.obs, plan.next_obs, plan.action, plan.reward, plan.done, plan.out, plan.state_dev,
                                    critic_only, actor_state)
        plan.__dict__.setdefault("_keep", {})[critic_only] = (cfg, bufs)
        cap = torch.cuda.Stream(device=self._dev)
        cap.wait_stream(torch.cuda.current_stream(self._dev))
        s = cap.cuda_stream
        gh = ctypes.c_void_p()
        _lib.check(lib.b2rl_graph_begin(s))
        try:
            _lib.check(lib.b2rl_step_state_write(ctypes.byref(plan.state_host), plan.state_dev.data_ptr(), s))
            if actor_state is not None:
                _lib.check(lib.b2rl_step_state_write(ctypes.byref(plan.actor_state_host), actor_state.data_ptr(), s))
            _lib.check(lib.b2rl_maddpg_learn(ctypes.cast(self._actor_descs, ctypes.c_void_p),
                                             ctypes.cast(self._critic_descs, ctypes.c_void_p), ctypes.byref(cfg), ctypes.byref(bufs), s))
        finally:
            _lib.check(lib.b2rl_graph_end(s, ctypes.byref(gh)))
        plan.graphs[critic_only] = gh.value
        torch.cuda.current_stream(self._dev).wait_stream(cap)

    def graph_ready(self, B: int) -> bool:
        """A captured learn call for batch size ``B`` and the next call's step kind exists (the next ``learn_device`` on
        ``batch_buffers(B)`` is one graph launch and touches no torch state: it may be given an explicit stream)."""
        plan = self._plans.get(B)
        return bool(self.use_graph and plan is not None and plan.graphs.get(self._next_critic_only()) is not None)

    def learn_device(self, experiences, stream: int | None = None) -> torch.Tensor:
        """``learn`` without the host read-back: device tensor ``[n_agents, 2]`` (actor_loss, critic_loss; the actor column
        is NaN after a MATD3 call without an actor step).  With ``use_graph`` the tensor is the plan's static result buffer:
        valid until the next learn call of this batch size.  ``stream`` (raw ``cudaStream_t``; only when ``graph_ready``
        and the batch sits in ``batch_buffers``): launch there instead of on torch's current stream."""
        states, actions, rewards, next_states, dones = experiences
        critic_only = self._next_critic_only()
        if self.use_graph:          # the replay gathered straight into a captured call's buffers: nothing to check or copy
            p = getattr(states, "packed", None)
            plan = self._plans.get(p.shape[0]) if p is not None else None
            if (plan is not None and plan.graphs.get(critic_only) is not None and p is plan.obs
                    and getattr(actions, "packed", None) is plan.action and getattr(rewards, "packed", None) is plan.reward
                    and getattr(next_states, "packed", None) is plan.next_obs and getattr(dones, "packed", None) is plan.done):
                return self._replay(plan, stream)
        assert stream is None, "an explicit stream is only valid for a captured call on batch_buffers()"
        n = self.n_agents
        SO, SA = sum(self.obs_dims.values()), sum(self.action_dims.values())
        obs, next_obs, act = self._packed(states, SO), self._packed(next_states, SO), self._packed(actions, SA)
        rew, done = self._packed(rewards, n), self._packed(dones, n)      # [B, n_agents]: the replay's own layout
        B = obs.shape[0]
        assert next_obs.shape[0] == B and act.shape[0] == B and rew.shape == (B, n) and done.shape == (B, n)
        lib = _lib.load()
        if self.use_graph:
            plan = self._plan(B)
            for dst, src in zip(plan.fields(), (obs, act, rew, next_obs, done)):
                if dst.data_ptr() != src.data_ptr():
                    dst.copy_(src)
            if plan.graphs.get(critic_only) is None:
                self._workspace(B)                                # also creates the library's side streams: not under capture
                self._capture(plan, B, critic_only)
            return self._replay(plan)
        critic_only = self._advance()
        out = torch.empty((n, 2), dtype=torch.float32, device=self._dev)
        cfg, bufs = self._call_args(B, obs, next_obs, act, rew, done, out, critic_only=critic_only)
        _lib.check(lib.b2rl_maddpg_learn(ctypes.cast(self._actor_descs, ctypes.c_void_p),
                                         ctypes.cast(self._critic_descs, ctypes.c_void_p), ctypes.byref(cfg), ctypes.byref(bufs),
                                         _lib.stream_ptr(self._dev)))
        self._keep = (obs, next_obs, act, rew, done, out)
        return out

    def _replay(self, plan: _LearnPlan, stream: int | None = None) -> torch.Tensor:
        critic_only = self._advance()
        self._launch(plan, plan.graphs[critic_only], critic_only, _lib.stream_ptr(self._dev) if stream is None else stream)
        return plan.out

    def _launch(self, plan: _LearnPlan, graph, critic_only: bool, stream: int) -> None:
        """Replay a captured call with this step's Adam bias corrections (MADDPG: every optimiser's step count is one)."""
        step = self._all_opts[-1].step
        plan.state_host.bias_correction1, plan.state_host.bias_correction2 = 1.0 - 0.9 ** step, 1.0 - 0.999 ** step
        _lib.check(self._lib.b2rl_graph_launch(graph, plan.state_ref, stream))

    def soft_update(self, net, target) -> None:
        """maddpg.py:733-746."""
        p, t = net.buffers.params, target.buffers.params
        t.copy_(self.tau * p + (1.0 - self.tau) * t)

    def test(self, env, swap_channels: bool = False, max_steps: int | None = None, loop: int = 3, sum_scores: bool = True):
        """maddpg.py:756-875: mean score over ``loop`` episodes of a (vectorised) PettingZoo-style parallel environment;
        NaN rewards (inactive agents) count as 0, NaN terminations as True; appends to ``fitness``."""
        if swap_channels:
            raise NotImplementedError("image observations are not implemented for MADDPG on the CUDA path")
        self.set_training_mode(False)
        rewards = []
        is_vectorised = hasattr(env, "num_envs")
        num_envs = env.num_envs if is_vectorised else 1
        width = 1 if sum_scores else len(self.agent_ids)
        for _ in range(loop):
            obs, info = env.reset()
            scores, completed = np.zeros((num_envs, width)), np.zeros((num_envs, width))
            finished = np.zeros(num_envs)
            step = 0
            while not np.all(finished):
                step += 1
                action, _ = self.get_action(obs, infos=info)
                if not is_vectorised:
                    action = {agent: act[0] for agent, act in action.items()}
                obs, reward, term, trunc, info = env.step(action)
                agent_rewards = np.array(list(reward.values())).transpose()
                agent_rewards = np.where(np.isnan(agent_rewards), 0, agent_rewards)
                if sum_scores:
                    inc = np.sum(agent_rewards, axis=-1)[:, np.newaxis] if is_vectorised else np.sum(agent_rewards, axis=-1)
                else:
                    inc = agent_rewards
                scores += inc
                dones = {}
                for agent_id in self.agent_ids:
                    terminated, truncated = term.get(agent_id, True), trunc.get(agent_id, False)
                    terminated = np.where(np.isnan(terminated), True, terminated).astype(bool)
                    truncated = np.where(np.isnan(truncated), False, truncated).astype(bool)
                    dones[agent_id] = terminated | truncated
                if not is_vectorised:
                    dones = {agent: np.array([dones[agent_id]]) for agent in self.agent_ids}      # sic (maddpg.py:855-859)
                for idx, agent_dones in enumerate(zip(*dones.values())):
                    if (np.all(agent_dones) or (max_steps is not None and step == max_steps)) and not finished[idx]:
                        completed[idx] = scores[idx]
                        finished[idx] = 1
            rewards.append(np.mean(completed, axis=0))
        mean_fit = np.mean(rewards, axis=0)
        mean_fit = mean_fit[0] if sum_scores else mean_fit
        self.fitness.append(mean_fit)
        return mean_fit
