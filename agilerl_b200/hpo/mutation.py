"""``Mutations`` — drop-in for agilerl/hpo/mutation.py:168-1207 for the single-agent learners of this package and, for
parameter / hyper-parameter mutations, MADDPG (a policy that is a dict of per-agent networks).

Five mutation kinds with the reference's relative probabilities and RNG use (``self.rng =
np.random.default_rng(rand_seed)`` :303, ``rng.choice`` over the option list :335-339):
none / architecture / parameters / activation / RL hyper-parameter.  After architecture and
activation mutations the shared networks (``actor_target``) are rebuilt from the mutated
evaluation network and loaded with its weights (``reinit_shared_networks`` :104-164) and the
optimiser restarts (``reinit_optimizers``).  All of it is host-side control; the Gaussian
parameter mutation edits the flat HBM parameter buffer in place through named views."""
from __future__ import annotations

import random
import warnings

import numpy as np
import torch


def set_global_seed(seed: int | None) -> None:
    """mutation.py:41-54 (fastrand is not in the image; numpy / torch / random are seeded)."""
    if seed is None:
        return
    torch.manual_seed(seed)
    np.random.seed(seed)
    random.seed(seed)


class MutationError(Exception):
    """mutation.py:1206-1207."""


def get_offspring_eval_modules(individual) -> tuple[dict, dict]:
    """mutation.py:57-82: clones of every registered evaluation network, split into (policy, the rest)."""
    policy, rest = {}, {}
    for group in individual.registry.groups:
        net = getattr(individual, group.eval_network)
        offspring = {k: v.clone() for k, v in net.items()} if isinstance(net, dict) else net.clone()
        (policy if group.policy else rest)[group.eval_network] = offspring
    return policy, rest


def get_exp_layer(offspring):
    """mutation.py:85-101 serves the bandit learners, which are outside this package."""
    raise TypeError(f"Bandit algorithm architecture {type(offspring)} not supported.")


class Mutations:
    def __init__(self, no_mutation: float, architecture: float, new_layer_prob: float, parameters: float,
                 activation: float, rl_hp: float, mutation_sd: float = 0.1, activation_selection: list | None = None,
                 mutate_elite: bool = True, rand_seed: int | None = None, device: str = "cuda", accelerator=None) -> None:
        if activation_selection is None:
            activation_selection = ["ReLU", "ELU", "GELU"]
        for name, v in (("no mutation", no_mutation), ("architecture mutation", architecture),
                        ("parameters mutation", parameters), ("activation mutation", activation),
                        ("reinforcement learning hyperparameter mutation", rl_hp)):
            assert isinstance(v, (float, int)), f"Probability of {name} must be a float or integer."
            assert v >= 0, f"Probability of {name} must be greater than or equal to zero."
        assert isinstance(new_layer_prob, (float, int)), (
            "Probability of new layer architecture mutation must be a float or integer.")
        assert 1 >= new_layer_prob >= 0, (
            "Probability of new layer architecture mutation must be between zero and one (inclusive).")
        assert mutation_sd >= 0, "Mutation strength must be greater than or equal to zero."
        assert isinstance(mutation_sd, (float, int)), "Mutation strength must be a float or integer."
        assert isinstance(mutate_elite, bool), "Mutate elite must be boolean value True or False."
        assert isinstance(rand_seed, int) or rand_seed is None, "Random seed must be an integer or None."
        if isinstance(rand_seed, int):
            assert rand_seed >= 0, "Random seed must be greater than or equal to zero."
        if accelerator is not None:
            raise NotImplementedError("accelerate is replaced by one-agent-per-GPU sharding")
        set_global_seed(rand_seed)
        self.rng = np.random.default_rng(rand_seed)
        self.no_mut, self.architecture_mut, self.new_layer_prob = no_mutation, architecture, new_layer_prob
        self.parameters_mut, self.activation_mut, self.rl_hp_mut = parameters, activation, rl_hp
        self.mutation_sd, self.activation_selection = mutation_sd, activation_selection
        self.mutate_elite, self.device, self.accelerator = mutate_elite, device, None
        self.mut_options, self.mut_proba = self._get_mutations_options()
        self.pretraining_mut_options, self.pretraining_mut_proba = self._get_mutations_options(pretraining=True)

    def _get_mutations_options(self, pretraining: bool = False):
        """mutation.py:586-621."""
        opts = [(self.no_mutation, self.no_mut), (self.architecture_mutate, self.architecture_mut),
                (self.parameter_mutation, self.parameters_mut), (self.activation_mutation, self.activation_mut),
                (self.rl_hyperparam_mutation, self.rl_hp_mut)]
        if pretraining:
            opts[0] = (self.no_mutation, 0)
        funcs, probs = zip(*opts)
        total = sum(probs)
        if total == 0:
            return [self.no_mutation], [1.0]
        return list(funcs), [p / total for p in probs]

    def mutation(self, population, pre_training_mut: bool = False):
        """mutation.py:311-362."""
        options = self.pretraining_mut_options if pre_training_mut else self.mut_options
        proba = self.pretraining_mut_proba if pre_training_mut else self.mut_proba
        choice = list(self.rng.choice(options, len(population), p=proba))
        if not self.mutate_elite:
            choice[0] = self.no_mutation
        out = []
        for mut, individual in zip(choice, population):
            individual = mut(individual)
            individual.mutation_hook()
            out.append(individual)
        return out

    # -- the five kinds -----------------------------------------------------------------------------
    def no_mutation(self, individual):
        individual.mut = "None"
        return individual

    def _reinit_shared(self, individual):
        """reinit_shared_networks (mutation.py:104-164): rebuild each shared network from the
        mutated evaluation network's init_dict and load its weights."""
        if individual.mut == "None":
            return individual
        for group in individual.registry.groups:
            if group.shared_networks is None:
                continue
            eval_net = getattr(individual, group.eval_network)
            for shared_name in group.shared_networks:
                shared = type(eval_net)(**eval_net.init_dict)
                shared.load_state_dict(eval_net.state_dict(), strict=False)
                setattr(individual, shared_name, shared)
        return individual

    def architecture_mutate(self, individual):
        """mutation.py:373-411 + _architecture_mutate_single :829-885."""
        registry = individual.registry
        policy = getattr(individual, registry.policy())
        if isinstance(policy, dict):
            raise NotImplementedError("architecture mutations of multi-agent networks (mutation.py:887-1010) are not implemented "
                                      "on the CUDA path: use parameter / RL hyper-parameter mutations for MADDPG / MATD3")
        if not policy.mutation_methods:
            individual.mut = "None"
            return individual
        method = policy.sample_mutation_method(self.new_layer_prob, self.rng)
        mut_dict = method()
        applied = policy.last_mutation_attr
        individual.mut = applied if applied is not None else "None"
        # mutation.py:875-879: the SAME mutation (name and the parameters the policy's mutation drew) goes to the other
        # evaluation networks that have it — the critics of DDPG / TD3 keep the policy's architecture
        if applied is not None:
            for group in registry.groups:
                if group.policy:
                    continue
                other = getattr(individual, group.eval_network)
                methods = other.get_mutation_methods() if hasattr(other, "get_mutation_methods") else {}
                if applied in methods:
                    methods[applied](**(mut_dict if isinstance(mut_dict, dict) else {}))
        self._reinit_shared(individual)
        individual.reinit_optimizers()
        return individual

    def rl_hyperparam_mutation(self, individual):
        """mutation.py:413-452."""
        hp_config = individual.registry.hp_config
        if not hp_config:
            individual.mut = "None"
            return individual
        attr, param = hp_config.sample()
        if param.value is None:
            param.value = getattr(individual, attr)
        new_value = param.mutate()
        setattr(individual, attr, new_value)
        if attr in individual.get_lr_names():
            individual.reinit_optimizers()
        individual.mut = attr
        return individual

    def _permutate_activation(self, network):
        """mutation.py:710-731: a different activation from the selection (one draw from ``self.rng``)."""
        possible = list(self.activation_selection)
        current = network.activation
        if len(possible) > 1 and current in possible:
            possible.remove(current)
        network.change_activation(str(self.rng.choice(possible, size=1)[0]), output=False)
        return network

    def activation_mutation(self, individual):
        """mutation.py:454-519."""
        if individual.algo in ["PPO", "DDPG", "TD3", "IPPO", "MADDPG", "MATD3", "GRPO"]:
            warnings.warn(f"Activation mutations are not supported for {individual.algo}.", stacklevel=2)
            individual.mut = "None"
            return individual
        for group in individual.registry.groups:
            net = getattr(individual, group.eval_network)
            if net.activation is None:
                individual.mut = "None"
                return individual
            self._permutate_activation(net)
        individual.mut = "act"
        self._reinit_shared(individual)
        individual.reinit_optimizers()
        return individual

    def parameter_mutation(self, individual):
        """mutation.py:521-584.  A multi-agent policy is a dict of networks keyed by agent id (the reference's
        ``ModuleDict`` branch, :545-547): every sub-agent's network is mutated in turn."""
        group = individual.registry.policy(return_group=True)
        policy = getattr(individual, group.eval_network)
        mutate = self._gaussian_parameter_mutation_device if getattr(self, "device_parameter_mutation", False) else \
            self._gaussian_parameter_mutation
        if isinstance(policy, dict):
            for agent_id, module in policy.items():
                policy[agent_id] = mutate(module)
            for shared in group.shared_networks or []:
                for agent_id, module in getattr(individual, shared).items():
                    module.load_state_dict(policy[agent_id].state_dict(), strict=False)
        else:
            mutate(policy)
            for shared in group.shared_networks or []:
                getattr(individual, shared).load_state_dict(policy.state_dict(), strict=False)
        individual.reinit_optimizers()
        individual.mut = "param"
        return individual

    #: opt-in (attribute, the constructor keeps the reference's signature): run the Gaussian parameter mutation ON THE
    #: DEVICE (SURVEY 8f-4).  Positions and branch uniforms still come from ``self.rng`` — the same keys, rows, columns
    #: and branches as the reference — but the noise comes from the library's Philox stream instead of torch's CPU
    #: generator, so weights are distributed like the reference's, not bit-identical to a seeded reference run.
    device_parameter_mutation = False
    _device_mutation_offset = 0

    def _gaussian_parameter_mutation_device(self, network, normals: dict | None = None):
        """mutation.py:733-827 with the ``index_put`` of the mutated 10 % of each chosen matrix done by
        ``b2rl_gaussian_mutate`` in place on the flat HBM parameter buffer (no host copy of the weights).
        ``normals`` ({key: float32 [n_mut]}, tests) injects the standard-normal draws."""
        from .. import _lib
        lib = _lib.load()
        entries = network.layout.entries
        keys = [k for k, e in entries.items() if "lstm" not in k and "norm" not in k and len(e.shape) == 2]
        how_many = int(self.rng.integers(1, len(keys) + 1))
        dev = network.buffers.params.device
        for key in self.rng.choice(keys, how_many, replace=False):
            key = str(key)
            view = network.buffers.view(key)
            n_rows, n_cols = int(view.shape[0]), int(view.shape[1])
            n_mut = int(np.ceil(0.1 * n_rows * n_cols))
            if n_mut < 1:
                continue
            rows = self.rng.integers(0, n_rows, size=n_mut)
            cols = self.rng.integers(0, n_cols, size=n_mut)
            u = self.rng.uniform(0, 1, size=n_mut).astype(np.float32)          # torch.tensor(rand_vals, dtype=W.dtype)
            flat = rows.astype(np.int64) * n_cols + cols.astype(np.int64)
            keep = np.zeros(n_mut, dtype=np.uint8)                             # index_put_: the last writer of a position wins
            _, last_from_end = np.unique(flat[::-1], return_index=True)
            keep[n_mut - 1 - last_from_end] = 1
            host = torch.from_numpy(np.concatenate([rows.astype(np.int64), cols.astype(np.int64)]))
            idx = host.to(dev)
            u_d, keep_d = torch.from_numpy(u).to(dev), torch.from_numpy(keep).to(dev)
            z = None
            if normals is not None:
                z = normals[key].to(dev, dtype=torch.float32).contiguous()
                assert z.numel() == n_mut
            _lib.check(lib.b2rl_gaussian_mutate(view.data_ptr(), n_rows, n_cols, idx.data_ptr(), idx[n_mut:].data_ptr(),
                                                u_d.data_ptr(), keep_d.data_ptr(), z.data_ptr() if z is not None else None,
                                                0x6D757461 + 7919 * int(getattr(self, "_device_mutation_seed", 0)),
                                                self._device_mutation_offset, float(self.mutation_sd), n_mut,
                                                _lib.stream_ptr(dev)))
            self._device_mutation_offset += n_mut
            self._keep_mut = (idx, u_d, keep_d, z)
        return network

    def _gaussian_parameter_mutation(self, network):
        """mutation.py:733-827, bit for bit.  The reference walks ``state_dict()`` — parameters AND the 2-D NoisyLinear
        epsilon buffers, in module order — picks keys / rows / columns / branch with ``self.rng`` and draws the noise from
        torch's global CPU generator; duplicate (row, col) pairs resolve to the last writer like a CPU ``index_put_``.
        Mutations are off the hot path: each chosen matrix is mutated on a host copy with exactly those torch calls and
        written back into the flat HBM buffer."""
        mut_strength, frac = self.mutation_sd, 0.1
        super_strength, super_prob = 10, 0.05
        reset_prob, mag_limit = super_prob + 0.05, 1000000
        entries = network.layout.entries
        keys = [k for k, e in entries.items() if "lstm" not in k and "norm" not in k and len(e.shape) == 2]
        how_many = int(self.rng.integers(1, len(keys) + 1))
        for key in self.rng.choice(keys, how_many, replace=False):
            view = network.buffers.view(str(key))
            W = view.cpu()
            n_mut = int(np.ceil(frac * W.shape[0] * W.shape[1]))
            if n_mut < 1:
                continue
            rows = torch.tensor(self.rng.integers(0, W.shape[0], size=n_mut), dtype=torch.long)
            cols = torch.tensor(self.rng.integers(0, W.shape[1], size=n_mut), dtype=torch.long)
            r = torch.tensor(self.rng.uniform(0, 1, size=n_mut), dtype=W.dtype)
            cur = W[rows, cols]
            new = cur.clone()
            m_super, m_reset = r < super_prob, (r >= super_prob) & (r < reset_prob)
            m_norm = r >= reset_prob
            if m_super.sum() > 0:
                std = (super_strength * cur[m_super]).abs()
                new[m_super] = cur[m_super] + torch.normal(mean=torch.zeros_like(std), std=std)
            if m_reset.sum() > 0:
                k = m_reset.sum()
                new[m_reset] = torch.normal(mean=torch.zeros(k), std=torch.ones(k))
            if m_norm.sum() > 0:
                std = (mut_strength * cur[m_norm]).abs()
                new[m_norm] = cur[m_norm] + torch.normal(mean=torch.zeros_like(std), std=std)
            W[rows, cols] = new.clamp(min=-mag_limit, max=mag_limit)
            view.copy_(W)
        return network
