"""Population helpers — mirrors of agilerl/utils/utils.py:218-653 (``create_population`` for the
learners of this package: DQN, Rainbow DQN, DDPG, TD3, MADDPG, MATD3) and :706-796 (``tournament_selection_and_mutation``, the
non-accelerate branch :785-786)."""
from __future__ import annotations

from typing import Any

from ..algorithms import DDPG, DQN, MADDPG, MATD3, TD3, RainbowDQN


def create_population(algo: str, observation_space, action_space, net_config: dict | None, INIT_HP: dict,
                      hp_config=None, actor_network=None, population_size: int = 1, num_envs: int = 1,
                      device: str = "cuda", accelerator: Any | None = None, torch_compiler=None,
                      first_index: int = 0, critic_network=None, algo_kwargs: dict | None = None) -> list:
    """utils/utils.py:218-474.  ``first_index`` numbers the agents of a population shard."""
    population = []
    algo_kwargs = algo_kwargs or {}
    if algo in ("MADDPG", "MATD3") and INIT_HP.get("SHARE_ENCODERS", False):
        raise NotImplementedError(f"SHARE_ENCODERS is not implemented for {algo} on the CUDA path")
    noise = dict(O_U_noise=INIT_HP.get("O_U_NOISE", True), expl_noise=INIT_HP.get("EXPL_NOISE", 0.1), vect_noise_dim=num_envs,
                 mean_noise=INIT_HP.get("MEAN_NOISE", 0.0), theta=INIT_HP.get("THETA", 0.15), dt=INIT_HP.get("DT", 0.01))
    pg = dict(hp_config=hp_config, net_config=net_config, batch_size=INIT_HP.get("BATCH_SIZE", 64),
              lr_actor=INIT_HP.get("LR_ACTOR", 0.0001), lr_critic=INIT_HP.get("LR_CRITIC", 0.001),
              learn_step=INIT_HP.get("LEARN_STEP", 5), device=device, accelerator=accelerator)
    for i in range(population_size):
        idx = first_index + i
        if algo == "DQN":
            agent = DQN(observation_space=observation_space, action_space=action_space, index=idx, hp_config=hp_config,
                        net_config=net_config, batch_size=INIT_HP.get("BATCH_SIZE", 64), lr=INIT_HP.get("LR", 1e-4),
                        learn_step=INIT_HP.get("LEARN_STEP", 5), gamma=INIT_HP.get("GAMMA", 0.99),
                        tau=INIT_HP.get("TAU", 1e-3), double=INIT_HP.get("DOUBLE", False),
                        actor_network=actor_network, device=device, accelerator=accelerator)
        elif algo == "Rainbow DQN":
            # note the create_population defaults differ from the class defaults (utils.py:308-311)
            agent = RainbowDQN(observation_space=observation_space, action_space=action_space, index=idx,
                               hp_config=hp_config, net_config=net_config, batch_size=INIT_HP.get("BATCH_SIZE", 64),
                               lr=INIT_HP.get("LR", 1e-4), learn_step=INIT_HP.get("LEARN_STEP", 5),
                               gamma=INIT_HP.get("GAMMA", 0.99), tau=INIT_HP.get("TAU", 1e-3),
                               beta=INIT_HP.get("BETA", 0.4), prior_eps=INIT_HP.get("PRIOR_EPS", 1e-5),
                               num_atoms=INIT_HP.get("NUM_ATOMS", 51), v_min=INIT_HP.get("V_MIN", -100),
                               v_max=INIT_HP.get("V_MAX", 100), n_step=INIT_HP.get("N_STEP", 3),
                               actor_network=actor_network, device=device, accelerator=accelerator)
        elif algo == "DDPG":                                                    # utils.py:320-352
            agent = DDPG(observation_space=observation_space, action_space=action_space, index=idx, gamma=INIT_HP.get("GAMMA", 0.99),
                         tau=INIT_HP.get("TAU", 0.001), policy_freq=INIT_HP.get("POLICY_FREQ", 2), actor_network=actor_network,
                         critic_network=critic_network, share_encoders=INIT_HP.get("SHARE_ENCODERS", True), **noise, **pg,
                         **algo_kwargs)
        elif algo == "TD3":                                                     # utils.py:414-442
            agent = TD3(observation_space=observation_space, action_space=action_space, index=idx, gamma=INIT_HP.get("GAMMA", 0.99),
                        tau=INIT_HP.get("TAU", 0.005), policy_freq=INIT_HP.get("POLICY_FREQ", 2), actor_network=actor_network,
                        critic_networks=critic_network, share_encoders=INIT_HP.get("SHARE_ENCODERS", True), **noise, **pg,
                        **algo_kwargs)
        elif algo == "MADDPG":                                                  # utils.py:444-472
            agent = MADDPG(observation_spaces=observation_space, action_spaces=action_space, agent_ids=INIT_HP["AGENT_IDS"],
                           index=idx, gamma=INIT_HP.get("GAMMA", 0.95), tau=INIT_HP.get("TAU", 0.01),
                           actor_networks=actor_network, critic_networks=critic_network, torch_compiler=torch_compiler,
                           **noise, **pg, **algo_kwargs)
        elif algo == "MATD3":                                                   # utils.py:474-500
            agent = MATD3(observation_spaces=observation_space, action_spaces=action_space, agent_ids=INIT_HP["AGENT_IDS"],
                          index=idx, policy_freq=INIT_HP.get("POLICY_FREQ", 2), gamma=INIT_HP.get("GAMMA", 0.95),
                          tau=INIT_HP.get("TAU", 0.01), actor_networks=actor_network, critic_networks=critic_network,
                          torch_compiler=torch_compiler, **noise, **pg, **algo_kwargs)
        else:
            raise NotImplementedError(f"{algo}: not one of the learners of this package (DQN, Rainbow DQN, DDPG, TD3, MADDPG, MATD3; "
                                      "SURVEY §8)")
        population.append(agent)
    return population


def tournament_selection_and_mutation(population: list, tournament, mutation, env_name: str = "", algo: str | None = None,
                                      elite_path: str | None = None, save_elite: bool = False, accelerator=None,
                                      language_model: bool = False) -> list:
    """utils/utils.py:706-796 without the accelerate/disk-checkpoint transport: selection (with the
    fitness all-gather when the population is sharded over ranks) then mutation."""
    elite, population = tournament.select(population)
    population = mutation.mutation(population)
    if save_elite:
        elite.save_checkpoint(elite_path if elite_path is not None else f"{env_name}-elite_{algo}.pt")
    return population
