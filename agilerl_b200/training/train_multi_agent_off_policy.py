"""``train_multi_agent_off_policy`` — same signature and control flow as
agilerl/training/train_multi_agent_off_policy.py:32-600 for the multi-agent learners of this package (MADDPG, MATD3), minus the
W&B / accelerate plumbing and image-observation channel swapping (the CUDA learners take vector observations).  The reference's
file cannot be imported on the GPU box (pettingzoo / accelerate / wandb are absent there), so this module restates its loop;
``tests/test_reference_driver_cpu.py`` runs both files on the same seeded population, environment and stand-in kernels and
requires identical fitnesses, scores, steps, mutations and replay contents.

Per environment step (:239-283): ``agent.get_action(obs, infos)`` -> processed actions to the environment, RAW actions into
the shared ``MultiAgentReplayBuffer``; learning every ``learn_step`` steps from ``Sampler(memory).sample(batch_size)``; episode
bookkeeping with NaN (dead agent) handling; per generation (:395-535) ``agent.test`` then tournament selection and mutation;
population checkpoints named like ``utils.save_population_checkpoint`` (utils.py:682-688).  Loops that keep the whole
population learning on the device use ``training.population.multi_agent_population_learn`` instead."""
from __future__ import annotations

import time
import warnings
from copy import deepcopy

import numpy as np

from ..components import Sampler
from ..utils.utils import tournament_selection_and_mutation


def train_multi_agent_off_policy(env, env_name: str, algo: str, pop: list, memory, sum_scores: bool = True,
                                 INIT_HP: dict | None = None, MUT_P: dict | None = None, swap_channels: bool = False,
                                 max_steps: int = 50000, evo_steps: int = 25, eval_steps: int | None = None, eval_loop: int = 1,
                                 learning_delay: int = 0, target: float | None = None, tournament=None, mutation=None,
                                 checkpoint: int | None = None, checkpoint_path: str | None = None,
                                 overwrite_checkpoints: bool = False, save_elite: bool = False, elite_path: str | None = None,
                                 wb: bool = False, verbose: bool = True, accelerator=None, wandb_api_key: str | None = None):
    assert isinstance(algo, str), "'algo' must be the name of the algorithm as a string."
    assert isinstance(max_steps, int), "Number of steps must be an integer."
    assert isinstance(evo_steps, int), "Evolution frequency must be an integer."
    if target is not None:
        assert isinstance(target, (float, int)), "Target score must be a float or an integer."
    if checkpoint is not None:
        assert isinstance(checkpoint, int), "Checkpoint must be an integer."
    assert isinstance(wb, bool), "'wb' must be a boolean flag, indicating whether to record run with W&B"
    assert isinstance(verbose, bool), "Verbose must be a boolean."
    if wb or accelerator is not None:
        raise NotImplementedError("W&B logging / accelerate are outside this package (the population shards one process per GPU)")
    if swap_channels:
        raise NotImplementedError(f"image observations are not implemented for {algo} on the CUDA path")
    if save_elite is False and elite_path is not None:
        warnings.warn("'save_elite' set to False but 'elite_path' has been defined, elite will not be saved unless 'save_elite' "
                      "is set to True.", stacklevel=2)
    if checkpoint is None and checkpoint_path is not None:
        warnings.warn("'checkpoint' set to None but 'checkpoint_path' has been defined, checkpoint will not be saved unless "
                      "'checkpoint' is defined.", stacklevel=2)
    is_vectorised = hasattr(env, "num_envs")
    num_envs = env.num_envs if is_vectorised else 1
    save_path = checkpoint_path.split(".pt")[0] if checkpoint_path is not None else \
        f"{env_name}-EvoHPO-{algo}-{time.strftime('%m%d%Y%H%M%S')}"
    sampler = Sampler(memory=memory)
    agent_ids = deepcopy(env.agents)
    pop_actor_loss = [{a: [] for a in agent_ids} for _ in pop]
    pop_critic_loss = [{a: [] for a in agent_ids} for _ in pop]
    pop_fitnesses, total_steps, checkpoint_count = [], 0, 0
    width = 1 if sum_scores else len(agent_ids)
    if mutation is not None:                                            # :204-206 pre-training mutation
        pop = mutation.mutation(pop, pre_training_mut=True)
    while np.less([agent.steps[-1] for agent in pop], max_steps).all():
        pop_episode_scores, pop_fps = [], []
        for agent_idx, agent in enumerate(pop):
            agent.set_training_mode(True)
            obs, info = env.reset()
            scores = np.zeros((num_envs, width))
            losses = {a: [] for a in agent_ids}
            completed_episode_scores, steps = [], 0
            start_time = time.time()
            for idx_step in range(evo_steps // num_envs):
                action, raw_action = agent.get_action(obs=obs, infos=info)
                if not is_vectorised:
                    action = {a: act[0] for a, act in action.items()}
                next_obs, reward, termination, truncation, info = env.step(action)
                agent_rewards = np.array(list(reward.values())).transpose()
                agent_rewards = np.where(np.isnan(agent_rewards), 0, agent_rewards)          # inactive agents score 0
                if sum_scores:
                    scores += np.sum(agent_rewards, axis=-1)[:, np.newaxis] if is_vectorised else np.sum(agent_rewards, axis=-1)
                else:
                    scores += agent_rewards
                total_steps += num_envs
                steps += num_envs
                memory.save_to_memory(obs, raw_action, reward, next_obs, termination, is_vectorised=is_vectorised)
                ready = len(memory) >= agent.batch_size and memory.counter > learning_delay
                if agent.learn_step > num_envs:
                    n_learn = 1 if (idx_step % (agent.learn_step // num_envs) == 0 and ready) else 0
                else:
                    n_learn = (num_envs // agent.learn_step) if ready else 0
                for _ in range(n_learn):
                    loss = agent.learn(sampler.sample(agent.batch_size))
                    for a in agent_ids:
                        losses[a].append(loss[a])
                obs = next_obs
                reset_noise_indices, dones = [], {}
                for a in agent.agent_ids:
                    terminated, truncated = termination.get(a, True), truncation.get(a, False)
                    terminated = np.where(np.isnan(terminated), True, terminated).astype(bool)      # NaN: a killed agent
                    truncated = np.where(np.isnan(truncated), False, truncated).astype(bool)
                    dones[a] = terminated | truncated
                if not is_vectorised:
                    dones = {a: np.array([dones[a]]) for a in agent.agent_ids}
                for idx, agent_dones in enumerate(zip(*dones.values())):
                    if all(agent_dones):
                        completed = np.asarray(scores[idx]).item() if sum_scores else list(scores[idx])
                        completed_episode_scores.append(completed)
                        agent.scores.append(completed)
                        scores[idx].fill(0)
                        reset_noise_indices.append(idx)
                        if not is_vectorised:
                            obs, info = env.reset()
                agent.reset_action_noise(reset_noise_indices)
            agent.steps[-1] += steps
            pop_fps.append(steps / max(time.time() - start_time, 1e-12))
            pop_episode_scores.append(completed_episode_scores)
            if len(losses[agent_ids[0]]) > 0 and all(losses[a] for a in agent_ids):
                for a in agent_ids:
                    actor_losses, critic_losses = list(zip(*losses[a]))
                    actor_losses = [l for l in actor_losses if l is not None]
                    if actor_losses:
                        pop_actor_loss[agent_idx][a].append(np.mean(actor_losses))
                    pop_critic_loss[agent_idx][a].append(np.mean(critic_losses))
        fitnesses = [agent.test(env, swap_channels=swap_channels, max_steps=eval_steps, loop=eval_loop, sum_scores=sum_scores)
                     for agent in pop]
        pop_fitnesses.append(fitnesses)
        for agent in pop:
            agent.steps.append(agent.steps[-1])
        if target is not None and np.all(np.greater([np.mean(a.fitness[-10:]) for a in pop], target)) and len(pop[0].steps) >= 100:
            return pop, pop_fitnesses
        if tournament and mutation is not None:
            pop = tournament_selection_and_mutation(population=pop, tournament=tournament, mutation=mutation, env_name=env_name,
                                                    algo=algo, elite_path=elite_path, save_elite=save_elite)
        if verbose:
            print(f"--- Global steps {total_steps} --- fitness {fitnesses} fps {['%.0f' % f for f in pop_fps]} "
                  f"agents {[a.index for a in pop]} steps {[a.steps[-1] for a in pop]} mutations {[a.mut for a in pop]}")
        if checkpoint is not None and pop[0].steps[-1] // checkpoint > checkpoint_count:
            for i, agent in enumerate(pop):
                agent.save_checkpoint(f"{save_path}_{i}.pt" if overwrite_checkpoints else f"{save_path}_{i}_{agent.steps[-1]}.pt")
            checkpoint_count += 1
    return pop, pop_fitnesses
