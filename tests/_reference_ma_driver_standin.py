"""Helper of tests/test_reference_driver_cpu.py (own process): the UNCHANGED reference multi-agent driver
``/root/reference/agilerl/training/train_multi_agent_off_policy.py`` drives THIS package's ``MADDPG`` population and
``MultiAgentReplayBuffer`` (BASELINE configs[4] flow: ``get_action(obs, infos)`` -> env -> ``memory.save_to_memory(...,
is_vectorised)`` -> ``Sampler(memory).sample(B)`` -> ``agent.learn`` -> ``agent.test`` -> tournament + mutation), with Python
stand-ins for the C entry points (bytes movers; actor forward = deterministic pseudo actions; the learn call checks the
batch matrices it is handed and reports losses).  Call-level drop-in evidence; numerics are tests/test_maddpg_gpu.py's."""
import ctypes
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ["B2RL_MADDPG_GRAPH"] = "0"                  # eager learn call: graph capture needs the real library

from oracle import refshim  # noqa: E402

REFERENCE = "--without-reference" not in sys.argv     # tests/_driver_equivalence_standin.py: our driver alone
if REFERENCE:
    refshim.install()
import agilerl_b200  # noqa: E402
from agilerl_b200 import _lib  # noqa: E402
from agilerl_b200.components import replay_buffer as rb  # noqa: E402
from test_multi_agent_host_cpu import StandIn, _f32  # noqa: E402

calls = {"learn": 0, "forward_rows": 0, "saves": 0}
IDS, OD, AD, E = ["speaker_0", "listener_0", "listener_1"], 6, 3, 2


class Lib(StandIn):
    def b2rl_actor_workspace_bytes(self, desc, rows, out):
        out._obj.value = 256
        return 0

    def b2rl_actor_forward(self, desc, params, obs, rows, out, ws, wsb, stream):
        d = desc._obj
        a = d.val[d.n_val - 1].out_c
        x = _f32(obs, rows * d.obs_elems).reshape(rows, d.obs_elems)
        _f32(out, rows * a).reshape(rows, a)[:] = np.tanh(x.sum(axis=1, keepdims=True) * (np.arange(a) + 1.0) * 0.1)
        calls["forward_rows"] += rows
        return 0

    def b2rl_maddpg_learn(self, actors, critics, cfg, bufs, stream):
        c, b = cfg._obj, bufs._obj
        B, n = c.batch, c.n_agents
        assert n == len(IDS) and b.step_state is None
        obs, act = _f32(b.obs, B * n * OD), _f32(b.action, B * n * AD)
        rew, done = _f32(b.reward, B * n).reshape(B, n), _f32(b.done, B * n).reshape(B, n)
        assert np.isfinite(obs).all() and (np.abs(act) <= 1.0 + 1e-6).all()            # RAW actions are stored (driver :274-281)
        assert np.isin(done[~np.isnan(done)], (0.0, 1.0)).all() and np.isfinite(rew[~np.isnan(rew)]).all()
        _f32(b.losses, 2 * n)[:] = np.arange(2 * n) * 0.1 + calls["learn"] * 1e-3
        calls["learn"] += 1
        return 0


lib = Lib()
_lib.as_device = lambda d: torch.device("cpu")
_lib.load = lambda require_cuda=False: lib
_lib.stream_ptr = lambda d=None: 0
_lib.check = lambda rc: None
_lib.require_cuda_tensor = lambda t, what="tensor": None
torch.Tensor.pin_memory = lambda self: self
rb._PinnedRing.sent = lambda self, k, dev: None

agilerl_b200.install(include_driver=False)
import agilerl_b200.algorithms as A  # noqa: E402
import agilerl_b200.components as C  # noqa: E402
import agilerl_b200.hpo as H  # noqa: E402

if REFERENCE:
    import inspect

    import agilerl.training.train_multi_agent_off_policy as T

    assert inspect.getsourcefile(T).startswith(refshim.REFERENCE_ROOT), inspect.getsourcefile(T)
    assert T.MADDPG is A.MADDPG and T.MultiAgentReplayBuffer is C.MultiAgentReplayBuffer and T.Sampler is C.Sampler
    assert T.Mutations is H.Mutations and T.TournamentSelection is H.TournamentSelection
from agilerl_b200.compat import spaces  # noqa: E402
from agilerl_b200.utils.utils import create_population  # noqa: E402


class ParallelVecEnv:
    """PettingZoo-style parallel environment, vectorised over E copies; listener_1 is dead (NaN reward / termination) on some
    steps, episodes end every 6 steps."""
    num_envs, agents = E, list(IDS)

    def __init__(self, seed=0):
        self.rng, self.t = np.random.default_rng(seed), 0

    def _obs(self):
        return {a: self.rng.standard_normal((E, OD)).astype(np.float32) for a in IDS}

    def reset(self):
        self.t = 0
        return self._obs(), {a: {} for a in IDS}

    def step(self, action):
        assert set(action) == set(IDS) and all(np.asarray(v).shape == (E, AD) for v in action.values())
        self.t += 1
        end = self.t % 6 == 0
        rew = {a: self.rng.standard_normal(E) for a in IDS}
        term = {a: np.full(E, float(end)) for a in IDS}
        if self.t % 4 == 1:
            rew["listener_1"] = np.full(E, np.nan)
            term["listener_1"] = np.full(E, np.nan)
        if end:
            self.t = 0
        return self._obs(), rew, term, {a: np.zeros(E, bool) for a in IDS}, {a: {} for a in IDS}


obs_spaces = [spaces.Box(-np.inf, np.inf, (OD,), np.float32) for _ in IDS]
act_spaces = [spaces.Box(-1.0, 1.0, (AD,), np.float32) for _ in IDS]
INIT_HP = {"AGENT_IDS": IDS, "BATCH_SIZE": 8, "LEARN_STEP": 2, "N_AGENTS": len(IDS)}
pop = create_population("MADDPG", obs_spaces, act_spaces, None, INIT_HP, population_size=3, num_envs=E)
memory = C.MultiAgentReplayBuffer(200, ["obs", "action", "reward", "next_obs", "done"], IDS, device="cuda")
orig_save = memory.save_to_memory


def counting_save(*a, **k):
    calls["saves"] += 1
    return orig_save(*a, **k)


memory.save_to_memory = counting_save
pop, fits = T.train_multi_agent_off_policy(ParallelVecEnv(), "synthetic", "MADDPG", pop, memory, INIT_HP=INIT_HP, MUT_P={}, max_steps=96,
                                           evo_steps=32, eval_steps=12, eval_loop=1, tournament=H.TournamentSelection(2, True, 3, 1),
                                           mutation=H.Mutations(0.5, 0, 0.2, 0.5, 0, 0, rand_seed=0, device="cuda"), wb=False, verbose=False)
print("RESULT " + json.dumps({"pop": len(pop), "generations": len(fits), "steps": [int(a.steps[-1]) for a in pop],
                              "types": sorted({type(a).__module__ for a in pop}), "calls": calls, "memory_len": len(memory),
                              "counter": memory.counter, "muts": [str(a.mut) for a in pop], "fitness_len": [len(a.fitness) for a in pop],
                              "scores": [len(a.scores) for a in pop]}))
