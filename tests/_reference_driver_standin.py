"""Helper of tests/test_reference_driver_cpu.py (run as a script in its own process): the UNCHANGED reference driver
``/root/reference/agilerl/training/train_off_policy.py`` drives THIS package's classes, bound under the ``agilerl.*`` names
by ``agilerl_b200.install()``, on BASELINE configs[0] (DQN, pop = 4, vector environment).

No GPU here, so the C entry points the run reaches are Python stand-ins: the data movers copy bytes, the network forward
returns deterministic pseudo Q-values, the learn call only counts and reports a loss.  What the run therefore proves is the
drop-in claim at the call level — every method, argument convention, attribute and return type the reference's loop relies
on (acting with epsilon and masks, ``Transition`` -> ``memory.add``, ``Sampler`` dispatch, ``agent.learn``, ``agent.test``,
``tournament_selection_and_mutation`` from the reference's own ``utils``) is served by our classes.  Numerics are the GPU
tests' business."""
import ctypes
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import refshim  # noqa: E402

REFERENCE = "--without-reference" not in sys.argv     # tests/_driver_equivalence_standin.py: our driver alone
if REFERENCE:
    refshim.install()
import agilerl_b200  # noqa: E402
from agilerl_b200 import _lib  # noqa: E402
from agilerl_b200.components import replay_buffer as rb  # noqa: E402
from test_multi_agent_host_cpu import StandIn, _f32  # noqa: E402

ALGO = sys.argv[1] if len(sys.argv) > 1 else "DQN"      # "DQN" (configs[0]) or "TD3" (the driver's deterministic-policy branch)
calls = {"learn": 0, "forward_rows": 0, "adds": 0, "policy_updates": 0}


class Lib(StandIn):
    def b2rl_ring_write(self, dst, src, row_bytes, start, n, max_size, stream):
        return self.b2rl_ring_write_multi(1, [dst], [src], [row_bytes], start, n, max_size, stream)

    def b2rl_gather_rows(self, dst, src, idx, row_bytes, n, stream):
        return self.b2rl_gather_rows_multi(1, [dst], [src], [row_bytes], idx, n, stream)

    def b2rl_noise_count(self, desc, out):
        out._obj.value = 0
        return 0

    def b2rl_net_workspace_bytes(self, desc, rows, backward, out):
        out._obj.value = 256
        return 0

    def b2rl_net_forward_q(self, desc, params, eps, use_noise, support, obs, row_idx, rows, q_out, argmax_out, ws, wsb, stream):
        d = desc._obj
        n_act, elems = d.n_actions, d.obs_elems
        x = _f32(obs, rows * elems).reshape(rows, elems)
        q = _f32(q_out, rows * n_act).reshape(rows, n_act)
        q[:] = np.sin(x.sum(axis=1, keepdims=True) * (np.arange(n_act) + 1.0))
        calls["forward_rows"] += rows
        return 0

    def b2rl_dqn_learn(self, desc, cfg, bufs, stream):
        b = bufs._obj
        _f32(b.loss_scalar, 1)[0] = 0.25 + 0.001 * calls["learn"]
        calls["learn"] += 1
        return 0


    # ---- TD3 / DDPG: actor forward and the fused learn call ------------------------------------------------------
    def b2rl_actor_workspace_bytes(self, desc, rows, out):
        out._obj.value = 256
        return 0

    def b2rl_ddpg_workspace_bytes(self, actor, critic, batch, out):
        out._obj.value = 256
        return 0

    def b2rl_actor_forward(self, desc, params, obs, rows, out, ws, wsb, stream):
        d = desc._obj
        a = d.val[d.n_val - 1].out_c
        x = _f32(obs, rows * d.obs_elems).reshape(rows, d.obs_elems)
        _f32(out, rows * a).reshape(rows, a)[:] = np.tanh(x.sum(axis=1, keepdims=True) * (np.arange(a) + 1.0) * 0.1)
        calls["forward_rows"] += rows
        return 0

    def b2rl_ddpg_learn(self, actor, critic, cfg, bufs, stream):
        c, b = cfg._obj, bufs._obj
        B, A = c.batch, actor._obj.val[actor._obj.n_val - 1].out_c
        assert c.twin == 1 and np.isfinite(_f32(b.action, B * A)).all() and np.isfinite(_f32(b.reward, B)).all()
        _f32(b.action, B * A)[:] = 0.125                         # the kept quirk: the batch's action tensor receives the noise
        _f32(b.critic_loss, 1)[0] = 0.5
        if c.policy_update:
            _f32(b.actor_loss, 1)[0] = -0.25
            calls["policy_updates"] += 1
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

    import agilerl.training.train_off_policy as T

    assert inspect.getsourcefile(T).startswith(refshim.REFERENCE_ROOT), inspect.getsourcefile(T)
    assert T.DQN is A.DQN and T.TD3 is A.TD3 and T.ReplayBuffer is C.ReplayBuffer and T.Sampler is C.Sampler and T.Mutations is H.Mutations
from agilerl_b200.compat import spaces  # noqa: E402
from agilerl_b200.utils.utils import create_population  # noqa: E402


class VecEnv:
    def __init__(self, num_envs=2, seed=0):
        self.num_envs, self.rng, self.t = num_envs, np.random.default_rng(seed), 0

    def _obs(self):
        return self.rng.standard_normal((self.num_envs, 4)).astype(np.float32)

    def reset(self):
        self.t = 0
        return self._obs(), {}

    def step(self, action):
        want = (self.num_envs,) if ALGO == "DQN" else (self.num_envs, 3)
        assert np.asarray(action).shape == want, np.asarray(action).shape
        if ALGO != "DQN":
            assert np.all(np.abs(action) <= 2.0 + 1e-6)           # rescaled to the action bounds [-2, 2] by the driver
        self.t += 1
        return (self._obs(), self.rng.standard_normal(self.num_envs), np.array([self.t % 7 == 0] * self.num_envs),
                np.zeros(self.num_envs, bool), {})


obs_space = spaces.Box(-1, 1, (4,), np.float32)
act_space = spaces.Discrete(2) if ALGO == "DQN" else spaces.Box(-2.0, 2.0, (3,), np.float32)
INIT_HP = {"BATCH_SIZE": 16, "LEARN_STEP": 2, "DOUBLE": True, "POLICY_FREQ": 2}
pop = create_population(ALGO, obs_space, act_space, None, INIT_HP, population_size=4, num_envs=2)
memory = C.ReplayBuffer(512, device="cuda")
orig_add = memory.add


def counting_add(data):
    calls["adds"] += 1
    return orig_add(data)


memory.add = counting_add
import glob  # noqa: E402
import tempfile  # noqa: E402

ckpt_dir = tempfile.mkdtemp()
pop, fits = T.train_off_policy(VecEnv(), "synthetic", ALGO, pop, memory, INIT_HP=INIT_HP, MUT_P={}, max_steps=120, evo_steps=40,
                               eval_steps=10, eval_loop=1, tournament=H.TournamentSelection(2, True, 4, 1),
                               mutation=H.Mutations(0.5, 0, 0.2, 0.25, 0, 0.25, rand_seed=0, device="cuda"), wb=False, verbose=False,
                               checkpoint=40, checkpoint_path=os.path.join(ckpt_dir, "pop.pt"), overwrite_checkpoints=True,
                               save_elite=True, elite_path=os.path.join(ckpt_dir, "elite.pt"))
ckpts = sorted(os.path.basename(f) for f in glob.glob(os.path.join(ckpt_dir, "*")))
restored = None
if ALGO == "DQN":                      # the population checkpoints the reference's utils wrote load back into our agents
    f = [c for c in ckpts if c.startswith("pop")][0]
    before = pop[0].actor.state_dict()
    twin = pop[0].clone()
    twin.actor.buffers.params.zero_()
    twin.load_checkpoint(os.path.join(ckpt_dir, f))
    restored = bool(twin.actor.buffers.params.abs().sum() > 0)
print("RESULT " + json.dumps({"pop": len(pop), "generations": len(fits), "fit_width": [len(f) for f in fits],
                              "steps": [int(a.steps[-1]) for a in pop], "types": sorted({type(a).__module__ for a in pop}),
                              "calls": calls, "memory_len": len(memory), "muts": [str(a.mut) for a in pop],
                              "fitness_len": [len(a.fitness) for a in pop], "checkpoints": ckpts, "restored": restored}))
