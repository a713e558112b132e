"""Helper of tests/test_reference_driver_cpu.py (own process): the UNCHANGED reference driver drives THIS package's classes
on the NORTH-STAR flow — Rainbow DQN with prioritized replay and 3-step returns, image observations
(train_off_policy.py:327-412: ``Transition`` -> ``n_step_memory.add`` -> ``memory.add``; ``sampler.sample(B, beta)`` ->
``n_step_sampler.sample(idxs)`` -> ``agent.learn(experiences, n_experiences, per=True)`` -> ``memory.update_priorities``).

Stand-ins for the C entry points, all host-side: bytes movers; the n-step fold / select / fused ingest restated in numpy
(quirk Q3); the priority trees through the oracle's C segment tree operating directly on the buffers our classes own
(so the PER arithmetic of the run is real: sampled indices, weights and updated leaves are checked for consistency);
network forward / learn calls return deterministic pseudo values and count.  Call-level drop-in evidence, not numerics."""
import ctypes
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
os.environ["B2RL_GRAPH"] = "0"                         # eager API path: graph capture needs the real library

from oracle import refshim  # noqa: E402

REFERENCE = "--without-reference" not in sys.argv     # tests/_driver_equivalence_standin.py: our driver alone
if REFERENCE:
    refshim.install()
import agilerl_b200  # noqa: E402
from agilerl_b200 import _lib  # noqa: E402
from agilerl_b200.components import replay_buffer as rb  # noqa: E402
from oracle.segtree import load_lib as oracle_tree  # noqa: E402
from test_multi_agent_host_cpu import StandIn, _bytes, _f32, _i64  # noqa: E402

OT = oracle_tree()
calls = {"loss": 0, "backward": 0, "optim": 0, "noise_resets": 0, "forward_rows": 0, "ingest": 0, "per_sample": 0, "tree_set": 0,
         "tree_set_range": 0}
checks = {"weights_in_0_1": True, "idx_in_range": True, "tree_sum_positive": True}


def _f64(ptr, n):
    return np.ctypeslib.as_array((ctypes.c_double * n).from_address(ptr))


class Lib(StandIn):
    def b2rl_ring_write(self, dst, src, row_bytes, start, n, max_size, stream):
        return self.b2rl_ring_write_multi(1, [dst], [src], [row_bytes], start, n, max_size, stream)

    def b2rl_gather_rows(self, dst, src, idx, row_bytes, n, stream):
        return self.b2rl_gather_rows_multi(1, [dst], [src], [row_bytes], idx, n, stream)

    # ---- n-step (replay_buffer.py:206-258, quirk Q3) ----------------------------------------------------------
    @staticmethod
    def _stop(done_steps, n, E):
        last = 0
        for k in range(1, n):
            last = k
            if np.any(_f32(done_steps[k], E) != 0):
                break
        return last

    def b2rl_nstep_fold(self, reward_steps, done_steps, n, E, gamma, reward_out, last_out, stream):
        last = self._stop(done_steps, n, E)
        r = _f32(reward_steps[0], E).copy()
        for k in range(1, last + 1):
            r += _f32(reward_steps[k], E) * np.float32(gamma ** k)
        _f32(reward_out, E)[:] = r
        np.ctypeslib.as_array((ctypes.c_int32 * 1).from_address(last_out))[0] = last
        return 0

    def b2rl_select_copy(self, dst, srcs, n, which, nbytes, stream):
        k = int(np.ctypeslib.as_array((ctypes.c_int32 * 1).from_address(which))[0])
        _bytes(dst, nbytes)[:] = _bytes(srcs[k], nbytes)
        return 0

    def b2rl_nstep_ingest(self, nf, ring, src, row_bytes, role, rew, don, n, E, gamma, cursor, max_size, stream):
        calls["ingest"] += 1
        last = self._stop(don, n, E)
        for f in range(nf):
            rbs = row_bytes[f]
            d = _bytes(ring[f], rbs * max_size)
            if role[f] == 2:
                r = _f32(rew[0], E).copy()
                for k in range(1, last + 1):
                    r += _f32(rew[k], E) * np.float32(gamma ** k)
                rows = r.view(np.uint8).reshape(E, 4)
            else:
                rows = _bytes(src[f * n + (last if role[f] == 1 else 0)], rbs * E).reshape(E, rbs)
            for e in range(E):
                slot = (cursor + e) % max_size
                d[slot * rbs:(slot + 1) * rbs] = rows[e]
        return 0

    # ---- priority trees: the oracle's C segment tree on OUR buffers ---------------------------------------------
    def b2rl_tree_init(self, s, m, cap, stream):
        OT.ost_init(s, cap, 0); OT.ost_init(m, cap, 1)
        return 0

    def b2rl_tree_set(self, s, m, cap, idx, pa, n, stream):
        calls["tree_set"] += 1
        ix, v = _i64(idx, n), _f64(pa, n)
        for i, x in zip(ix, v):
            if s:
                OT.ost_set(s, cap, 0, int(i), float(x))
            if m:
                OT.ost_set(m, cap, 1, int(i), float(x))
        return 0

    def b2rl_tree_set_range(self, s, m, cap, tree_ptr, n, max_size, p_alpha, stream):
        calls["tree_set_range"] += 1
        for k in range(n):
            i = (tree_ptr + k) % max_size
            OT.ost_set(s, cap, 0, i, p_alpha); OT.ost_set(m, cap, 1, i, p_alpha)
        return 0

    def b2rl_per_sample(self, s, m, cap, u, B, beta, size, idx_out, w_out, stream):
        calls["per_sample"] += 1
        OT.oper_sample(s, cap, u, B, idx_out)
        ix = _i64(idx_out, B)
        checks["idx_in_range"] &= bool(((ix >= 0) & (ix < size)).all())
        checks["tree_sum_positive"] &= bool(_f64(s, 2 * cap)[1] > 0)
        if w_out:
            OT.oper_weights(s, m, cap, idx_out, B, beta, size, w_out)
            w = _f32(w_out, B)
            checks["weights_in_0_1"] &= bool(((w > 0) & (w <= 1.0 + 1e-6)).all())
        return 0

    def b2rl_host_priority_pow(self, pri, n, alpha, floor_, out, mx):
        p = np.maximum(_f32(pri, n).astype(np.float64), floor_)
        _f64(out, n)[:] = [float(x) ** alpha for x in p]
        mx._obj.value = max(mx._obj.value, float(p.max()))
        return 0

    # ---- networks ---------------------------------------------------------------------------------------------
    def b2rl_noise_count(self, desc, out):
        out._obj.value = 64
        return 0

    def b2rl_net_workspace_bytes(self, desc, rows, backward, out):
        out._obj.value = 256
        return 0

    def b2rl_net_forward_q(self, desc, params, eps, use_noise, support, obs, row_idx, rows, q_out, argmax_out, ws, wsb, stream):
        d = desc._obj
        x = (_bytes(obs, rows * d.obs_elems) if d.obs_u8 else _f32(obs, rows * d.obs_elems)).reshape(rows, d.obs_elems)
        q = _f32(q_out, rows * d.n_actions).reshape(rows, d.n_actions)
        q[:] = np.sin(x[:, :16].astype(np.float64).sum(axis=1, keepdims=True) * (np.arange(d.n_actions) + 1.0))
        if argmax_out:
            _i64(argmax_out, rows)[:] = q.argmax(axis=1)
        calls["forward_rows"] += rows
        return 0

    def b2rl_rainbow_loss(self, desc, cfg, bufs, stream):
        c, b = cfg._obj, bufs._obj
        B = c.batch
        assert b.weights and c.weights_mode in (1, 2) and b.obs and b.next_obs and b.action and b.reward and b.done
        w = _f32(b.weights, B)
        assert np.isfinite(w).all() and np.isfinite(_f32(b.reward, B)).all()
        if not c.accumulate:
            _f32(b.priorities, B)[:] = 0.0
        _f32(b.priorities, B)[:] += 0.5 + 0.01 * np.arange(B, dtype=np.float32) + np.float32(c.prior_eps)
        _f32(b.loss_scalar, 1)[0] = 1.0 + 0.001 * calls["loss"]
        calls["loss"] += 1
        return 0

    def b2rl_rainbow_backward(self, desc, cfg, bufs, stream):
        calls["backward"] += 1
        return 0

    def b2rl_optim_step(self, desc, cfg, bufs, stream):
        calls["optim"] += 1
        return 0

    def _noise(self, *a):
        calls["noise_resets"] += 1
        return 0
    b2rl_noise_reset_philox = b2rl_noise_reset_from_normals = _noise


class _Event:
    def record(self, *a): pass
    def synchronize(self): pass
    def wait(self, *a): pass
    def query(self): return True


lib = Lib()
_lib.as_device = lambda d: torch.device("cpu")
_lib.load = lambda require_cuda=False: lib
_lib.stream_ptr = lambda d=None: 0
_lib.check = lambda rc: None
_lib.require_cuda_tensor = lambda t, what="tensor": None
torch.Tensor.pin_memory = lambda self: self
torch.cuda.Event = _Event
rb._PinnedRing.sent = lambda self, k, dev: None

agilerl_b200.install(include_driver=False)
import agilerl_b200.algorithms as A  # noqa: E402
import agilerl_b200.components as C  # noqa: E402
import agilerl_b200.hpo as H  # noqa: E402

if REFERENCE:
    import inspect

    import agilerl.training.train_off_policy as T

    assert inspect.getsourcefile(T).startswith(refshim.REFERENCE_ROOT), inspect.getsourcefile(T)
    assert T.RainbowDQN is A.RainbowDQN and T.PrioritizedReplayBuffer is C.PrioritizedReplayBuffer
    assert T.MultiStepReplayBuffer is C.MultiStepReplayBuffer and T.Sampler is C.Sampler
from agilerl_b200.compat import spaces  # noqa: E402
from agilerl_b200.utils.utils import create_population  # noqa: E402


class VecEnv:
    def __init__(self, num_envs=2, seed=0):
        self.num_envs, self.rng, self.t = num_envs, np.random.default_rng(seed), 0

    def _obs(self):
        return self.rng.integers(0, 256, (self.num_envs, 3, 20, 20), dtype=np.uint8)

    def reset(self):
        self.t = 0
        return self._obs(), {}

    def step(self, action):
        assert np.asarray(action).shape == (self.num_envs,), np.asarray(action).shape
        self.t += 1
        return (self._obs(), self.rng.standard_normal(self.num_envs), np.array([self.t % 7 == 0] * self.num_envs),
                np.zeros(self.num_envs, bool), {})


NET = {"encoder_config": {"channel_size": [8, 16], "kernel_size": [4, 3], "stride_size": [2, 1]},
       "head_config": {"hidden_size": [32]}, "latent_dim": 16}
obs_space, act_space = spaces.Box(0, 255, (3, 20, 20), np.uint8), spaces.Discrete(4)
INIT_HP = {"BATCH_SIZE": 8, "LEARN_STEP": 2, "V_MIN": -10.0, "V_MAX": 10.0, "N_STEP": 3}
pop = create_population("Rainbow DQN", obs_space, act_space, dict(NET), INIT_HP, population_size=2)
memory = C.PrioritizedReplayBuffer(256, 0.6, device="cuda")
n_step_memory = C.MultiStepReplayBuffer(256, 3, 0.99, device="cuda")
beta0 = [a.beta for a in pop]
pop, fits = T.train_off_policy(VecEnv(), "synthetic", "Rainbow DQN", pop, memory, INIT_HP=INIT_HP, MUT_P={}, max_steps=80,
                               evo_steps=40, eval_steps=10, eval_loop=1, n_step=True, per=True, n_step_memory=n_step_memory,
                               tournament=H.TournamentSelection(2, True, 2, 1),
                               mutation=H.Mutations(0.6, 0, 0.2, 0.4, 0, 0, rand_seed=0, device="cuda"), wb=False, verbose=False)
leaves = _f64(memory.sum_tree.data_ptr, 2 * memory._cap)[memory._cap:memory._cap + len(memory)]
print("RESULT " + json.dumps({"pop": len(pop), "generations": len(fits), "steps": [int(a.steps[-1]) for a in pop],
                              "types": sorted({type(a).__module__ for a in pop}), "calls": calls, "checks": checks,
                              "per_len": len(memory), "nstep_len": len(n_step_memory), "beta_grew": [a.beta > b for a, b in zip(pop, beta0)],
                              "max_priority": memory.max_priority, "distinct_leaves": int(len(set(np.round(leaves, 12)))),
                              "tree_ptr": memory.tree_ptr}))
