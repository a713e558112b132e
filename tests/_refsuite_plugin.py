"""pytest plugin used by tests/test_reference_suite_cpu.py: makes the REFERENCE's OWN unit tests (run in place from
/root/reference/tests, unmodified) exercise THIS package's classes.  On import: oracle.refshim (the reference importable,
stand-ins for its missing third-party dependencies), Python stand-ins for the C entry points those tests reach (no GPU
here: bytes movers, the n-step fold, and the priority trees through the oracle's C segment tree operating on the buffers
our classes own), then ``agilerl_b200.install()`` so ``from agilerl.components... import ...`` binds our classes."""
import ctypes
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)
os.environ.setdefault("B2RL_GRAPH", "0")

from oracle import refshim  # noqa: E402

if refshim.available():           # the reference's own tests import it; the stand-ins below do not need it
    refshim.install()
import agilerl_b200  # noqa: E402
from agilerl_b200 import _lib  # noqa: E402
from agilerl_b200.components import replay_buffer as rb  # noqa: E402
from oracle.segtree import load_lib as _oracle_tree  # noqa: E402
from test_multi_agent_host_cpu import StandIn, _bytes, _f32, _i64  # noqa: E402

OT = _oracle_tree()


def _f64(ptr, n):
    return np.ctypeslib.as_array((ctypes.c_double * n).from_address(ptr))


class Lib(StandIn):
    def b2rl_ring_write(self, dst, src, row_bytes, start, n, max_size, stream):
        return self.b2rl_ring_write_multi(1, [dst], [src], [row_bytes], start, n, max_size, stream)

    def b2rl_gather_rows(self, dst, src, idx, row_bytes, n, stream):
        return self.b2rl_gather_rows_multi(1, [dst], [src], [row_bytes], idx, n, stream)

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

    def b2rl_tree_init(self, s, m, cap, stream):
        OT.ost_init(s, cap, 0); OT.ost_init(m, cap, 1)
        return 0

    def b2rl_tree_set(self, s, m, cap, idx, pa, n, stream):
        for i, x in zip(_i64(idx, n), _f64(pa, n)):
            if s:
                OT.ost_set(s, cap, 0, int(i), float(x))
            if m:
                OT.ost_set(m, cap, 1, int(i), float(x))
        return 0

    def b2rl_tree_set_range(self, s, m, cap, tree_ptr, n, max_size, p_alpha, stream):
        for k in range(n):
            i = (tree_ptr + k) % max_size
            OT.ost_set(s, cap, 0, i, p_alpha); OT.ost_set(m, cap, 1, i, p_alpha)
        return 0

    def b2rl_tree_retrieve(self, s, cap, ub, n, out, stream):
        u, o = _f64(ub, n), _i64(out, n)
        for k in range(n):
            o[k] = OT.ost_retrieve(s, cap, float(u[k]))
        return 0

    def b2rl_per_sample(self, s, m, cap, u, B, beta, size, idx_out, w_out, stream):
        OT.oper_sample(s, cap, u, B, idx_out)
        if w_out:
            OT.oper_weights(s, m, cap, idx_out, B, beta, size, w_out)
        return 0

    def b2rl_host_priority_pow(self, pri, n, alpha, floor_, out, mx):
        p = np.maximum(_f32(pri, n).astype(np.float64), floor_)
        _f64(out, n)[:] = [float(x) ** alpha for x in p]
        mx._obj.value = max(mx._obj.value, float(p.max()))
        return 0


    # construction of the value-based agents only asks for the size of their noise vector
    def b2rl_noise_count(self, desc, out):
        d = desc._obj
        out._obj.value = sum(layers[i].in_c + layers[i].out_c for layers, cnt in ((d.enc, d.n_enc), (d.val, d.n_val), (d.adv, d.n_adv))
                             for i in range(cnt) if layers[i].noisy)
        return 0


    def _noop(self, *a):
        return 0
    b2rl_noise_reset_philox = b2rl_noise_reset_from_normals = _noop          # fresh noise at construction / clone


class _Event:
    def record(self, *a): pass
    def synchronize(self): pass
    def wait(self, *a): pass
    def query(self): return True


_lib.as_device = lambda d: torch.device("cpu")
_lib.load = lambda require_cuda=False, _l=Lib(): _l
_lib.stream_ptr = lambda d=None: 0
_lib.check = lambda rc: None
_lib.require_cuda_tensor = lambda t, what="tensor": None
torch.Tensor.pin_memory = lambda self: self
torch.cuda.Event = _Event
rb._PinnedRing.sent = lambda self, k, dev: None
agilerl_b200.install(include_driver=False)

# tests/test_hpo/test_tournament.py imports a helper of the LLM tests at module level (transformers / peft / accelerate): an
# inert stand-in keeps the file importable; the LLM cases themselves are outside this package and fail as expected
import types  # noqa: E402

_grpo = types.ModuleType("tests.test_algorithms.test_llms.test_grpo")
_grpo.create_module = lambda *a, **k: None
sys.modules.setdefault("tests.test_algorithms.test_llms.test_grpo", _grpo)


# ---- the learners' entry points, for the reference's ALGORITHM tests (construct / act / learn / clone / test loop): the
# ---- forwards return deterministic pseudo values that depend on the first parameter, the learn calls MOVE the parameter
# ---- buffers (and soft-update the targets), so "learning changed the weights" / "the clone is a deep copy" assertions see
# ---- what they would on the device.  Numerics are the GPU tests' business.
_cls = type(_lib.load())


def _obs_rows(d, obs, rows):
    x = _bytes(obs, rows * d.obs_elems) if d.obs_u8 else _f32(obs, rows * d.obs_elems)
    return x.reshape(rows, d.obs_elems)[:, :16].astype(np.float64).sum(axis=1, keepdims=True)

def net_workspace_bytes(self, desc, rows, backward, out):
    out._obj.value = 256; return 0
def forward_q(self, desc, params, eps, use_noise, support, obs, row_idx, rows, q_out, argmax_out, ws, wsb, stream):
    d = desc._obj
    q = _f32(q_out, rows * d.n_actions).reshape(rows, d.n_actions)
    q[:] = np.sin(_obs_rows(d, obs, rows) * (np.arange(d.n_actions) + 1.0) + float(_f32(params, 1)[0]))
    if argmax_out: _i64(argmax_out, rows)[:] = q.argmax(axis=1)
    return 0
def forward_dist(self, desc, params, eps, use_noise, support, obs, rows, log_probs, dist_out, ws, wsb, stream):
    d = desc._obj
    out = _f32(dist_out, rows * d.n_actions * d.n_atoms)
    out[:] = np.log(1.0 / d.n_atoms) if log_probs else 1.0 / d.n_atoms
    return 0
def rainbow_loss(self, desc, cfg, bufs, stream):
    c, b = cfg._obj, bufs._obj
    B = c.batch
    if b.priorities:
        pr = _f32(b.priorities, B)
        if not c.accumulate: pr[:] = 0
        pr += np.float32(0.5 + c.prior_eps)
    if b.loss_elem: _f32(b.loss_elem, B)[:] = 0.5
    if b.loss_scalar: _f32(b.loss_scalar, 1)[0] = 0.5
    return 0
def optim_step(self, desc, cfg, bufs, stream):
    d, c, b = desc._obj, cfg._obj, bufs._obj
    p, t = _f32(b.actor_params, d.n_params), _f32(b.target_params, d.n_params)
    p += 0.01
    t[:] = c.tau * p + (1 - c.tau) * t
    return 0
def dqn_learn(self, desc, cfg, bufs, stream):
    optim_step(self, desc, cfg, bufs, stream)
    _f32(bufs._obj.loss_scalar, 1)[0] = 0.25
    return 0
def ok(self, *a): return 0
def actor_ws(self, desc, rows, out): out._obj.value = 256; return 0
def ddpg_ws(self, a, c, B, out): out._obj.value = 256; return 0
def actor_forward(self, desc, params, obs, rows, out, ws, wsb, stream):
    d = desc._obj; a = d.val[d.n_val - 1].out_c
    x = _f32(obs, rows * d.obs_elems).reshape(rows, d.obs_elems)
    _f32(out, rows * a).reshape(rows, a)[:] = np.tanh(x.sum(axis=1, keepdims=True) * (np.arange(a) + 1.0) * 0.1 + float(_f32(params, 1)[0]))
    return 0
def ddpg_learn(self, actor, critic, cfg, bufs, stream):
    c, b = cfg._obj, bufs._obj
    na, nc = actor._obj.n_params, critic._obj.n_params
    for i in range(2 if c.twin else 1):
        p, t = _f32(b.critic[i], nc), _f32(b.critic_target[i], nc)
        p += 0.01
        if c.policy_update: t[:] = c.tau * p + (1 - c.tau) * t
    if c.policy_update:
        p, t = _f32(b.actor, na), _f32(b.actor_target, na)
        p += 0.01; t[:] = c.tau * p + (1 - c.tau) * t
        _f32(b.actor_loss, 1)[0] = -0.5
    _f32(b.critic_loss, 1)[0] = 0.5
    return 0
def maddpg_ws(self, actors, critics, n, B, out): out._obj.value = 256; return 0
def maddpg_learn(self, actors, critics, cfg, bufs, stream):
    c, b = cfg._obj, bufs._obj
    ap = ctypes.cast(actors, ctypes.POINTER(ctypes.POINTER(_lib.NetDesc)))
    cp = ctypes.cast(critics, ctypes.POINTER(ctypes.POINTER(_lib.NetDesc)))
    for i in range(c.n_agents):
        for ptr, tgt, n in ((b.actor[i], b.actor_target[i], ap[i].contents.n_params), (b.critic[i], b.critic_target[i], cp[i].contents.n_params)):
            p, t = _f32(ptr, n), _f32(tgt, n)
            p += 0.01
            t[:] = c.tau * p + (1 - c.tau) * t
    _f32(b.losses, 2 * c.n_agents)[:] = 0.5
    return 0
for name, fn in dict(b2rl_maddpg_workspace_bytes=maddpg_ws, b2rl_maddpg_learn=maddpg_learn, b2rl_net_workspace_bytes=net_workspace_bytes, b2rl_net_forward_q=forward_q, b2rl_net_forward_dist=forward_dist,
                     b2rl_rainbow_loss=rainbow_loss, b2rl_rainbow_backward=ok, b2rl_optim_step=optim_step, b2rl_dqn_learn=dqn_learn,
                     b2rl_noise_reset_state=ok, b2rl_noise_reset_state_pair=ok, b2rl_actor_workspace_bytes=actor_ws,
                     b2rl_ddpg_workspace_bytes=ddpg_ws, b2rl_actor_forward=actor_forward, b2rl_ddpg_learn=ddpg_learn).items():
    setattr(_cls, name, fn)
