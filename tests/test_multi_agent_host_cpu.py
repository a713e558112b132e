"""CPU: the HOST side of the multi-agent path (SURVEY 8f-4) with Python stand-ins for the C-ABI entry points it calls
(test-only: the product has no CPU path and raises without CUDA — tests/test_abi_cpu.py).  The stand-ins move bytes
(``b2rl_ring_write_multi`` / ``b2rl_gather_rows_multi``), apply the mutation rule slot by slot (``b2rl_gaussian_mutate``)
or record what they were handed (``b2rl_maddpg_learn``), which pins everything the host decides:

* ``MultiAgentReplayBuffer``: field packing (agents side by side), staging offsets, ring cursor / deque-head mapping,
  ``random.sample`` positions -> slots, binary-field casting, NaN passthrough — against the reference's golden samples;
* ``MADDPG.learn``: the [B, sum] matrices (reward / done as [B, n_agents]), every network / optimiser pointer,
  Adam bias corrections, the layer tables of actors and critics;
* ``Mutations._gaussian_parameter_mutation_device``: keys / rows / columns / branches drawn like the reference, the
  last-writer mask of duplicate positions."""
import ctypes
import warnings
import random

import numpy as np
import pytest
import torch

from conftest import load_golden

FIELDS = ("obs", "action", "reward", "next_obs", "done")


def _bytes(ptr, n):
    return np.ctypeslib.as_array((ctypes.c_uint8 * n).from_address(ptr))


def _f32(ptr, n):
    return np.ctypeslib.as_array((ctypes.c_float * n).from_address(ptr))


def _i64(ptr, n):
    return np.ctypeslib.as_array((ctypes.c_int64 * n).from_address(ptr))


class StandIn:
    def __init__(self):
        self.seen = {}

    def b2rl_ring_write_multi(self, nf, dst, src, row_bytes, start, n, max_size, stream):
        for f in range(nf):
            rb = row_bytes[f]
            d, s = _bytes(dst[f], rb * max_size), _bytes(src[f], rb * n)
            for r in range(n):
                slot = (start + r) % max_size
                d[slot * rb:(slot + 1) * rb] = s[r * rb:(r + 1) * rb]
        return 0

    def b2rl_gather_rows_multi(self, nf, dst, src, row_bytes, idx, n, stream):
        ix = _i64(idx, n)
        for f in range(nf):
            rb = row_bytes[f]
            d = _bytes(dst[f], rb * n)
            for r in range(n):
                d[r * rb:(r + 1) * rb] = _bytes(src[f] + int(ix[r]) * rb, rb)
        return 0

    def b2rl_gaussian_mutate(self, W, nr, nc, rows, cols, u, keep, z, seed, off, sd, n, stream):
        Wv, orig = _f32(W, nr * nc), _f32(W, nr * nc).copy()
        r, c, uu, kk, zz = _i64(rows, n), _i64(cols, n), _f32(u, n), _bytes(keep, n), _f32(z, n)
        for j in range(n):
            if not kk[j]:
                continue
            w = np.float32(orig[r[j] * nc + c[j]])
            if uu[j] < np.float32(0.05):
                v = w + abs(np.float32(10) * w) * zz[j]
            elif uu[j] < np.float32(0.1):
                v = zz[j]
            else:
                v = w + abs(np.float32(sd) * w) * zz[j]
            Wv[r[j] * nc + c[j]] = np.clip(np.float32(v), -1e6, 1e6)
        return 0

    def b2rl_maddpg_workspace_bytes(self, actors, critics, n, B, out):
        out._obj.value = 4096
        return 0

    def b2rl_maddpg_learn(self, actors, critics, cfg, bufs, stream):
        from agilerl_b200 import _lib
        cfg, bufs = cfg._obj, bufs._obj
        B, n = cfg.batch, cfg.n_agents
        ap = ctypes.cast(actors, ctypes.POINTER(ctypes.POINTER(_lib.NetDesc)))
        cp = ctypes.cast(critics, ctypes.POINTER(ctypes.POINTER(_lib.NetDesc)))
        SO = sum(ap[i].contents.enc[0].in_c for i in range(n))
        SA = sum(ap[i].contents.val[ap[i].contents.n_val - 1].out_c for i in range(n))
        s = self.seen
        s["cfg"] = {f[0]: getattr(cfg, f[0]) for f in cfg._fields_}
        s["actor_layers"] = [[(l.in_c, l.out_c, l.ln, l.act) for l in list(ap[i].contents.enc)[:ap[i].contents.n_enc] +
                              list(ap[i].contents.val)[:ap[i].contents.n_val]] for i in range(n)]
        s["critic_layers"] = [[(l.in_c, l.out_c, l.ln, l.act) for l in list(cp[i].contents.enc)[:cp[i].contents.n_enc] +
                               list(cp[i].contents.val)[:cp[i].contents.n_val]] for i in range(n)]
        s["obs"], s["next_obs"] = _f32(bufs.obs, B * SO).reshape(B, SO).copy(), _f32(bufs.next_obs, B * SO).reshape(B, SO).copy()
        s["act"] = _f32(bufs.action, B * SA).reshape(B, SA).copy()
        s["rew"], s["done"] = _f32(bufs.reward, n * B).reshape(B, n).copy(), _f32(bufs.done, n * B).reshape(B, n).copy()
        s["step_state"] = bufs.step_state
        s["ptrs"] = [{k: getattr(bufs, k)[i] for k in ("actor", "actor_target", "actor_grads", "actor_m", "actor_v", "critic",
                                                        "critic_target", "critic_grads", "critic_m", "critic_v")} for i in range(n)]
        _f32(bufs.losses, 2 * n)[:] = np.arange(2 * n)
        return 0


@pytest.fixture
def standin(monkeypatch):
    from agilerl_b200 import _lib
    from agilerl_b200.components import replay_buffer as rb
    lib = StandIn()
    monkeypatch.setattr(_lib, "as_device", lambda d: torch.device("cpu"))
    monkeypatch.setattr(_lib, "load", lambda require_cuda=False: lib)
    monkeypatch.setattr(_lib, "stream_ptr", lambda d=None: 0)
    monkeypatch.setattr(_lib, "check", lambda rc: None)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self: self)
    monkeypatch.setattr(rb._PinnedRing, "sent", lambda self, k, dev: None)
    return lib


def _sd(g, tag):
    return {k[len(tag) + 1:]: torch.from_numpy(g[k].copy()) for k in g.files if k.startswith(tag + "/")}


def test_replay_host_logic_reproduces_reference_samples(standin):
    from agilerl_b200.components import MultiAgentReplayBuffer
    g = load_golden("ma_replay.npz")
    ids, fields = [str(a) for a in g["agent_ids"]], [str(f) for f in g["fields"]]
    buf = MultiAgentReplayBuffer(int(g["cap"]), fields, ids, device="cuda")
    for t in range(int(g["n_steps"])):
        buf.save_to_memory(*[{a: g[f"t{t}_{f}/{a}"] for a in ids} for f in fields], is_vectorised=bool(int(g[f"t{t}_vect"])))
    assert len(buf) == int(g["final_len"]) and buf.counter == int(g["final_counter"])
    for c in range(int(g["n_samples"])):
        random.seed(int(g[f"sample{c}_seed"]))
        batch = buf.sample(int(g[f"sample{c}_B"]))
        for f, d in zip(fields, batch):
            assert d.packed.shape[0] == int(g[f"sample{c}_B"])
            for a in ids:
                np.testing.assert_array_equal(d[a].numpy(), g[f"sample{c}_{f}/{a}"], err_msg=f"{c} {f} {a}")


def test_maddpg_learn_marshalling(standin):
    from agilerl_b200.algorithms import MADDPG
    from agilerl_b200.compat import spaces
    from agilerl_b200.components import MultiAgentReplayBuffer
    g = load_golden("maddpg_vector.npz")
    ids = [str(a) for a in g["agent_ids"]]
    agent = MADDPG([spaces.Box(-1.0, 1.0, (int(d),), np.float32) for d in g["obs_dims"]],
                   [spaces.Box(-1.0, 1.0, (int(d),), np.float32) for d in g["act_dims"]], agent_ids=ids, batch_size=int(g["B"]))
    agent.use_graph = False                      # the eager call: graph capture needs the real library
    a0 = ids[0]
    assert list(agent.actors[a0].state_dict()) == list(_sd(g, f"actor0/{a0}"))           # the reference's keys, in order
    assert list(agent.critics[a0].state_dict()) == list(_sd(g, f"critic0/{a0}"))
    assert agent.gamma == float(g["gamma"]) and agent.tau == float(g["tau"]) and agent.lr_critic == float(g["lr_critic"])
    batch = tuple({a: torch.from_numpy(g[f"s1_{f}/{a}"].copy()) for a in ids} for f in FIELDS)
    losses = agent.learn(batch)
    assert losses == {a: (2.0 * i, 2.0 * i + 1.0) for i, a in enumerate(ids)}            # [n_agents, 2] = (actor, critic)
    s = standin.seen
    LN_AFFINE, LN_PLAIN, RELU, TANH = 1, 2, 1, 4
    assert s["actor_layers"][0] == [(18, 64, LN_AFFINE, RELU), (64, 64, LN_AFFINE, RELU), (64, 32, LN_PLAIN, RELU),
                                    (32, 64, LN_AFFINE, RELU), (64, 5, 0, TANH)]
    assert s["critic_layers"][0] == [(72, 32, 0, RELU), (52, 64, LN_AFFINE, RELU), (64, 1, 0, 0)]
    cat = lambda f: np.concatenate([g[f"s1_{f}/{a}"] for a in ids], axis=1)
    np.testing.assert_array_equal(s["obs"], cat("obs")); np.testing.assert_array_equal(s["next_obs"], cat("next_obs"))
    np.testing.assert_array_equal(s["act"], cat("action"))
    for i, a in enumerate(ids):
        np.testing.assert_array_equal(s["rew"][:, i], g[f"s1_reward/{a}"][:, 0])          # [B, n_agents]; NaN travels as NaN
        np.testing.assert_array_equal(s["done"][:, i], g[f"s1_done/{a}"][:, 0])
        p = s["ptrs"][i]
        assert p["actor"] == agent.actors[a].buffers.params.data_ptr() and p["actor_target"] == agent.actor_targets[a].buffers.params.data_ptr()
        assert p["critic"] == agent.critics[a].buffers.params.data_ptr() and p["critic_target"] == agent.critic_targets[a].buffers.params.data_ptr()
        ao, co = agent.actor_optimizers[a], agent.critic_optimizers[a]
        assert (p["actor_grads"], p["actor_m"], p["actor_v"]) == (ao.grads.data_ptr(), ao.exp_avg.data_ptr(), ao.exp_avg_sq.data_ptr())
        assert (p["critic_grads"], p["critic_m"], p["critic_v"]) == (co.grads.data_ptr(), co.exp_avg.data_ptr(), co.exp_avg_sq.data_ptr())
    assert s["cfg"]["bc1_actor"] == 1.0 - 0.9 ** 1 and s["cfg"]["bc2_critic"] == 1.0 - 0.999 ** 1
    assert s["cfg"]["serial"] == 0 and s["step_state"] is None                            # concurrent agents, eager scalars
    agent.learn(batch)
    assert standin.seen["cfg"]["bc1_critic"] == 1.0 - 0.9 ** 2
    # the replay's packed matrices go in as they are
    buf = MultiAgentReplayBuffer(64, list(FIELDS), ids, device="cuda")
    buf.save_to_memory(*tuple({a: g[f"s0_{f}/{a}"] for a in ids} for f in FIELDS), is_vectorised=True)
    random.seed(5)
    agent.learn(buf.sample(int(g["B"])))
    random.seed(5)
    pos = random.sample(range(int(g["B"])), int(g["B"]))
    np.testing.assert_array_equal(standin.seen["obs"], np.concatenate([g[f"s0_obs/{a}"] for a in ids], axis=1)[pos])
    np.testing.assert_array_equal(standin.seen["rew"], np.stack([g[f"s0_reward/{a}"][pos, 0] for a in ids], axis=1))
    # clone: same networks, optimiser step counts travel
    c = agent.clone(index=3)
    assert c.index == 3 and c.actor_optimizers[a0].step == 3 and torch.equal(c.critics[a0].buffers.params, agent.critics[a0].buffers.params)
    # cross-rank move (sharded tournament): pickled description + flat tensors rebuild the same member
    import pickle
    agent.fitness, agent.scores = [1.5, 2.5], [3.0]
    meta, tensors = agent.export_state()
    assert len(tensors) == 8 * len(ids)
    moved = MADDPG.from_state(pickle.loads(pickle.dumps(meta)), [t.clone() for t in tensors], agent)
    assert moved.index == agent.index and moved.fitness == [1.5, 2.5] and moved.critic_optimizers[a0].step == 3
    assert moved.lr_critic == agent.lr_critic and moved.agent_ids == agent.agent_ids
    for a in ids:
        assert torch.equal(moved.actors[a].buffers.params, agent.actors[a].buffers.params)
        assert torch.equal(moved.critic_targets[a].buffers.params, agent.critic_targets[a].buffers.params)
        assert torch.equal(moved.actor_optimizers[a].exp_avg_sq, agent.actor_optimizers[a].exp_avg_sq)
    # checkpoints: into an existing member (hyper-parameters included) and from the file alone
    import os
    import tempfile
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "member.pt")
        agent.lr_critic = 0.004
        agent.actor_optimizers[a0].exp_avg.fill_(0.25)
        agent.save_checkpoint(path)
        other = MADDPG(agent.observation_spaces, agent.action_spaces, agent_ids=ids, batch_size=int(g["B"]), index=9)
        other.load_checkpoint(path)
        fresh = MADDPG.load(path, device="cuda")
        with pytest.raises(ValueError):                      # other agents: refused, not silently half-loaded
            MADDPG(agent.observation_spaces[:3], agent.action_spaces[:3], agent_ids=ids[:3]).load_checkpoint(path)
    for m in (other, fresh):
        assert m.lr_critic == 0.004 and m.critic_optimizers[a0].lr == 0.004 and m.index == agent.index
        assert m.actor_optimizers[a0].step == 3 and float(m.actor_optimizers[a0].exp_avg[0]) == 0.25
        for a in ids:
            assert torch.equal(m.critics[a].buffers.params, agent.critics[a].buffers.params)
            assert torch.equal(m.actor_targets[a].buffers.params, agent.actor_targets[a].buffers.params)


def test_device_mutation_decisions_match_index_put_semantics(standin):
    from agilerl_b200.engine import NetBuffers
    from agilerl_b200.hpo import Mutations
    from agilerl_b200.networks.spec import FlatLayout, MlpSpec, NetSpec
    spec = NetSpec("q", MlpSpec("encoder.model.", "encoder", 18, 32, [64, 64]),
                   MlpSpec("head_net.model.", "actor", 32, 5, [64], output_activation="Tanh"), None, 5, 1)

    class Net:
        pass

    def mk():
        n = Net()
        n.layout = FlatLayout(spec)
        n.buffers = NetBuffers(n.layout, "cpu")
        n.buffers.params.copy_(torch.randn(n.buffers.params.numel(), generator=torch.Generator().manual_seed(0)))
        return n
    ours, ref = mk(), mk()
    keys = [k for k, e in ours.layout.entries.items() if "norm" not in k and len(e.shape) == 2]
    gz = torch.Generator().manual_seed(9)
    normals = {k: torch.randn(int(np.ceil(0.1 * np.prod(ours.layout.entries[k].shape))), generator=gz) for k in keys}
    Mutations(0, 0, 0.5, 1, 0, 0, rand_seed=3, device="cuda")._gaussian_parameter_mutation_device(ours, normals=normals)
    rng = np.random.default_rng(3)                                   # mutation.py:760-822 restated with the same noise per slot
    for key in rng.choice(keys, int(rng.integers(1, len(keys) + 1)), replace=False):
        W = ref.buffers.view(str(key))
        n_mut = int(np.ceil(0.1 * W.shape[0] * W.shape[1]))
        rows, cols = torch.tensor(rng.integers(0, W.shape[0], size=n_mut)), torch.tensor(rng.integers(0, W.shape[1], size=n_mut))
        r, z = torch.tensor(rng.uniform(0, 1, size=n_mut), dtype=W.dtype), normals[str(key)]
        cur = W[rows, cols]
        new = cur.clone()
        ms, mr, mn = r < 0.05, (r >= 0.05) & (r < 0.1), r >= 0.1
        new[ms] = cur[ms] + (10 * cur[ms]).abs() * z[ms]
        new[mr] = z[mr]
        new[mn] = cur[mn] + (0.1 * cur[mn]).abs() * z[mn]
        Wc = W.clone()
        Wc[rows, cols] = new.clamp(-1000000, 1000000)                # CPU index_put_: the last writer of a position wins
        W.copy_(Wc)
    assert torch.equal(ours.buffers.params, ref.buffers.params)


class _ParallelEnv:
    """Deterministic PettingZoo-style parallel environment (optionally vectorised): rewards depend on the step and the
    action, agent_1 is 'killed' (NaN reward / termination) for a while, episodes end at different steps per env."""

    def __init__(self, ids, num_envs=None):
        self.ids, self.t = ids, 0
        if num_envs is not None:
            self.num_envs = num_envs
        self.n = num_envs or 1

    def reset(self):
        self.t = 0
        shape = (self.n, 4) if hasattr(self, "num_envs") else (4,)
        return {a: np.zeros(shape, np.float32) for a in self.ids}, {a: {} for a in self.ids}

    def step(self, action):
        self.t += 1
        vec = hasattr(self, "num_envs")
        base = np.arange(self.n, dtype=np.float64) + self.t
        rew, term, trunc = {}, {}, {}
        for k, a in enumerate(self.ids):
            r = base * (k + 1) + float(np.sum(action[a])) * 0.01
            d = (self.t >= 3 + np.arange(self.n)).astype(np.float64)
            if k == 1 and self.t == 2:
                r, d = np.full(self.n, np.nan), np.full(self.n, np.nan)
            rew[a], term[a], trunc[a] = (r, d, np.zeros(self.n)) if vec else (float(r[0]), float(d[0]), False)
        shape = (self.n, 4) if vec else (4,)
        return {a: np.full(shape, self.t, np.float32) for a in self.ids}, rew, term, trunc, {a: {} for a in self.ids}


_TEST_LOOP_CASES = [(True, True, None), (True, False, 4), (False, True, None)]
_TL_IDS = ["agent_0", "agent_1", "agent_2"]


def _fake_get_action(n):
    def fake_get_action(self, obs, infos=None, **kw):
        rows = n or 1
        act = {a: np.full((rows, 2), 0.1 * (k + 1), np.float32) for k, a in enumerate(_TL_IDS)}
        return act, act
    return fake_get_action


def reference_test_loop_outputs():
    """``MADDPG.test`` of the unmodified reference (maddpg.py:756-875, run through oracle/refshim) on the cases of
    test_maddpg_test_loop_matches_the_unmodified_reference; tests/golden/make_golden.py stores them in maddpg_host.npz."""
    from oracle import refshim
    refshim.install()
    import agilerl.algorithms.maddpg as r_ma
    out = {}
    for vect, sum_scores, max_steps in _TEST_LOOP_CASES:
        n = 3 if vect else None
        ref = r_ma.MADDPG.__new__(r_ma.MADDPG)                   # the method under test only needs these attributes
        ref.agent_ids, ref.fitness = _TL_IDS, []
        ref.set_training_mode = lambda training: None
        ref.get_action = _fake_get_action(n).__get__(ref)
        key = f"test_loop/{vect}-{sum_scores}-{max_steps}"
        out[key + "/scores"] = np.asarray(r_ma.MADDPG.test(ref, _ParallelEnv(_TL_IDS, n), max_steps=max_steps, loop=2,
                                                         sum_scores=sum_scores))
        out[key + "/fitness"] = np.asarray(ref.fitness[-1])
    return out


@pytest.mark.parametrize("vect,sum_scores,max_steps", _TEST_LOOP_CASES)
def test_maddpg_test_loop_matches_the_unmodified_reference(standin, vect, sum_scores, max_steps):
    """``MADDPG.test`` (maddpg.py:756-875) against the reference's own method (its results stored in maddpg_host.npz) on the
    same environment with the same (stubbed) actions: identical fitness, NaN handling and episode bookkeeping."""
    from agilerl_b200.algorithms import MADDPG
    from agilerl_b200.compat import spaces
    g = load_golden("maddpg_host.npz")
    key = f"test_loop/{vect}-{sum_scores}-{max_steps}"
    n = 3 if vect else None
    ours = MADDPG([spaces.Box(-1.0, 1.0, (4,), np.float32)] * 3, [spaces.Box(-1.0, 1.0, (2,), np.float32)] * 3, agent_ids=_TL_IDS)
    ours.get_action = _fake_get_action(n).__get__(ours)
    got = ours.test(_ParallelEnv(_TL_IDS, n), max_steps=max_steps, loop=2, sum_scores=sum_scores)
    np.testing.assert_array_equal(np.asarray(got), g[key + "/scores"])
    np.testing.assert_array_equal(np.asarray(ours.fitness[-1]), g[key + "/fitness"])
    assert ours.training is False


_GA_IDS = ["a", "b"]


def _ga_spaces(sp):
    return ([sp.Box(-1.0, 1.0, (6,), np.float32), sp.Box(-1.0, 1.0, (4,), np.float32)],
            [sp.Box(-2.0, 3.0, (3,), np.float32), sp.Box(-0.5, 1.5, (3,), np.float32)])


def _ga_calls():
    """(training, obs, infos, seed) of every ``get_action`` call: three plain ones, then actions dictated by the environment
    (maddpg.py:518-529): NaN rows are the agent's own, the rest overwrite."""
    g = torch.Generator().manual_seed(0)
    calls = []
    for training in (True, True, False):
        calls.append((training, {"a": torch.randn(4, 6, generator=g).numpy(), "b": torch.randn(4, 4, generator=g).numpy()},
                      None, 77))
    eda = np.full((4, 3), np.nan)
    eda[1] = [0.5, -0.25, 1.0]
    eda[3] = [-2.0, 3.0, 0.0]
    infos = {"a": {"env_defined_actions": eda}, "b": {"env_defined_actions": np.full((4, 3), np.nan)}}
    calls.append((False, {"a": torch.randn(4, 6, generator=g).numpy(), "b": torch.randn(4, 4, generator=g).numpy()}, infos, 78))
    return calls


def _copy_args(obs, infos):
    return ({k: v.copy() for k, v in obs.items()},
            None if infos is None else {k: {kk: vv.copy() for kk, vv in v.items()} for k, v in infos.items()})


def reference_get_action_outputs():
    """``get_action`` / ``action_noise`` / ``reset_action_noise`` of the unmodified reference (maddpg.py:428-558) on the calls
    of ``_ga_calls``, with what its actors were handed and returned; tests/golden/make_golden.py stores them in
    maddpg_host.npz."""
    from oracle import refshim
    refshim.install()
    import agilerl.algorithms.maddpg as r_ma
    from gymnasium import spaces as r_spaces
    out = {}
    for ou_noise in (True, False):
        pre = f"get_action/{ou_noise}"
        torch.manual_seed(5)
        ref = r_ma.MADDPG(*_ga_spaces(r_spaces), agent_ids=_GA_IDS, O_U_noise=ou_noise, vect_noise_dim=4, expl_noise=0.3,
                          device="cpu")
        seen = {a: [] for a in _GA_IDS}
        for a in _GA_IDS:
            actor = ref.actors[a]
            out[f"{pre}/{a}/action_low"], out[f"{pre}/{a}/action_high"] = actor.action_low.cpu().numpy(), actor.action_high.cpu().numpy()
            out[f"{pre}/{a}/output_activation"] = np.asarray(actor.output_activation)
        cls = type(ref.actors[_GA_IDS[0]])
        call = cls.__call__                  # the actors override __call__, so module hooks do not see their calls

        def recording_call(self, x, *args, **kw):
            y = call(self, x, *args, **kw)
            a = next(a for a in _GA_IDS if ref.actors[a] is self)
            seen[a].append((x.detach().cpu().numpy().copy(), y.detach().cpu().numpy().copy()))
            return y
        cls.__call__ = recording_call
        try:
            for c, (training, obs, infos, seed) in enumerate(_ga_calls()):
                ref.set_training_mode(training)
                torch.manual_seed(seed)
                want_p, want_r = ref.get_action(*_copy_args(obs, infos))
                for a in _GA_IDS:
                    out[f"{pre}/{c}/{a}/processed"], out[f"{pre}/{c}/{a}/raw"] = np.asarray(want_p[a]), np.asarray(want_r[a])
        finally:
            cls.__call__ = call
        for a in _GA_IDS:
            out[f"{pre}/{a}/actor_in"] = np.stack([x for x, _ in seen[a]])
            out[f"{pre}/{a}/actor_out"] = np.stack([y for _, y in seen[a]])
        ref.reset_action_noise([1, 3])
        for a in _GA_IDS:
            out[f"{pre}/{a}/noise_after_reset"] = ref.current_noise[a].cpu().numpy()
    return out


@pytest.mark.parametrize("ou_noise", [True, False])
def test_maddpg_get_action_noise_and_rescaling_match_the_unmodified_reference(standin, ou_noise):
    """``get_action`` / ``action_noise`` (maddpg.py:428-558) around the actor forward: exploration noise from torch's global
    generator (Ornstein-Uhlenbeck state carried across calls, or Gaussian), clamp to [-1, 1], rescale to the action bounds (kept quirk: the LAST agent's bounds for every agent, maddpg.py:504-511) —
    against the reference object's results (stored in maddpg_host.npz), our actors stubbed to return what the reference actors
    returned on the same inputs."""
    from agilerl_b200.algorithms import MADDPG
    from agilerl_b200.compat import spaces
    g = load_golden("maddpg_host.npz")
    pre = f"get_action/{ou_noise}"
    torch.manual_seed(5)
    ours = MADDPG(*_ga_spaces(spaces), agent_ids=_GA_IDS, O_U_noise=ou_noise, vect_noise_dim=4, expl_noise=0.3)

    class Stub:
        def __init__(self, a):
            self.a, self.calls = a, 0
            self.action_low = torch.from_numpy(g[f"{pre}/{a}/action_low"])
            self.action_high = torch.from_numpy(g[f"{pre}/{a}/action_high"])
            self.output_activation = str(g[f"{pre}/{a}/output_activation"])

        def __call__(self, obs):
            k, self.calls = self.calls, self.calls + 1
            np.testing.assert_array_equal(obs.cpu().numpy(), g[f"{pre}/{self.a}/actor_in"][k])
            return torch.from_numpy(g[f"{pre}/{self.a}/actor_out"][k].copy())
    ours.actors = {a: Stub(a) for a in _GA_IDS}
    for c, (training, obs, infos, seed) in enumerate(_ga_calls()):
        ours.set_training_mode(training)
        torch.manual_seed(seed)
        got_p, got_r = ours.get_action(*_copy_args(obs, infos))
        for a in _GA_IDS:
            np.testing.assert_array_equal(got_r[a], g[f"{pre}/{c}/{a}/raw"], err_msg=f"raw {a} call {c} training={training}")
            np.testing.assert_array_equal(got_p[a], g[f"{pre}/{c}/{a}/processed"], err_msg=f"processed {a} call {c}")
    # the environment's actions overwrite the processed ones, and the overwritten dict also comes back as the "raw" actions
    np.testing.assert_array_equal(got_p["a"][1], [0.5, -0.25, 1.0])
    assert all(s.calls == len(g[f"{pre}/{a}/actor_in"]) for a, s in ours.actors.items())
    ours.reset_action_noise([1, 3])
    for a in _GA_IDS:
        np.testing.assert_array_equal(ours.current_noise[a].cpu().numpy(), g[f"{pre}/{a}/noise_after_reset"])


def test_rl_hyperparameter_and_parameter_mutations_on_a_maddpg_member(standin):
    """mutation.py:413-452 / :521-584 on a multi-agent member: a learning-rate mutation restarts every optimiser of that
    kind's owner (fresh Adam state, like ``reinit_optimizers``), a parameter mutation walks every sub-agent's actor and
    reloads the targets; architecture mutations are refused loudly."""
    from agilerl_b200.algorithms import MADDPG
    from agilerl_b200.algorithms.core.registry import HyperparameterConfig, RLParameter
    from agilerl_b200.compat import spaces
    from agilerl_b200.hpo import Mutations
    ids = ["a", "b"]
    hp = HyperparameterConfig(lr_actor=RLParameter(min=1e-5, max=1e-2), lr_critic=RLParameter(min=1e-5, max=1e-2),
                              batch_size=RLParameter(min=8, max=512, dtype=int))
    m = MADDPG([spaces.Box(-1.0, 1.0, (6,), np.float32)] * 2, [spaces.Box(-1.0, 1.0, (3,), np.float32)] * 2, agent_ids=ids, hp_config=hp)
    m.use_graph = False
    for o in m._all_opts:
        o.step = 5
    c = m.clone(index=1)
    assert c.registry.hp_config.names() == ["lr_actor", "lr_critic", "batch_size"] and c._all_opts[0].step == 5
    mut = Mutations(0, 0, 0.5, 0, 0, 1, rand_seed=4, device="cuda")
    seen = set()
    for _ in range(12):
        before = (c.lr_actor, c.lr_critic, c.batch_size)
        [c] = mut.mutation([c])
        seen.add(c.mut)
        after = (c.lr_actor, c.lr_critic, c.batch_size)
        assert c.mut in ("lr_actor", "lr_critic", "batch_size") and sum(x != y for x, y in zip(before, after)) <= 1
        if c.mut.startswith("lr"):
            assert all(o.step == 0 for o in c._all_opts)                        # reinit_optimizers: fresh Adam state
            assert c.actor_optimizers["a"].lr == c.lr_actor and c.critic_optimizers["b"].lr == c.lr_critic
    assert len(seen) >= 2
    pm = Mutations(0, 0, 0.5, 1, 0, 0, rand_seed=2, device="cuda")
    before = {a: c.actors[a].buffers.params.clone() for a in ids}
    [c] = pm.mutation([c])
    assert c.mut == "param"
    for a in ids:
        assert not torch.equal(c.actors[a].buffers.params, before[a])
        assert torch.equal(c.actor_targets[a].buffers.params, c.actors[a].buffers.params)
    with pytest.raises(NotImplementedError):
        Mutations(0, 1, 0.5, 0, 0, 0, rand_seed=2, device="cuda").mutation([c])
    am = Mutations(0, 0, 0.5, 0, 1, 0, rand_seed=2, device="cuda")
    with pytest.warns(UserWarning):
        [c] = am.mutation([c])
    assert c.mut == "None"                                                      # mutation.py:473-480: not supported for MADDPG


# ---- the behaviours the reference's own buffer tests pin (tests/test_components/test_multi_agent_replay_buffer.py), on the
# ---- HBM layout with the stand-in data movers --------------------------------------------------------------------------
def _step(k, ids=("agent1", "agent2")):
    return ({a: np.array([k, k + 1, k + 2]) for a in ids}, {a: np.array([10 * k, 10 * k + 1]) for a in ids},
            {a: np.array([100 * k + i]) for i, a in enumerate(ids)})


def test_buffer_attributes_length_and_counter(standin):
    from agilerl_b200.components import MultiAgentReplayBuffer
    fields, ids = ["state", "action", "reward"], ["agent1", "agent2"]
    buf = MultiAgentReplayBuffer(100, fields, ids)
    assert len(buf) == 0 and buf.memory_size == 100 and buf.field_names == fields and buf.agent_ids == ids
    assert buf.counter == 0 and buf.device is None
    for k in range(3):
        buf.save_to_memory(*_step(k))
    assert len(buf) == 3 and buf.counter == 3
    for bad in (dict(memory_size=0), dict(field_names=[]), dict(agent_ids=[])):
        kw = dict(memory_size=4, field_names=fields, agent_ids=ids) | bad
        with pytest.raises(AssertionError):
            MultiAgentReplayBuffer(**kw)


def test_oldest_step_falls_out_when_full(standin):
    from agilerl_b200.components import MultiAgentReplayBuffer
    ids = ["agent1", "agent2"]
    buf = MultiAgentReplayBuffer(2, ["state", "action", "reward"], ids)
    for k in (1, 2, 3):
        buf.save_to_memory(*_step(k))
    assert len(buf) == 2 and buf.counter == 3
    state, action, reward = buf.sample(2)
    assert sorted(state["agent1"][:, 0].tolist()) == [2.0, 3.0]                 # step 1 is gone (deque(maxlen) semantics)
    for row in range(2):                                                       # fields of one step stay together
        k = int(state["agent1"][row, 0])
        assert action["agent2"][row].tolist() == [10.0 * k, 10.0 * k + 1] and reward["agent2"][row].tolist() == [100.0 * k + 1]


def test_vectorised_and_single_saves_mix_and_samples_stay_aligned(standin):
    from agilerl_b200.components import MultiAgentReplayBuffer
    ids = ["agent1", "agent2"]
    buf = MultiAgentReplayBuffer(100, ["environments", "state"], ids, "cuda")
    num_envs = 50
    envs = {a: np.array([[e] for e in range(num_envs)]) for a in ids}
    states = {a: np.array([[(e + 1) * (i + 1)] for e in range(num_envs)]) for i, a in enumerate(ids)}
    buf.save_to_memory(envs, states, is_vectorised=True)
    assert len(buf) == num_envs
    buf.save_to_memory({a: np.array([77]) for a in ids}, {a: np.array([78 * (i + 1)]) for i, a in enumerate(ids)}, is_vectorised=False)
    assert len(buf) == num_envs + 1
    s_envs, s_states = buf.sample(batch_size=25)
    for i, a in enumerate(ids):
        assert s_envs[a].dtype == torch.float32 and s_envs[a].shape == (25, 1)
        for row in range(25):
            e = int(s_envs[a][row])
            assert float(s_states[a][row]) == (e + 1) * (i + 1)


def test_sampled_shapes_follow_the_leaves_including_images(standin):
    from agilerl_b200.components import MultiAgentReplayBuffer
    ids = ["agent1", "agent2"]
    buf = MultiAgentReplayBuffer(10, ["state", "action", "reward"], ids)
    rng = np.random.default_rng(0)
    state = {a: rng.random((3, 16, 16)) for a in ids}
    buf.save_to_memory(state, {a: np.array([4, 5]) for a in ids}, {a: 6.5 for a in ids})
    s, a_, r = buf.sample(1)
    assert s["agent1"].shape == (1, 3, 16, 16) and a_["agent1"].shape == (1, 2) and r["agent1"].shape == (1, 1)
    np.testing.assert_array_equal(s["agent2"][0].numpy(), state["agent2"].astype(np.float32))      # float64 -> .float()
    assert a_["agent2"].dtype == torch.float32 and float(r["agent1"]) == 6.5
    with pytest.raises(NotImplementedError):
        MultiAgentReplayBuffer(4, ["state"], ids).save_to_memory({a: {"x": np.zeros(2)} for a in ids})
    with pytest.raises(TypeError):
        buf.save_to_memory(state)                                                                  # a field is missing


def test_create_population_builds_maddpg_members_with_the_references_defaults(standin):
    """utils/utils.py:444-472: the INIT_HP -> constructor mapping (gamma 0.95, tau 0.01, lr 1e-4 / 1e-3 defaults of
    create_population, ``vect_noise_dim = num_envs``)."""
    from agilerl_b200.compat import spaces
    from agilerl_b200.utils.utils import create_population
    ids = ["a", "b"]
    pop = create_population("MADDPG", [spaces.Box(-1.0, 1.0, (6,), np.float32)] * 2, [spaces.Box(-1.0, 1.0, (3,), np.float32)] * 2,
                            None, {"AGENT_IDS": ids, "BATCH_SIZE": 32, "LEARN_STEP": 16}, population_size=3, num_envs=4, first_index=5)
    assert [m.index for m in pop] == [5, 6, 7] and all(m.algo == "MADDPG" and m.agent_ids == ids for m in pop)
    m = pop[0]
    assert (m.batch_size, m.learn_step, m.gamma, m.tau, m.lr_actor, m.lr_critic) == (32, 16, 0.95, 0.01, 0.0001, 0.001)
    assert m.vect_noise_dim == 4 and m.current_noise["a"].shape == (4, 3) and m.O_U_noise is True
    with pytest.raises(NotImplementedError):
        create_population("MADDPG", m.observation_spaces, m.action_spaces, None, {"AGENT_IDS": ids, "SHARE_ENCODERS": True})
    with pytest.raises(NotImplementedError):
        create_population("PPO", m.observation_spaces[0], m.action_spaces[0], None, {})
    # the single-agent deterministic-policy learners go through the same helper (utils.py:320-352, 414-442)
    osp, asp = spaces.Box(-np.inf, np.inf, (17,), np.float32), spaces.Box(-1.0, 1.0, (6,), np.float32)
    [td3] = create_population("TD3", osp, asp, None, {"POLICY_FREQ": 3}, num_envs=2)
    [ddpg] = create_population("DDPG", osp, asp, None, {"TAU": 0.002})
    assert (td3.algo, td3.tau, td3.policy_freq, td3.gamma, td3.vect_noise_dim) == ("TD3", 0.005, 3, 0.99, 2)
    assert (ddpg.algo, ddpg.tau, ddpg.policy_freq, ddpg.lr_critic) == ("DDPG", 0.002, 2, 0.001)


def test_share_encoders_pins_the_critics_encoders_through_learn(standin):
    """ddpg.py:289-296, 335-351 (``share_encoder_parameters``): with ``share_encoders=True`` the critics and target critics
    carry a detached copy of the actor's encoder taken at construction / after a mutation, outside every optimiser.  The
    fused learn call updates whole parameter buffers, so ``learn`` restores the critics' encoder block afterwards.
    (Restated from the reference's code: its ``tensordict.from_module / to_module`` cannot run in this image, so this
    behaviour is not pinned by a golden run.)"""
    from agilerl_b200.algorithms import TD3
    from agilerl_b200.compat import spaces

    def fake_learn(actor, critic, cfg, bufs, stream):          # a learn call that moves EVERY parameter of every network
        b = bufs._obj
        for ptr, n in ((b.actor, actor._obj.n_params), (b.actor_target, actor._obj.n_params)) + tuple(
                (p, critic._obj.n_params) for i in range(2) for p in (b.critic[i], b.critic_target[i])):
            _f32(ptr, n)[:] += 1.0
        _f32(b.critic_loss, 1)[0] = 1.0
        _f32(b.actor_loss, 1)[0] = -1.0
        return 0
    standin.b2rl_ddpg_learn = fake_learn
    standin.b2rl_ddpg_workspace_bytes = lambda a, c, B, out: setattr(out._obj, "value", 64) or 0
    osp, asp = spaces.Box(-np.inf, np.inf, (17,), np.float32), spaces.Box(-1.0, 1.0, (6,), np.float32)
    agent = TD3(osp, asp, batch_size=8, share_encoders=True, policy_freq=1)
    enc_keys = [k for k in agent.actor.state_dict() if k.startswith("encoder.")]
    snap = {k: agent.actor.state_dict()[k].clone() for k in enc_keys}
    nets = agent._critics() + agent._targets()
    assert enc_keys and all(torch.equal(n.state_dict()[k], snap[k]) for n in nets for k in enc_keys)
    heads0 = [{k: v.clone() for k, v in n.state_dict().items() if not k.startswith("encoder.")} for n in nets]
    g = torch.Generator().manual_seed(0)
    exp = dict(obs=torch.randn(8, 17, generator=g), action=torch.rand(8, 6, generator=g), reward=torch.randn(8, generator=g),
               next_obs=torch.randn(8, 17, generator=g), done=torch.zeros(8))
    agent.learn(exp)
    assert all(not torch.equal(agent.actor.state_dict()[k], snap[k]) for k in enc_keys)            # the actor's encoder learns
    for n, h0 in zip(nets, heads0):
        assert all(torch.equal(n.state_dict()[k], snap[k]) for k in enc_keys)                       # the critics' stay pinned
        assert all(not torch.equal(n.state_dict()[k], v) for k, v in h0.items())                    # their heads moved
    clone = agent.clone(index=1)                                                                    # the pinned values travel
    assert all(torch.equal(n.state_dict()[k], snap[k]) for n in clone._critics() + clone._targets() for k in enc_keys)
    agent.mutation_hook()                                                                           # re-share after a mutation
    assert all(torch.equal(n.state_dict()[k], agent.actor.state_dict()[k]) for n in nets for k in enc_keys)
    plain = TD3(osp, asp, batch_size=8)                                                             # default: nothing is pinned
    e0 = plain.critic_1.state_dict()[enc_keys[0]].clone()
    plain.learn(dict(exp, action=torch.rand(8, 6, generator=g)))
    assert not torch.equal(plain.critic_1.state_dict()[enc_keys[0]], e0)


def test_td3_checkpoint_carries_every_optimiser(standin, tmp_path):
    """core/base.py:919-1049 for a learner with several optimisers: actor AND critic Adam moments / step counts, the
    learn counter (policy_freq phase) and the mutated hyper-parameters come back."""
    from agilerl_b200.algorithms import DDPG, TD3
    from agilerl_b200.compat import spaces
    osp, asp = spaces.Box(-np.inf, np.inf, (17,), np.float32), spaces.Box(-1.0, 1.0, (6,), np.float32)
    for cls, crit in ((TD3, "critic_2"), (DDPG, "critic")):
        a = cls(osp, asp, batch_size=8)
        opt = getattr(a, crit + "_optimizer")
        opt.exp_avg.fill_(0.5); opt.exp_avg_sq.fill_(0.25); opt.step = 7
        a.actor_optimizer.step, a.learn_counter, a.lr_critic = 3, 5, 0.005
        a.actor.buffers.params.add_(1.0)
        path = str(tmp_path / f"{cls.__name__}.pt")
        a.save_checkpoint(path)
        b = cls(osp, asp, batch_size=8)
        b.load_checkpoint(path)
        bopt = getattr(b, crit + "_optimizer")
        assert torch.equal(a.actor.buffers.params, b.actor.buffers.params)
        assert torch.equal(getattr(a, crit).buffers.params, getattr(b, crit).buffers.params)
        assert float(bopt.exp_avg[0]) == 0.5 and float(bopt.exp_avg_sq[0]) == 0.25 and bopt.step == 7 and bopt.lr == 0.005
        assert b.actor_optimizer.step == 3 and b.learn_counter == 5 and b.lr_critic == 0.005


def test_mutation_sweep_keeps_td3_and_ddpg_members_consistent(standin):
    """Every mutation kind over DDPG (``share_encoders=True``: the reference ``create_population``'s default) and TD3 members,
    a learn call after each: the architecture mutation the policy drew is applied — same name, same drawn parameters — to the
    critics too (mutation.py:875-879), targets are rebuilt, shared encoders re-pinned by the mutation hook, optimisers
    restarted; the layer tables the kernels would walk stay consistent and the member still clones / moves."""
    import pickle
    from agilerl_b200.algorithms import DDPG, TD3
    from agilerl_b200.algorithms.core.registry import HyperparameterConfig, RLParameter
    from agilerl_b200.compat import spaces
    from agilerl_b200.hpo import Mutations

    def learn(actor, critic, cfg, bufs, stream):
        a, c = actor._obj, critic._obj
        assert c.val[0].in_c == c.enc[c.n_enc - 1].out_c + a.val[a.n_val - 1].out_c and a.val[0].in_c == a.enc[a.n_enc - 1].out_c
        for d in (a, c):
            for layers, n in ((d.enc, d.n_enc), (d.val, d.n_val)):
                assert all(layers[i].in_c == layers[i - 1].out_c for i in range(1, n))
        _f32(bufs._obj.critic_loss, 1)[0] = 0.5
        _f32(bufs._obj.actor_loss, 1)[0] = 0.1
        return 0
    standin.b2rl_ddpg_learn = learn
    standin.b2rl_ddpg_workspace_bytes = lambda a, c, B, out: setattr(out._obj, "value", 64) or 0
    hp = HyperparameterConfig(lr_actor=RLParameter(min=1e-5, max=1e-2), lr_critic=RLParameter(min=1e-5, max=1e-2),
                              batch_size=RLParameter(min=8, max=64, dtype=int))
    osp, asp = spaces.Box(-np.inf, np.inf, (17,), np.float32), spaces.Box(-1.0, 1.0, (6,), np.float32)
    g = torch.Generator().manual_seed(0)
    for cls in (DDPG, TD3):
        agent = cls(osp, asp, batch_size=8, hp_config=hp, share_encoders=(cls is DDPG))
        muts = Mutations(0.1, 0.4, 0.3, 0.2, 0.1, 0.2, rand_seed=3, device="cuda")
        seen = set()
        for _ in range(30):
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                [agent] = muts.mutation([agent.clone()])
            seen.add(agent.mut)
            B = agent.batch_size
            agent.learn(dict(obs=torch.randn(B, 17, generator=g), action=torch.rand(B, 6, generator=g), reward=torch.randn(B, generator=g),
                             next_obs=torch.randn(B, 17, generator=g), done=torch.zeros(B)))
            pairs = (("actor", "actor_target"),) + tuple(zip(agent._critic_names, agent._target_names))
            for n, t in pairs:
                sd_n, sd_t = getattr(agent, n).state_dict(), getattr(agent, t).state_dict()
                assert list(sd_n) == list(sd_t) and all(sd_n[k].shape == sd_t[k].shape for k in sd_n), (agent.mut, n)
            crit = getattr(agent, agent._critic_names[0])
            assert list(crit.encoder.hidden_size) == list(agent.actor.encoder.hidden_size), agent.mut      # analogous mutation
            if agent.share_encoders:
                enc = [k for k in agent.actor.state_dict() if k.startswith("encoder.")]
                assert all(torch.equal(crit.state_dict()[k], getattr(agent, agent._target_names[0]).state_dict()[k]) for k in enc)
            meta, tensors = agent.export_state()
            moved = cls.from_state(pickle.loads(pickle.dumps(meta)), [t.clone() for t in tensors], agent)
            assert torch.equal(moved.actor.buffers.params, agent.actor.buffers.params)
        assert {"param", "None"} <= seen and any(m.startswith("encoder.") for m in seen) and any(m.startswith("lr_") for m in seen), seen
