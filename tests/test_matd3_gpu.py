"""GPU parity of ``MATD3`` (twin centralised critics, delayed policy updates) on the multi-agent CUDA path:
``b2rl_maddpg_learn`` with ``twin = 1`` and, on calls without an actor step, ``critic_only = 1``.

Golden data recorded from the UNMODIFIED reference (tests/golden/make_golden_matd3.py, read by tests/_matd3_golden.py: the
reference's gradients and final parameters are recomputed by the oracle, which tests/test_matd3_cpu.py pins to the
recorded digests): five consecutive learn calls with policy_freq = 2, so calls 2 and 4 step the actors and every
target.  Bars as tests/test_maddpg_gpu.py's: losses within 1e-5, every gradient tensor within 2e-5 of its largest element,
parameters after the five calls within Adam's reach of the reference's."""
import ctypes
import pickle

import numpy as np
import pytest
import torch

import _matd3_golden as G
from conftest import load_golden

pytestmark = pytest.mark.gpu

FIELDS = ("obs", "action", "reward", "next_obs", "done")
SETS = (("actor", "actors", "actor"), ("actor_target", "actor_targets", "actor"), ("critic_1", "critics_1", "critic"),
        ("critic_target_1", "critic_targets_1", "critic"), ("critic_2", "critics_2", "critic"),
        ("critic_target_2", "critic_targets_2", "critic"))
OPTS = ("actor_optimizers", "critic_1_optimizers", "critic_2_optimizers")


def _agent(g, **kw):
    from agilerl_b200.algorithms import MATD3
    from agilerl_b200.compat import spaces
    ids = [str(a) for a in g["agent_ids"]]
    obs = [spaces.Box(-1.0, 1.0, (int(d),), np.float32) for d in g["obs_dims"]]
    act = [spaces.Box(-1.0, 1.0, (int(d),), np.float32) for d in g["act_dims"]]
    net = {"head_config": {"hidden_size": [int(h) for h in g["a_hidden"]]}}
    agent = MATD3(obs, act, agent_ids=ids, net_config=net, batch_size=int(g["B"]), gamma=float(g["gamma"]), tau=float(g["tau"]),
                  lr_actor=float(g["lr_actor"]), lr_critic=float(g["lr_critic"]), policy_freq=int(g["policy_freq"]), **kw)
    for tag, attr, _ in SETS:
        for a in ids:
            getattr(agent, attr)[a].load_state_dict(G.initial_sd(g, tag, a))
    return ids, agent


def _batch(g, st, ids, device="cuda"):
    return G.batch(g, st, device)


def _state(agent):
    """Every parameter, target and Adam moment, and the step counts."""
    out = {}
    for a in agent.agent_ids:
        for _, attr, _ in SETS:
            out[f"{attr}/{a}"] = getattr(agent, attr)[a].buffers.params.clone()
        for name in OPTS:
            o = getattr(agent, name)[a]
            out[f"{name}/{a}/m"], out[f"{name}/{a}/v"] = o.exp_avg.clone(), o.exp_avg_sq.clone()
            out[f"{name}/{a}/step"] = o.step
    out["learn_counter"] = dict(agent.learn_counter)
    return out


def _assert_same(x, y, what=""):
    assert x.keys() == y.keys()
    for k in x:
        if isinstance(x[k], torch.Tensor):
            assert torch.equal(x[k], y[k]), (what, k)
        else:
            assert x[k] == y[k], (what, k, x[k], y[k])


def test_state_dict_keys_and_shapes_are_the_references():
    g = load_golden("matd3_vector.npz")
    ids, agent = _agent(g)
    assert not hasattr(agent, "critics") and agent.learn_counter == {a: 0 for a in ids}
    for tag, attr, _ in SETS:
        for a in ids:
            ref = G.initial_sd(g, tag, a)
            sd = getattr(agent, attr)[a].state_dict()
            assert list(sd) == list(ref), (tag, a)
            assert all(tuple(sd[k].shape) == tuple(v.shape) for k, v in ref.items()), (tag, a)


def test_learn_matches_reference_golden():
    g = load_golden("matd3_vector.npz")
    ids, agent = _agent(g)
    run = G.oracle_run(g)              # the reference's gradients / parameters (bit-exact: tests/test_matd3_cpu.py)
    for st in range(int(g["steps"])):
        losses = agent.learn(_batch(g, st, ids))
        for a in ids:
            assert (losses[a][0] is None) == bool(g[f"s{st}_actor_none/{a}"]), (st, a, losses[a])
            pairs = [("critic_loss", losses[a][1])] + ([] if losses[a][0] is None else [("actor_loss", losses[a][0])])
            for name, got in pairs:
                ref = float(g[f"s{st}_{name}/{a}"])
                assert abs(got - ref) <= 1e-5 * max(1.0, abs(ref)), (st, a, name, got, ref)
        checks = {0: (("critic_1", agent.critics_1, agent.critic_1_optimizers), ("critic_2", agent.critics_2, agent.critic_2_optimizers)),
                  1: (("actor", agent.actors, agent.actor_optimizers),)}.get(st, ())
        for group, nets, opts in checks:
            for a in ids:
                lay, grads = nets[a].layout, opts[a].grads
                for key, e in lay.entries.items():
                    if e.buf != "param":
                        continue
                    ref_g = run["grads"][st][f"{group}/{a}/{key}"]
                    got = grads[e.offset:e.offset + ref_g.numel()].view(ref_g.shape).cpu()
                    tol = 2e-5 * max(float(ref_g.abs().max()), 1e-6)
                    assert float((got - ref_g).abs().max()) <= tol, (group, a, key, float((got - ref_g).abs().max()), tol)
    steps, pf = int(g["steps"]), int(g["policy_freq"])
    for a in ids:
        assert agent.critic_1_optimizers[a].step == agent.critic_2_optimizers[a].step == steps
        assert agent.actor_optimizers[a].step == steps // pf and agent.learn_counter[a] == steps
    lr = {"actor": float(g["lr_actor"]), "critic": float(g["lr_critic"])}
    for tag, attr, kind in SETS:                      # tests/test_maddpg_gpu.py's bar
        for a in ids:
            sd = getattr(agent, attr)[a].state_dict()
            ref_sd = run["final"][tag][a]
            d = torch.cat([(sd[k].cpu() - ref).abs().reshape(-1) for k, ref in ref_sd.items()])
            r = torch.cat([ref.abs().reshape(-1) for ref in ref_sd.values()])
            tight = d <= 2e-3 * lr[kind] + 1e-5 * r
            assert float(d.max()) <= 3 * lr[kind], (tag, a, float(d.max()))
            assert float(tight.float().mean()) >= 0.995, (tag, a, float(tight.float().mean()), float(d.max()))


@pytest.mark.parametrize("use_graph", [False, True])
def test_critic_only_call_leaves_actors_and_targets_bitwise_unchanged(use_graph):
    g = load_golden("matd3_vector.npz")
    ids, agent = _agent(g)
    agent.use_graph = use_graph
    untouched = lambda: {k: v for k, v in _state(agent).items()
                         if isinstance(v, torch.Tensor) and (k.startswith(("actors/", "actor_targets/", "critic_targets_", "actor_optimizers/")))}
    before = untouched()
    out = agent.learn_device(_batch(g, 0, ids))
    assert torch.isnan(out[:, 0]).all() and torch.isfinite(out[:, 1]).all()          # the actor column is NaN, not stale
    _assert_same(before, untouched(), "critic-only")
    assert all(not torch.equal(agent.critics_1[a].buffers.params, agent.critic_targets_1[a].buffers.params) for a in ids)
    agent.learn(_batch(g, 1, ids))                                                     # a policy call moves all of them
    after = untouched()
    assert all(not torch.equal(before[k], after[k]) for k in before), [k for k in before if torch.equal(before[k], after[k])]


@pytest.mark.parametrize("mode", ["graph+streams", "eager+streams", "graph+serial"])
def test_graph_replay_and_side_streams_are_bit_identical_to_the_serial_eager_call(mode):
    g = load_golden("matd3_vector.npz")
    ids, ref = _agent(g)
    ref.use_graph, ref.concurrent_agents = False, False
    ids, alt = _agent(g)
    alt.use_graph, alt.concurrent_agents = mode.startswith("graph"), mode.endswith("streams")
    for st in range(int(g["steps"])):
        l_ref, l_alt = ref.learn(_batch(g, st, ids)), alt.learn(_batch(g, st, ids))
        assert l_ref == l_alt, (mode, st, l_ref, l_alt)
        _assert_same(_state(ref), _state(alt), (mode, st))
    if alt.use_graph:
        from agilerl_b200 import _lib
        plan = alt._plans[int(g["B"])]
        assert plan.graphs.get(True) is not None and plan.graphs.get(False) is not None
        n = {}
        for kind, gr in plan.graphs.items():
            c = ctypes.c_int(0)
            _lib.check(_lib.load().b2rl_graph_kernel_count(gr, ctypes.byref(c)))
            n[kind] = c.value
        assert n[True] < n[False], n


def test_workspace_sizes():
    from agilerl_b200 import _lib
    g = load_golden("matd3_vector.npz")
    ids, agent = _agent(g)
    lib = _lib.load()
    descs = ctypes.cast(agent._actor_descs, ctypes.c_void_p), ctypes.cast(agent._critic_descs, ctypes.c_void_p)
    old, cfg_sz = ctypes.c_size_t(), ctypes.c_size_t()
    cfg = _lib.MaddpgCfg()
    cfg.batch, cfg.n_agents = 64, len(ids)
    _lib.check(lib.b2rl_maddpg_workspace_bytes(*descs, len(ids), 64, ctypes.byref(old)))
    _lib.check(lib.b2rl_maddpg_workspace_bytes_cfg(*descs, ctypes.byref(cfg), ctypes.byref(cfg_sz)))
    assert old.value == cfg_sz.value                                    # twin = 0: MADDPG's size
    cfg.twin = 1
    _lib.check(lib.b2rl_maddpg_workspace_bytes_cfg(*descs, ctypes.byref(cfg), ctypes.byref(cfg_sz)))
    assert cfg_sz.value > old.value


def test_replay_gathers_into_captured_buffers_and_packed_equals_dict():
    from agilerl_b200.components import MultiAgentReplayBuffer
    g = load_golden("matd3_vector.npz")
    ids, a1 = _agent(g)
    a2 = a1.clone()
    a2.use_graph = False
    B = 16
    buf = MultiAgentReplayBuffer(64, list(FIELDS), ids, device="cuda")
    buf.save_to_memory(*tuple({a: d[a].numpy() for a in ids} for d in G.batch(g, 0)), is_vectorised=True)
    for _ in range(4):
        batch = buf.sample_device(B, out=a1.batch_buffers(B))
        assert batch[0].packed.data_ptr() == a1.batch_buffers(B)[0].data_ptr()
        plain = tuple({a: d[a].clone() for a in ids} for d in batch)
        assert a1.learn(batch) == a2.learn(plain)
    _assert_same(_state(a1), _state(a2))


def test_overlapped_population_learn_equals_member_by_member():
    from agilerl_b200.components import MultiAgentReplayBuffer
    from agilerl_b200.training.population import multi_agent_population_learn
    g = load_golden("matd3_vector.npz")
    ids, base = _agent(g)
    B = 16

    def run(overlap):
        torch.manual_seed(0)
        pop = [base.clone(index=k) for k in range(3)]
        for k, m in enumerate(pop):
            for a in ids:
                m.actors[a].buffers.params.mul_(1.0 + 0.01 * k)
        buf = MultiAgentReplayBuffer(64, list(FIELDS), ids, device="cuda")
        buf.save_to_memory(*tuple({a: d[a].numpy() for a in ids} for d in G.batch(g, 0)), is_vectorised=True)
        outs = []
        for _ in range(4):
            outs.append([o.clone() for o in multi_agent_population_learn(pop, buf, B, overlap=overlap)])
        torch.cuda.synchronize()
        return pop, outs
    p1, l1 = run(True)
    p2, l2 = run(False)
    for x, y in zip(l1, l2):
        for u, v in zip(x, y):
            assert torch.equal(torch.nan_to_num(u, nan=7.0), torch.nan_to_num(v, nan=7.0))
    for m1, m2 in zip(p1, p2):
        _assert_same(_state(m1), _state(m2))


def test_learn_at_bench_batch_matches_oracle():
    from oracle import maddpg as om
    from oracle.matd3 import OracleMATD3
    g = load_golden("matd3_vector.npz")
    ids, agent = _agent(g)
    B = 256
    a_hidden = [int(h) for h in g["a_hidden"]]
    a_specs = {a: om.actor_specs(int(o), int(d), head_hidden=a_hidden) for a, o, d in zip(ids, g["obs_dims"], g["act_dims"])}
    sds = {tag: {a: G.initial_sd(g, tag, a) for a in ids} for tag, _, _ in SETS}
    orc = OracleMATD3(ids, a_specs, om.critic_head_spec(int(g["act_dims"].sum()), head_hidden=a_hidden), sds["actor"],
                      sds["actor_target"], sds["critic_1"], sds["critic_target_1"], sds["critic_2"], sds["critic_target_2"],
                      gamma=float(g["gamma"]), tau=float(g["tau"]), lr_actor=float(g["lr_actor"]), lr_critic=float(g["lr_critic"]),
                      policy_freq=int(g["policy_freq"]))
    gen = torch.Generator().manual_seed(3)
    for _ in range(4):
        exp = ({a: torch.randn(B, int(o), generator=gen) for a, o in zip(ids, g["obs_dims"])},
               {a: torch.rand(B, int(d), generator=gen) * 2 - 1 for a, d in zip(ids, g["act_dims"])},
               {a: torch.randn(B, 1, generator=gen) for a in ids},
               {a: torch.randn(B, int(o), generator=gen) for a, o in zip(ids, g["obs_dims"])},
               {a: (torch.rand(B, 1, generator=gen) < 0.2).float() for a in ids})
        ref = orc.learn(tuple({a: v.clone() for a, v in d.items()} for d in exp))
        got = agent.learn(tuple({a: v.cuda() for a, v in d.items()} for d in exp))
        for a in ids:
            assert (got[a][0] is None) == (ref[a][0] is None)
            for j in range(2):
                if ref[a][j] is not None:
                    assert abs(got[a][j] - ref[a][j]) <= 1e-5 * max(1.0, abs(ref[a][j])), (a, j, got[a][j], ref[a][j])


@pytest.mark.parametrize("how", ["clone", "export_state", "checkpoint"])
def test_member_moved_at_odd_learn_counter_continues_bit_identically(how, tmp_path):
    from agilerl_b200.algorithms import MATD3
    g = load_golden("matd3_vector.npz")
    ids, src = _agent(g)
    for st in range(3):                                  # learn_counter 3: the next call is a policy call
        src.learn(_batch(g, st, ids))
    assert all(c == 3 for c in src.learn_counter.values())
    if how == "clone":
        moved = src.clone()
    elif how == "export_state":
        meta, tensors = src.export_state()
        moved = MATD3.from_state(pickle.loads(pickle.dumps(meta)), [t.clone() for t in tensors], src)
    else:
        path = str(tmp_path / "m.pt")
        src.save_checkpoint(path)
        moved = MATD3.load(path)
        _, other = _agent(g)
        other.load_checkpoint(path)
        _assert_same(_state(moved), _state(other), "load vs load_checkpoint")
    _assert_same(_state(src), _state(moved), how)
    assert moved.policy_freq == src.policy_freq
    for st in (3, 4):
        assert src.learn(_batch(g, st, ids)) == moved.learn(_batch(g, st, ids))
        _assert_same(_state(src), _state(moved), (how, st))


def test_tournament_and_device_parameter_mutation():
    from agilerl_b200.hpo import Mutations, TournamentSelection
    g = load_golden("matd3_vector.npz")
    ids, base = _agent(g)
    pop = [base.clone(index=k) for k in range(4)]
    for k, m in enumerate(pop):
        m.fitness = [float(k)]
        m.learn(_batch(g, 0, ids))
    np.random.seed(0)
    elite, new_pop = TournamentSelection(2, True, 4, 1).select(pop)
    assert elite.index == 3 and len(new_pop) == 4 and all(type(m) is type(base) for m in new_pop)
    assert torch.equal(new_pop[0].critics_2[ids[0]].buffers.params, pop[3].critics_2[ids[0]].buffers.params)
    assert new_pop[0].learn_counter == pop[3].learn_counter
    m = Mutations(0, 0, 0.5, 1, 0, 0, rand_seed=1, device="cuda")
    m.device_parameter_mutation = True
    clone = new_pop[1]
    before = {a: clone.actors[a].buffers.params.clone() for a in ids}
    [mutated] = m.mutation([clone])
    assert mutated.mut == "param"
    for a in ids:
        p = mutated.actors[a].buffers.params
        assert not torch.equal(p, before[a]) and torch.isfinite(p).all()
        assert torch.equal(mutated.actor_targets[a].buffers.params, p)
    losses = mutated.learn(_batch(g, 1, ids))
    assert all(v is not None and np.isfinite(v) for pair in losses.values() for v in pair)
