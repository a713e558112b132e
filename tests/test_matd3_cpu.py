"""CPU: MATD3's host side and its oracle.

* The oracle (oracle/matd3.py) reproduces the reference's five recorded learn calls (tests/golden/matd3_vector.npz, read by
  tests/_matd3_golden.py) bit for bit: losses, ``None`` actor losses, the digests of the recorded gradients and of every
  final parameter of the six network sets.
* The constructor signature, defaults and public methods are the reference's (tests/golden/matd3_api.json).
* ``create_population("MATD3")`` maps ``POLICY_FREQ``.
* With a Python stand-in for ``b2rl_maddpg_learn`` (tests/_matd3_standin.py): the step-kind sequence, the ``twin`` /
  ``critic_only`` flags, ``(None, critic_loss)`` returns, the separate actor / critic Adam step counts and bias
  corrections, and what clone / export_state / checkpoints carry."""
import inspect
import json
import os
import pickle

import numpy as np
import pytest
import torch

import _matd3_golden as G
from conftest import load_golden

HERE = os.path.dirname(os.path.abspath(__file__))
FIELDS = ("obs", "action", "reward", "next_obs", "done")
SETS = (("actor", "actors"), ("actor_target", "actor_targets"), ("critic_1", "critics_1"), ("critic_target_1", "critic_targets_1"),
        ("critic_2", "critics_2"), ("critic_target_2", "critic_targets_2"))


def _batch(g, st, ids):
    return G.batch(g, st)


def test_oracle_reproduces_the_reference_bit_for_bit():
    g = load_golden("matd3_vector.npz")
    ids = G.ids_of(g)
    run = G.oracle_run(g)
    for st in range(int(g["steps"])):
        out = run["losses"][st]
        for a in ids:
            none = bool(g[f"s{st}_actor_none/{a}"])
            assert (out[a][0] is None) == none, (st, a)
            if not none:
                assert out[a][0] == float(g[f"s{st}_actor_loss/{a}"]), (st, a)
            assert out[a][1] == float(g[f"s{st}_critic_loss/{a}"]), (st, a)
    sha = G.digests(g)
    grads = [k for k in sha if k.startswith("s")]
    finals = [k for k in sha if not k.startswith("s")]
    assert len(finals) == sum(len(G.initial_sd(g, tag, a)) for tag in G.ONLINE for a in ids)      # every final parameter
    assert {k.split("/")[0] for k in grads} == {"s0_grad", "s1_grad"}
    for k in grads:
        st = int(k[1:k.index("_")])
        assert G.digest(run["grads"][st][k[k.index("/") + 1:]]) == sha[k], k
    for k in finals:
        tag1, a, key = k.split("/", 2)
        assert G.digest(run["final"][tag1[:-1]][a][key]) == sha[k], k


def test_constructor_defaults_and_methods_are_the_references():
    from agilerl_b200.algorithms import MATD3
    with open(os.path.join(HERE, "golden", "matd3_api.json")) as f:
        api = json.load(f)
    params = [p for p in inspect.signature(MATD3.__init__).parameters if p != "self"]
    assert params == api["ctor"]
    ours = {n: p.default for n, p in inspect.signature(MATD3.__init__).parameters.items()
            if n not in ("self", "device") and p.default is not inspect.Parameter.empty}
    assert ours == api["defaults"]
    # learn_individual / process_infos are per-agent internals of the reference's learn / get_action; here one fused call
    for name, ref_params in api["methods"].items():
        if name in ("learn_individual", "process_infos"):
            continue
        assert [p for p in inspect.signature(getattr(MATD3, name)).parameters if p != "self"] == ref_params, name


@pytest.fixture
def standin(monkeypatch):
    from agilerl_b200 import _lib
    from agilerl_b200.components import replay_buffer as rb
    from _matd3_standin import Matd3StandIn
    lib = Matd3StandIn()
    monkeypatch.setattr(_lib, "as_device", lambda d: torch.device("cpu"))
    monkeypatch.setattr(_lib, "load", lambda require_cuda=False: lib)
    monkeypatch.setattr(_lib, "stream_ptr", lambda d=None: 0)
    monkeypatch.setattr(_lib, "check", lambda rc: None)
    monkeypatch.setattr(torch.Tensor, "pin_memory", lambda self: self)
    monkeypatch.setattr(rb._PinnedRing, "sent", lambda self, k, dev: None)
    return lib


def _member(policy_freq=2):
    from agilerl_b200.algorithms import MATD3
    from agilerl_b200.compat import spaces
    g = load_golden("matd3_vector.npz")
    ids = [str(a) for a in g["agent_ids"]]
    agent = MATD3([spaces.Box(-1.0, 1.0, (int(d),), np.float32) for d in g["obs_dims"]],
                  [spaces.Box(-1.0, 1.0, (int(d),), np.float32) for d in g["act_dims"]], agent_ids=ids, batch_size=int(g["B"]),
                  policy_freq=policy_freq)
    agent.use_graph = False
    return g, ids, agent


def test_step_kinds_flags_returns_and_separate_step_counts(standin):
    g, ids, agent = _member(policy_freq=3)
    assert agent.algo == "MATD3" and not hasattr(agent, "critics") and agent.learn_counter == {a: 0 for a in ids}
    kinds = []
    for st in range(7):
        losses = agent.learn(_batch(g, st % 5, ids))
        c = standin.calls[-1]
        kinds.append(c["critic_only"])
        assert c["twin"] == 1 and c["step_state"] is None and c["actor_step_state"] is None
        for i, a in enumerate(ids):
            assert losses[a][1] == i + 0.5
            assert losses[a][0] is None if c["critic_only"] else losses[a][0] == -i - 1.0
            assert c["critic2"][i] == agent.critics_2[a].buffers.params.data_ptr()
            assert c["critic2_target"][i] == agent.critic_targets_2[a].buffers.params.data_ptr()
            assert c["critic2_m"][i] == agent.critic_2_optimizers[a].exp_avg.data_ptr()
        n_crit, n_act = st + 1, (st + 1) // 3
        assert c["bc1_critic"] == 1.0 - 0.9 ** n_crit and c["bc2_critic"] == 1.0 - 0.999 ** n_crit
        if not c["critic_only"]:
            assert c["bc1_actor"] == 1.0 - 0.9 ** n_act and c["bc2_actor"] == 1.0 - 0.999 ** n_act
        for a in ids:
            assert agent.critic_1_optimizers[a].step == agent.critic_2_optimizers[a].step == n_crit
            assert agent.actor_optimizers[a].step == n_act and agent.learn_counter[a] == n_crit
    assert kinds == [1, 1, 0, 1, 1, 0, 1]
    out = agent.learn_device(_batch(g, 0, ids))           # the device result: the actor column NaN on a critic-only call
    assert torch.isnan(out[:, 0]).all()


def test_moves_carry_both_step_counts_and_the_counter_dict(standin, tmp_path):
    from agilerl_b200.algorithms import MATD3
    g, ids, agent = _member()
    for st in range(3):
        agent.learn(_batch(g, st, ids))
    agent.lr_critic = 0.005
    meta, tensors = agent.export_state()
    assert len(tensors) == 12 * len(ids)
    moved = [agent.clone(), MATD3.from_state(pickle.loads(pickle.dumps(meta)), [t.clone() for t in tensors], agent)]
    path = str(tmp_path / "m.pt")
    agent.save_checkpoint(path)
    moved.append(MATD3.load(path, device="cuda"))
    _, _, fresh = _member()
    fresh.load_checkpoint(path)
    moved.append(fresh)
    for m in moved:
        assert m.learn_counter == {a: 3 for a in ids} and m.learn_counter is not agent.learn_counter
        assert m.policy_freq == 2 and m.lr_critic == 0.005
        for a in ids:
            assert m.actor_optimizers[a].step == 1 and m.critic_1_optimizers[a].step == m.critic_2_optimizers[a].step == 3
            for _, attr in SETS:
                assert torch.equal(getattr(m, attr)[a].buffers.params, getattr(agent, attr)[a].buffers.params)
            assert torch.equal(m.critic_2_optimizers[a].exp_avg_sq, agent.critic_2_optimizers[a].exp_avg_sq)
        m.use_graph = False
        standin.calls.clear()
        m.learn(_batch(g, 3, ids))
        assert standin.calls[-1]["critic_only"] == 0 and standin.calls[-1]["bc1_actor"] == 1.0 - 0.9 ** 2


def test_changing_policy_freq_drops_the_captured_plans(standin):
    g, ids, agent = _member()
    agent._plans = {64: type("P", (), {"destroy": lambda self: None})()}
    agent.policy_freq = 3
    assert agent._plans == {}


def test_create_population_maps_policy_freq(standin):
    from agilerl_b200.compat import spaces
    from agilerl_b200.utils.utils import create_population
    ids = ["a", "b"]
    osp, asp = [spaces.Box(-1.0, 1.0, (6,), np.float32)] * 2, [spaces.Box(-1.0, 1.0, (3,), np.float32)] * 2
    pop = create_population("MATD3", osp, asp, None, {"AGENT_IDS": ids, "BATCH_SIZE": 32, "POLICY_FREQ": 3}, population_size=2,
                            num_envs=4, first_index=2)
    assert [m.index for m in pop] == [2, 3] and all(m.algo == "MATD3" for m in pop)
    m = pop[0]
    assert (m.policy_freq, m.batch_size, m.gamma, m.tau, m.lr_actor, m.lr_critic, m.vect_noise_dim) == (3, 32, 0.95, 0.01, 1e-4, 1e-3, 4)
    [d] = create_population("MATD3", osp, asp, None, {"AGENT_IDS": ids})
    assert d.policy_freq == 2
    with pytest.raises(NotImplementedError):
        create_population("MATD3", osp, asp, None, {"AGENT_IDS": ids, "SHARE_ENCODERS": True})


def test_parameter_and_rl_hyperparameter_mutations_and_tournament(standin):
    from agilerl_b200.hpo import Mutations, TournamentSelection
    g, ids, agent = _member()
    pop = [agent.clone(index=k) for k in range(3)]
    for k, m in enumerate(pop):
        m.fitness = [float(k)]
    np.random.seed(0)
    elite, new_pop = TournamentSelection(2, True, 3, 1).select(pop)
    assert elite.index == 2 and all(type(m) is type(agent) for m in new_pop)
    mut = Mutations(0, 0, 0, 1, 0, 0, rand_seed=1, device="cuda")
    before = {a: new_pop[1].actors[a].buffers.params.clone() for a in ids}
    [m1] = mut.mutation([new_pop[1]])
    assert m1.mut == "param" and any(not torch.equal(m1.actors[a].buffers.params, before[a]) for a in ids)
    assert all(torch.equal(m1.actor_targets[a].buffers.params, m1.actors[a].buffers.params) for a in ids)
    from agilerl_b200.algorithms.core.registry import HyperparameterConfig, RLParameter
    hp = HyperparameterConfig(lr_actor=RLParameter(min=1e-5, max=1e-2), lr_critic=RLParameter(min=1e-5, max=1e-2),
                              batch_size=RLParameter(min=8, max=512, dtype=int))
    from agilerl_b200.compat import spaces
    c = type(agent)([spaces.Box(-1.0, 1.0, (6,), np.float32)] * 2, [spaces.Box(-1.0, 1.0, (3,), np.float32)] * 2, agent_ids=["a", "b"],
                    hp_config=hp)
    c.use_graph = False
    for o in c._all_opts:
        o.step = 5
    rl = Mutations(0, 0, 0.5, 0, 0, 1, rand_seed=4, device="cuda")
    seen = set()
    for _ in range(12):
        [c] = rl.mutation([c])
        seen.add(c.mut)
        assert c.mut in ("lr_actor", "lr_critic", "batch_size")
        if c.mut.startswith("lr"):                       # reinit_optimizers: fresh Adam state of all three optimiser sets
            assert all(o.step == 0 for o in c._all_opts) and len(c._all_opts) == 6
            assert c.critic_2_optimizers["b"].lr == c.lr_critic and c.actor_optimizers["a"].lr == c.lr_actor
    assert len(seen) >= 2
    with pytest.raises(NotImplementedError):
        Mutations(0, 1, 0.5, 0, 0, 0, rand_seed=2, device="cuda").mutation([c])
