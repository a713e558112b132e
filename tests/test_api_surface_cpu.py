"""CPU: static drop-in check against the UNMODIFIED reference (AgileRL 2.6.1): constructor parameters and public methods of
every replaced class must be present with the same names (and order for constructors).  The reference's signatures are
stored in tests/golden/api_surface.json (``python tests/golden/make_golden.py api_surface`` reads them from the reference)."""
import inspect
import json
import os

import pytest

from conftest import GOLDEN


@pytest.fixture(scope="module")
def ref():
    with open(os.path.join(GOLDEN, "api_surface.json")) as f:
        return json.load(f)


def _ctor(cls):
    return [p for p in inspect.signature(cls.__init__).parameters if p != "self"]


def _public(cls):
    return {n for n, m in inspect.getmembers(cls) if not n.startswith("_") and (inspect.isfunction(m) or isinstance(m, property))}


def test_constructors_and_methods_match(ref):
    import agilerl_b200.algorithms as a
    import agilerl_b200.components as c
    import agilerl_b200.hpo as h
    ours = [c.ReplayBuffer, c.MultiStepReplayBuffer, c.PrioritizedReplayBuffer, a.RainbowDQN, a.DQN, h.TournamentSelection,
            h.Mutations, c.SumSegmentTree, c.MinSegmentTree]
    for m in ours:
        rc, mc = ref["ctor"][m.__name__], _ctor(m)
        assert mc[:len(rc)] == rc or set(rc) <= set(mc), f"{m.__name__}: ctor {rc} vs {mc}"
    need = {
        c.ReplayBuffer: {"add", "sample", "clear", "storage", "size", "is_full"},
        c.MultiStepReplayBuffer: {"add", "sample_from_indices"},
        c.PrioritizedReplayBuffer: {"add", "sample", "update_priorities"},
        a.RainbowDQN: {"learn", "get_action", "test", "soft_update", "clone", "save_checkpoint", "load_checkpoint"},
        a.DQN: {"learn", "get_action", "test", "soft_update", "clone"},
        h.TournamentSelection: {"select"}, h.Mutations: {"mutation", "no_mutation", "architecture_mutate",
                                                         "parameter_mutation", "activation_mutation",
                                                         "rl_hyperparam_mutation"},
    }
    for cls, names in need.items():
        assert names <= _public(cls) | set(dir(cls)), f"{cls.__name__} lacks {names - set(dir(cls))}"


def test_reference_defaults_match(ref):
    import agilerl_b200.algorithms as a
    for m in (a.RainbowDQN, a.DQN):
        ms = inspect.signature(m.__init__).parameters
        for name, default in ref["defaults"][m.__name__].items():
            assert ms[name].default == default, f"{m.__name__}.{name}: {ms[name].default} != {default}"


def test_driver_signature_matches(ref):
    from agilerl_b200.training import train_off_policy as mine
    rs = ref["train_off_policy"]
    ms = list(inspect.signature(mine).parameters)
    assert ms[:len(rs)] == rs, (rs, ms)


def test_multi_agent_surface_matches(ref):
    """MADDPG / MultiAgentReplayBuffer (SURVEY 8f-4): same constructor parameters in the same order with the same
    defaults (``device`` aside), same public methods of the replay and the learner's hot-path methods."""
    import agilerl_b200.algorithms as a
    import agilerl_b200.components as c
    assert _ctor(a.MADDPG) == ref["ctor"]["MADDPG"]
    assert _ctor(c.MultiAgentReplayBuffer) == ref["ctor"]["MultiAgentReplayBuffer"]
    ms = inspect.signature(a.MADDPG.__init__).parameters
    for name, default in ref["defaults"]["MADDPG"].items():
        assert ms[name].default == default, f"MADDPG.{name}: {ms[name].default} != {default}"
    for name, r_sig in ref["multi_agent_buffer_methods"].items():
        m_sig = [p for p in inspect.signature(getattr(c.MultiAgentReplayBuffer, name)).parameters if p != "self"]
        assert m_sig[:len(r_sig)] == r_sig, (name, r_sig, m_sig)
    assert {"learn", "get_action", "action_noise", "reset_action_noise", "soft_update", "test", "clone"} <= set(dir(a.MADDPG))
