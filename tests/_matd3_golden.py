"""Reader of tests/golden/matd3_vector.npz (written by tests/golden/make_golden_matd3.py), shared by the MATD3 tests.

The fixture holds no parameter tensors.  The initial networks are seeded draws (``init_sd``: per state_dict entry ones,
zeros or a uniform(-bound, bound) draw from a ``torch.Generator``, targets as copies of their online network) loaded into
the reference before its run; the five input batches are seeded draws too (``matd3_batch``).  Both are checked against
the SHA-256 of what the reference started from and was fed.  Stored as values: the per-call losses and which actor
losses were ``None``.  Stored as SHA-256 digests of their float32 bytes: the reference's gradients and the final
parameters of all six network sets.  ``oracle_run`` recomputes those tensors with the oracle (oracle/matd3.py);
tests/test_matd3_cpu.py requires every digest to match (the oracle reproduces the reference bit for bit), and the GPU
tests compare against the recomputed tensors."""
import hashlib

import numpy as np
import torch

FIELDS = ("obs", "action", "reward", "next_obs", "done")
ONLINE = {"actor": "actor", "actor_target": "actor", "critic_1": "critic_1", "critic_target_1": "critic_1",
          "critic_2": "critic_2", "critic_target_2": "critic_2"}


def digest(x) -> str:
    a = x.detach().cpu().numpy() if isinstance(x, torch.Tensor) else np.asarray(x)
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.float32).tobytes()).hexdigest()


def matd3_batch(seed: int, ids, obs_dims, act_dims, B: int, with_nan: bool):
    """One learn call's (states, actions, rewards, next_states, dones) dicts; ``with_nan``: an agent that was not alive
    (NaN reward / done) in two rows."""
    g = torch.Generator().manual_seed(seed)
    st = {a: torch.randn(B, o, generator=g) for a, o in zip(ids, obs_dims)}
    ac = {a: torch.rand(B, d, generator=g) * 2 - 1 for a, d in zip(ids, act_dims)}
    rw = {a: torch.randn(B, 1, generator=g) for a in ids}
    ns = {a: torch.randn(B, o, generator=g) for a, o in zip(ids, obs_dims)}
    dn = {a: (torch.rand(B, 1, generator=g) < 0.2).float() for a in ids}
    if with_nan:
        rw[ids[1]][3, 0] = float("nan")
        dn[ids[1]][3, 0] = float("nan")
        dn[ids[2]][7, 0] = float("nan")
    return st, ac, rw, ns, dn


def batch_digest(batch, ids) -> str:
    h = hashlib.sha256()
    for d in batch:
        for a in ids:
            h.update(np.ascontiguousarray(d[a].numpy(), dtype=np.float32).tobytes())
    return h.hexdigest()


def ids_of(g):
    return [str(a) for a in g["agent_ids"]]


def batch(g, st: int, device=None):
    """The ``st``-th input batch, checked against the digest of what the reference was fed."""
    ids = ids_of(g)
    b = matd3_batch(int(g["seed0"]) + st, ids, [int(d) for d in g["obs_dims"]], [int(d) for d in g["act_dims"]], int(g["B"]),
                    st == int(g["nan_call"]))
    assert batch_digest(b, ids) == str(g[f"s{st}_inputs_sha256"]), f"torch.Generator draws differ from the recorded batch {st}"
    return b if device is None else tuple({a: v.to(device) for a, v in d.items()} for d in b)


def init_sd(spec, seed: int) -> dict:
    """A state_dict from ``spec`` = [(key, shape, kind, bound)]: kind "ones" / "zeros", else uniform(-bound, bound) drawn
    in key order from ``torch.Generator().manual_seed(seed)``."""
    gen = torch.Generator().manual_seed(seed)
    out = {}
    for key, shape, kind, bound in spec:
        if kind == "ones":
            out[key] = torch.ones(shape)
        elif kind == "zeros":
            out[key] = torch.zeros(shape)
        else:
            out[key] = torch.empty(shape).uniform_(-bound, bound, generator=gen)
    return out


def init_seed(g, tag: str, agent_index: int) -> int:
    return int(g["init_seed"]) + 100 * ("actor", "critic_1", "critic_2").index(ONLINE[tag]) + agent_index


def init_spec(g, tag: str):
    t = ONLINE[tag]
    shapes = [tuple(int(x) for x in str(s).split("x")) if str(s) else () for s in g[f"init_shapes/{t}"]]
    return [(str(k), sh, str(kind), float(b)) for k, sh, kind, b in zip(g[f"init_keys/{t}"], shapes, g[f"init_kinds/{t}"],
                                                                      g[f"init_bounds/{t}"])]


def initial_sd(g, tag: str, agent: str) -> dict:
    """The initial state_dict of network set ``tag`` the reference started from (targets: copies of their online network),
    checked against its recorded digest."""
    ids = ids_of(g)
    sd = init_sd(init_spec(g, tag), init_seed(g, tag, ids.index(agent)))
    assert sd_digest(sd) == str(g[f"init_sha256/{ONLINE[tag]}/{agent}"]), f"torch.Generator draws differ from the recorded {tag}"
    return sd


def sd_digest(sd) -> str:
    h = hashlib.sha256()
    for v in sd.values():
        h.update(np.ascontiguousarray(v.detach().cpu().numpy(), dtype=np.float32).tobytes())
    return h.hexdigest()


def digests(g) -> dict:
    """{name: SHA-256} of the reference's gradients (``s{call}_grad/{set}/{agent}/{key}``) and final parameters
    (``{set}1/{agent}/{key}``)."""
    return dict(zip((str(k) for k in g["sha256_keys"]), (v.decode() if isinstance(v, bytes) else str(v) for v in g["sha256_values"])))


_RUNS: dict = {}


def oracle_run(g):
    """The oracle over the recorded calls from the recorded initial state (one CPU thread, as when recording):
    ``{"losses": [per call {agent: (actor | None, critic)}], "grads": [per call {name: tensor}], "final": {tag: {agent: sd}}}``."""
    key = str(g["s0_inputs_sha256"])
    if key in _RUNS:
        return _RUNS[key]
    from oracle import maddpg as om
    from oracle.matd3 import OracleMATD3
    ids = ids_of(g)
    a_hidden, c_hidden = [int(h) for h in g["a_hidden"]], [int(h) for h in g["c_hidden"]]
    a_specs = {a: om.actor_specs(int(o), int(d), head_hidden=a_hidden) for a, o, d in zip(ids, g["obs_dims"], g["act_dims"])}
    sds = {tag: {a: initial_sd(g, tag, a) for a in ids} for tag in ONLINE}
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        orc = OracleMATD3(ids, a_specs, om.critic_head_spec(int(g["act_dims"].sum()), head_hidden=c_hidden), sds["actor"],
                          sds["actor_target"], sds["critic_1"], sds["critic_target_1"], sds["critic_2"], sds["critic_target_2"],
                          gamma=float(g["gamma"]), tau=float(g["tau"]), lr_actor=float(g["lr_actor"]),
                          lr_critic=float(g["lr_critic"]), policy_freq=int(g["policy_freq"]))
        losses, grads = [], []
        for st in range(int(g["steps"])):
            losses.append(orc.learn(batch(g, st)))
            grads.append(dict(orc.last_grads))
    finally:
        torch.set_num_threads(threads)
    nets = dict(actor=orc.actors, actor_target=orc.actor_targets, critic_1=orc.critics_1, critic_target_1=orc.critic_targets_1,
                critic_2=orc.critics_2, critic_target_2=orc.critic_targets_2)
    final = {tag: {a: {k: v.detach().clone() for k, v in nets[tag][a].items()} for a in ids} for tag in ONLINE}
    _RUNS[key] = {"losses": losses, "grads": grads, "final": final}
    return _RUNS[key]
