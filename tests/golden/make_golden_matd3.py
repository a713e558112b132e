"""Generate the MATD3 golden data by running the UNMODIFIED reference (AgileRL 2.6.1) through ``oracle.refshim`` and
check the oracle restatement (``oracle/matd3.py``) against it while doing so.  Same conventions as ``make_golden.py``,
whose fixtures this script does not touch; what ``matd3_vector.npz`` holds and how the tests read it:
``tests/_matd3_golden.py``.

    python tests/golden/make_golden_matd3.py           # matd3_vector.npz and matd3_api.json
    python tests/golden/make_golden_matd3.py matd3     # the same

The reference's own ``MATD3.learn`` (DeterministicActor + the EvolvableMultiInput critics) runs; ``tensordict`` and
``gymnasium.spaces`` are the stand-ins of ``agilerl_b200.compat``.
"""
from __future__ import annotations

import inspect
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from oracle import refshim  # noqa: E402

refshim.install()

from gymnasium import spaces  # noqa: E402


def save(name, **arrays):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **arrays)
    print(f"wrote {name}: {os.path.getsize(path) / 1024:.1f} KiB")


def sd_np(sd):
    return {k: v.detach().cpu().numpy().copy() for k, v in sd.items()}


GROUPS = ("actor", "actor_target", "critic_1", "critic_target_1", "critic_2", "critic_target_2")
REF_ATTR = dict(actor="actors", actor_target="actor_targets", critic_1="critics_1", critic_target_1="critic_targets_1",
                critic_2="critics_2", critic_target_2="critic_targets_2")


def float64_losses(spec_sds, ids, a_specs, c_head, batches, **kw):
    """The oracle's losses in float64 from the same initial state and inputs: how far fp32 rounding alone moves them."""
    import torch.nn.functional as F
    import oracle.matd3 as M
    from oracle import nets as onets
    saved = M.actor_forward, M.critic_forward

    def critic64(sd, head, obs_list, acts):
        lat = F.relu(F.linear(torch.cat(obs_list, dim=1), sd["encoder.final_dense.weight"], sd["encoder.final_dense.bias"]))
        return onets.mlp_forward(sd, head, torch.cat([lat, acts], dim=-1))
    M.actor_forward = lambda sd, specs, obs: onets.mlp_forward(sd, specs[1], onets.mlp_forward(sd, specs[0], obs))
    M.critic_forward = critic64
    try:
        d = {t: {a: {k: v.double() for k, v in spec_sds[t][a].items()} for a in ids} for t in GROUPS}
        orc = M.OracleMATD3(ids, a_specs, c_head, d["actor"], d["actor_target"], d["critic_1"], d["critic_target_1"], d["critic_2"],
                            d["critic_target_2"], **kw)
        return [orc.learn(tuple({a: v.double() for a, v in f.items()} for f in b)) for b in batches]
    finally:
        M.actor_forward, M.critic_forward = saved


def gen_matd3():
    """MATD3.learn (matd3.py:630-846) on BASELINE config 5's shapes (4 agents x 18-dim observations, 5-dim actions), B = 32,
    policy_freq = 2: five consecutive learn calls of the UNMODIFIED reference (calls 2 and 4 step the actors and the
    targets), oracle == reference bit for bit (losses, ``None`` actor losses, every gradient, every parameter of the six
    network sets).  A NaN reward and a NaN done (an agent that was not alive) ride in the second batch.

    The reference's networks are loaded with seeded draws before the run (``init_sd``: its LayerNorm ones / zeros kept,
    every other entry uniform within the largest magnitude of the reference's own initial values), targets as copies.
    Stored (tests/_matd3_golden.py reads it): that initialisation spec and the digests of the initial networks, per-call
    losses (``actor_none`` marks ``None``), the SHA-256 of each input batch (seeded ``torch.Generator`` draws, regenerated
    by the tests), and SHA-256 digests of the reference's critic_1 / critic_2 gradients of call 1, actor gradients of the
    first policy call (call 2) and final parameters of all six sets — the oracle recomputes those tensors and must hit
    every digest.  No parameter tensor is stored.

    The fixture's bars (losses within 1e-5 between two fp32 implementations) only mean something where fp32 rounding alone
    moves the losses far less than that: Adam's first steps move every parameter by about lr whatever the size of its
    gradient, so an element whose gradient nearly cancels over the batch can take either sign.  The initialisation seed is
    the first from ``init_seed`` whose float64 oracle run stays within ``max_rel_fp64`` of the float32 reference on every
    loss of the five calls."""
    from agilerl.algorithms.matd3 import MATD3
    from oracle import maddpg as om
    from oracle.matd3 import OracleMATD3
    from _matd3_golden import batch_digest, digest, init_sd, matd3_batch, sd_digest
    ids = [f"agent_{i}" for i in range(4)]
    obs_dims, act_dims = [18, 18, 18, 18], [5, 5, 5, 5]
    obs_spaces = [spaces.Box(-1, 1, (d,), np.float32) for d in obs_dims]
    act_spaces = [spaces.Box(-1, 1, (d,), np.float32) for d in act_dims]
    B, steps, policy_freq, seed0, nan_call, init_seed = 32, 5, 2, 90, 1, 1300
    torch.manual_seed(13)
    ref = MATD3(obs_spaces, act_spaces, agent_ids=ids, batch_size=B, policy_freq=policy_freq, device="cpu")
    a_hidden = list(ref.actors[ids[0]].head_net.net_config["hidden_size"])
    c_hidden = list(ref.critics_1[ids[0]].head_net.net_config["hidden_size"])
    a_specs = {a: om.actor_specs(o, d, head_hidden=a_hidden) for a, o, d in zip(ids, obs_dims, act_dims)}
    c_head = om.critic_head_spec(sum(act_dims), head_hidden=c_hidden)
    out = {"B": B, "steps": steps, "policy_freq": policy_freq, "seed0": seed0, "nan_call": nan_call, "init_seed": init_seed, "agent_ids": np.array(ids),
           "obs_dims": np.array(obs_dims), "act_dims": np.array(act_dims), "a_hidden": np.array(a_hidden),
           "c_hidden": np.array(c_hidden), "gamma": ref.gamma, "tau": ref.tau, "lr_actor": ref.lr_actor, "lr_critic": ref.lr_critic}
    specs = {}
    for online in ("actor", "critic_1", "critic_2"):
        spec = []
        for k, v in getattr(ref, REF_ATTR[online])[ids[0]].state_dict().items():
            kind = "ones" if bool((v == 1).all()) else "zeros" if bool((v == 0).all()) else "uniform"
            bound = float(np.float32(max(float(getattr(ref, REF_ATTR[online])[a].state_dict()[k].abs().max()) for a in ids)))
            spec.append((k, tuple(v.shape), kind, bound))
        specs[online] = spec
    batches = [matd3_batch(seed0 + s_, ids, obs_dims, act_dims, B, s_ == nan_call) for s_ in range(steps)]
    hp = dict(gamma=ref.gamma, tau=ref.tau, lr_actor=ref.lr_actor, lr_critic=ref.lr_critic, policy_freq=policy_freq)
    max_rel_fp64 = 2e-6

    def init_state(seed):
        pairs = (("actor", "actor_target"), ("critic_1", "critic_target_1"), ("critic_2", "critic_target_2"))
        return {name: {a: init_sd(specs[online], seed + 100 * t + i) for i, a in enumerate(ids)}
                for t, (online, target) in enumerate(pairs) for name in (online, target)}

    def rel_fp64(seed):
        st0 = init_state(seed)
        o32 = OracleMATD3(ids, a_specs, c_head, *(st0[n] for n in ("actor", "actor_target", "critic_1", "critic_target_1",
                                                                    "critic_2", "critic_target_2")), **hp)
        l32 = [o32.learn(b) for b in [matd3_batch(seed0 + s_, ids, obs_dims, act_dims, B, s_ == nan_call) for s_ in range(steps)]]
        l64 = float64_losses(st0, ids, a_specs, c_head, batches, **hp)
        return max(abs(x64 / x32 - 1.0) for r32, r64 in zip(l32, l64) for a in ids
                   for x32, x64 in zip(r32[a], r64[a]) if x32 is not None)
    while (rel := rel_fp64(init_seed)) > max_rel_fp64:
        print(f"  init seed {init_seed}: fp32 vs fp64 losses differ by {rel:.2e} relative; next seed")
        init_seed += 1000
    out["init_seed"], out["max_rel_fp64"] = init_seed, max_rel_fp64
    for t, (online, target) in enumerate((("actor", "actor_target"), ("critic_1", "critic_target_1"), ("critic_2", "critic_target_2"))):
        spec = specs[online]
        out[f"init_keys/{online}"] = np.array([k for k, _, _, _ in spec])
        out[f"init_shapes/{online}"] = np.array(["x".join(str(x) for x in sh) for _, sh, _, _ in spec])
        out[f"init_kinds/{online}"] = np.array([kind for _, _, kind, _ in spec])
        out[f"init_bounds/{online}"] = np.array([b for _, _, _, b in spec])
        for i, a in enumerate(ids):
            sd = init_sd(spec, init_seed + 100 * t + i)
            for attr in (REF_ATTR[online], REF_ATTR[target]):
                getattr(ref, attr)[a].load_state_dict(sd)
            out[f"init_sha256/{online}/{a}"] = sd_digest(sd)
    sds = {g: {a: getattr(ref, REF_ATTR[g])[a].state_dict() for a in ids} for g in GROUPS}
    orc = OracleMATD3(ids, a_specs, c_head, sds["actor"], sds["actor_target"], sds["critic_1"], sds["critic_target_1"],
                      sds["critic_2"], sds["critic_target_2"], gamma=ref.gamma, tau=ref.tau, lr_actor=ref.lr_actor,
                      lr_critic=ref.lr_critic, policy_freq=policy_freq)
    ref_params = {g: {a: dict(getattr(ref, REF_ATTR[g])[a].named_parameters()) for a in ids} for g in ("actor", "critic_1", "critic_2")}

    sha = {}

    def grads_of(groups):
        return {f"{g}/{a}/{k}": p.grad.detach().clone() for g in groups for a in ids for k, p in ref_params[g][a].items()}

    for s_ in range(steps):
        e_ref = matd3_batch(seed0 + s_, ids, obs_dims, act_dims, B, s_ == nan_call)
        e_orc = matd3_batch(seed0 + s_, ids, obs_dims, act_dims, B, s_ == nan_call)
        out[f"s{s_}_inputs_sha256"] = batch_digest(e_ref, ids)
        r_loss = ref.learn(e_ref)
        o_loss = orc.learn(e_orc)
        for a in ids:
            assert tuple(r_loss[a]) == tuple(o_loss[a]), (s_, a, r_loss[a], o_loss[a])
            actor_loss, critic_loss = r_loss[a]
            out[f"s{s_}_actor_none/{a}"] = actor_loss is None
            out[f"s{s_}_actor_loss/{a}"] = np.nan if actor_loss is None else actor_loss
            out[f"s{s_}_critic_loss/{a}"] = critic_loss
        assert ref.learn_counter == orc.learn_counter
        groups = {0: ("critic_1", "critic_2"), 1: ("actor",)}.get(s_, ())
        for k, v in grads_of(groups).items():           # the reference's own .grad tensors, equal to the oracle's
            assert torch.equal(v, orc.last_grads[k]), (s_, k)
            sha[f"s{s_}_grad/{k}"] = digest(v)
        if s_ == nan_call:
            assert all(r_loss[a][0] is not None for a in ids)
    onets = {"actor": orc.actors, "actor_target": orc.actor_targets, "critic_1": orc.critics_1,
             "critic_target_1": orc.critic_targets_1, "critic_2": orc.critics_2, "critic_target_2": orc.critic_targets_2}
    for gname in GROUPS:
        for a in ids:
            sd = getattr(ref, REF_ATTR[gname])[a].state_dict()
            for k, v in sd.items():
                assert torch.equal(v, onets[gname][a][k].data), (gname, a, k)
                sha[f"{gname}1/{a}/{k}"] = digest(v)
    for a in ids:                      # Adam step counts: critics every call, actors on the two policy calls
        assert ref.critic_1_optimizers.optimizer[a].state[next(iter(ref.critics_1[a].parameters()))]["step"] == steps
        assert ref.actor_optimizers.optimizer[a].state[next(iter(ref.actors[a].parameters()))]["step"] == steps // policy_freq
    out["sha256_keys"] = np.array(list(sha))
    out["sha256_values"] = np.array(list(sha.values()), dtype="S64")
    save("matd3_vector.npz", **out)
    print(f"  matd3: oracle == reference over {steps} learn calls (losses, None actor losses, gradients, every parameter)")


def gen_matd3_api():
    """The reference MATD3's constructor parameters (in order), defaults and public methods with their parameters."""
    from agilerl.algorithms.matd3 import MATD3

    def params(fn):
        return [p for p in inspect.signature(fn).parameters if p != "self"]

    defaults = {n: p.default for n, p in inspect.signature(MATD3.__init__).parameters.items()
                if n not in ("self", "device") and p.default is not inspect.Parameter.empty}
    own = {n: params(f) for n, f in vars(MATD3).items() if inspect.isfunction(f) and not n.startswith("_")}
    out = {"ctor": params(MATD3.__init__), "defaults": defaults, "methods": own}
    with open(os.path.join(HERE, "matd3_api.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote matd3_api.json")


if __name__ == "__main__":
    torch.set_num_threads(1)   # deterministic CPU reductions while generating
    if len(sys.argv) > 1 and sys.argv[1] not in ("matd3",):
        sys.exit(f"unknown fixture {sys.argv[1]!r} (matd3)")
    gen_matd3()
    gen_matd3_api()
