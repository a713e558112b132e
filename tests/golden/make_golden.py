"""Generate golden vectors by running the UNMODIFIED reference (/root/reference, AgileRL 2.6.1)
through ``oracle.refshim`` and check the oracle restatement against it while doing so.

Run here (the build container) only:   python tests/golden/make_golden.py
Outputs small ``.npz`` fixtures next to this file; they travel to the GPU box, /root/reference
does not.  Every fixture stores the inputs, any injected randomness, and the reference's outputs.

What is real and what is a stand-in: the reference's own code runs for segment trees, replay
buffers, Transition, Sampler, NoisyLinear/MLP/CNN/RainbowQNetwork/QNetwork, RainbowDQN/DQN
``learn``, DDPG/TD3 ``learn``, MADDPG ``learn`` (DeterministicActor + the EvolvableMultiInput critics),
MultiAgentReplayBuffer, RolloutBuffer's return/advantage loop, Mutations and TournamentSelection.  ``tensordict`` and ``gymnasium.spaces`` are the stand-ins of
``agilerl_b200.compat`` (the real packages are not in the image); torch is 2.11 (reference pins
2.9).
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import refshim  # noqa: E402

refshim.install()

from gymnasium import spaces  # noqa: E402
from tensordict import TensorDict  # noqa: E402

from agilerl.algorithms.dqn import DQN  # noqa: E402
from agilerl.algorithms.dqn_rainbow import RainbowDQN  # noqa: E402
from agilerl.components.data import Transition  # noqa: E402
from agilerl.components.replay_buffer import (  # noqa: E402
    MultiStepReplayBuffer, PrioritizedReplayBuffer, ReplayBuffer)
from agilerl.components.segment_tree import MinSegmentTree, SumSegmentTree  # noqa: E402
from agilerl.hpo.tournament import TournamentSelection  # noqa: E402

from oracle import learn as olearn, nets as onets, replay as oreplay, tournament as otourn  # noqa: E402
from oracle.segtree import CSegTree, PySegTree  # noqa: E402


def save(name, **arrays):
    path = os.path.join(HERE, name)
    np.savez_compressed(path, **arrays)
    print(f"wrote {name}: {os.path.getsize(path) / 1024:.1f} KiB")


def sd_np(sd):
    return {k: v.detach().cpu().numpy().copy() for k, v in sd.items()}


# ------------------------------------------------------------------------------------------------
def gen_tree():
    rng = np.random.default_rng(7)
    cap = 64
    n_ops = 400
    idx = rng.integers(0, cap, n_ops)
    val = rng.random(n_ops) ** 0.6 * 3.0
    rs, rm = SumSegmentTree(cap), MinSegmentTree(cap)
    ps, pm = PySegTree(cap, "sum"), PySegTree(cap, "min")
    cs, cm = CSegTree(cap, "sum"), CSegTree(cap, "min")
    snap_sum, snap_min = [], []
    for k, (i, v) in enumerate(zip(idx, val)):
        for t in (rs, rm, ps, pm, cs, cm):
            t[int(i)] = float(v)
        if k % 50 == 49:
            snap_sum.append(np.array(rs.tree)); snap_min.append(np.array(rm.tree))
    assert rs.tree == ps.tree == list(cs.tree) and rm.tree == pm.tree == list(cm.tree)
    ubs = rng.random(200) * rs.sum()
    ret = np.array([rs.retrieve(float(u)) for u in ubs])
    assert all(ps.retrieve(float(u)) == r == cs.retrieve(float(u)) for u, r in zip(ubs, ret))
    ranges = np.array([(a, b) for a in range(0, cap, 7) for b in range(a + 1, cap + 1, 9)])
    rsum = np.array([rs.sum(int(a), int(b)) for a, b in ranges])
    rmin = np.array([rm.min(int(a), int(b)) for a, b in ranges])
    save("tree_ops.npz", cap=cap, idx=idx, val=val, snap_sum=np.stack(snap_sum),
         snap_min=np.stack(snap_min), final_sum=np.array(rs.tree), final_min=np.array(rm.tree),
         ubs=ubs, retrieve=ret, ranges=ranges, range_sum=rsum, range_min=rmin)


# ------------------------------------------------------------------------------------------------
def _mk_transition(g, E, obs_shape, n_act, p_done, t):
    return dict(
        obs=torch.randint(0, 256, (E, *obs_shape), dtype=torch.uint8, generator=g),
        action=torch.randint(0, n_act, (E,), generator=g),
        reward=torch.randn(E, generator=g),
        next_obs=torch.randint(0, 256, (E, *obs_shape), dtype=torch.uint8, generator=g),
        done=(torch.rand(E, generator=g) < p_done),
    )


def gen_replay():
    """PER + n-step ingest through the real Transition/MultiStep/PER classes, then sampling with
    injected uniforms, then priority updates; checks the oracle along the way."""
    g = torch.Generator().manual_seed(11)
    E, obs_shape, n_act, max_size, n_step, gamma, alpha = 2, (3, 6, 6), 4, 48, 3, 0.99, 0.6
    mem = PrioritizedReplayBuffer(max_size, alpha=alpha)
    nmem = MultiStepReplayBuffer(max_size, n_step=n_step, gamma=gamma)
    omem = oreplay.OraclePER(max_size, alpha=alpha)
    onmem = oreplay.OracleNStep(max_size, n_step=n_step, gamma=gamma)
    raw = []
    for t in range(40):  # 40 steps x 2 envs -> wraps the 48-slot ring
        tr = _mk_transition(g, E, obs_shape, n_act, 0.15, t)
        raw.append(tr)
        td = Transition(obs=tr["obs"].numpy(), action=tr["action"].numpy(), reward=tr["reward"].numpy(),
                        next_obs=tr["next_obs"].numpy(), done=tr["done"].numpy(),
                        batch_size=[E]).to_tensordict()
        one = nmem.add(td)
        if one is not None:
            mem.add(one)
        # oracle side: same casts as Transition.__post_init__ (data.py:85-87)
        od = dict(obs=tr["obs"], action=tr["action"].float(), reward=tr["reward"].float(),
                  next_obs=tr["next_obs"], done=tr["done"].float())
        oone = onmem.add(od)
        if oone is not None:
            omem.add(oone)
    for k in mem.storage.keys():
        assert torch.equal(mem.storage[k], omem.storage[k]), k
        assert torch.equal(nmem.storage[k], onmem.storage[k]), k
    assert (mem._cursor, mem._size, mem.tree_ptr) == (omem.cursor, omem.size, omem.tree_ptr)

    # priority updates (numpy f32 priorities like learn() returns, and [B,1] idxs like sample())
    rng = np.random.default_rng(5)
    upd_idx = rng.integers(0, mem.size, (3, 16))
    upd_pri = np.abs(rng.standard_normal((3, 16))).astype(np.float32)
    upd_pri[0, 0] = 1e-9  # exercises the 1e-5 floor
    upd_idx[1, 3] = upd_idx[1, 2]  # duplicate index inside one batch (last writer wins)
    trees_after = []
    for r in range(3):
        mem.update_priorities(torch.from_numpy(upd_idx[r]).unsqueeze(1), upd_pri[r])
        omem.update_priorities(torch.from_numpy(upd_idx[r]), upd_pri[r])
        assert mem.sum_tree.tree == list(omem.sum_tree.tree) and mem.min_tree.tree == list(omem.min_tree.tree)
        trees_after.append((np.array(mem.sum_tree.tree), np.array(mem.min_tree.tree)))
    assert mem.max_priority == omem.max_priority

    # sampling with injected uniforms (the reference test's own trick, test_replay_buffer.py:859-883)
    B, beta = 16, 0.4
    uniforms = torch.rand(B, generator=g)
    it = iter(uniforms.tolist())
    orig = torch.rand
    torch.rand = lambda *a, **k: torch.tensor([next(it)])
    try:
        batch = mem.sample(B, beta)
    finally:
        torch.rand = orig
    obatch = omem.sample(B, beta, uniforms=uniforms)
    for k in batch.keys():
        assert torch.equal(batch[k], obatch[k]), k
    nbatch = nmem.sample_from_indices(batch["idxs"].squeeze(1))
    save("replay_per_nstep.npz",
         E=E, max_size=max_size, n_step=n_step, gamma=gamma, alpha=alpha, beta=beta,
         **{f"raw_{k}": torch.stack([r[k] for r in raw]).numpy() for k in raw[0]},
         **{f"per_{k}": v.numpy() for k, v in mem.storage.items()},
         **{f"nstep_{k}": v.numpy() for k, v in nmem.storage.items()},
         cursor=mem._cursor, size=mem._size, tree_ptr=mem.tree_ptr, max_priority=mem.max_priority,
         upd_idx=upd_idx, upd_pri=upd_pri,
         sum_after=np.stack([t[0] for t in trees_after]), min_after=np.stack([t[1] for t in trees_after]),
         uniforms=uniforms.numpy(), sample_idxs=batch["idxs"].numpy(), sample_weights=batch["weights"].numpy(),
         **{f"batch_{k}": batch[k].numpy() for k in ("obs", "action", "reward", "next_obs", "done")},
         **{f"nbatch_{k}": nbatch[k].numpy() for k in ("obs", "action", "reward", "next_obs", "done")})

    # uniform buffer ring layout incl. wrap (test_replay_buffer.py:144-177)
    rb = ReplayBuffer(max_size=3)
    d1 = TensorDict({"obs": torch.tensor([[1.0, 2.0], [3.0, 4.0]]), "reward": torch.tensor([1.0, 2.0])}, batch_size=[2])
    d2 = TensorDict({"obs": torch.tensor([[5.0, 6.0], [7.0, 8.0]]), "reward": torch.tensor([3.0, 4.0])}, batch_size=[2])
    rb.add(d1); rb.add(d2)
    save("replay_ring.npz", obs=rb.storage["obs"].numpy(), reward=rb.storage["reward"].numpy(),
         cursor=rb._cursor, size=rb._size, counter=rb.counter)


# ------------------------------------------------------------------------------------------------
def _draw_noise(spec):
    """Same RNG calls reset_noise makes (custom_components.py:116-131), per net."""
    return torch.cat([torch.cat([torch.randn(a), torch.randn(b)]) for _, a, b in onets.noisy_layer_keys(spec)])


def _rainbow_case(name, obs_shape, n_act, net_config, spec, B, *, weights_shape, driver_shapes=False,
                  n_step=True, combined=False, seed=0, v_min=-10.0, v_max=10.0, full=True):
    torch.manual_seed(seed)
    obs_space = spaces.Box(0, 255, obs_shape, np.uint8) if len(obs_shape) == 3 else spaces.Box(-1, 1, obs_shape, np.float32)
    agent = RainbowDQN(obs_space, spaces.Discrete(n_act), net_config=net_config, batch_size=B,
                       v_min=v_min, v_max=v_max, lr=1e-3, combined_reward=combined)
    # make target differ from online and give the net a non-trivial state
    with torch.no_grad():
        for p in agent.actor_target.parameters():
            p.add_(0.01 * torch.randn_like(p))
    actor0, target0 = sd_np(agent.actor.state_dict()), sd_np(agent.actor_target.state_dict())
    g = torch.Generator().manual_seed(seed + 100)
    def mk(shape_extra=()):
        if len(obs_shape) == 3:
            o = torch.randint(0, 256, (B, *obs_shape), dtype=torch.uint8, generator=g)
            no = torch.randint(0, 256, (B, *obs_shape), dtype=torch.uint8, generator=g)
        else:
            o = torch.randn((B, *obs_shape), generator=g); no = torch.randn((B, *obs_shape), generator=g)
        return dict(obs=o, action=torch.randint(0, n_act, (B, 1), generator=g).float(),
                    reward=torch.randn(B, 1, generator=g) * 3.0, next_obs=no,
                    done=(torch.rand(B, 1, generator=g) < 0.2).float())
    exp, nexp = mk(), mk()
    # hit the projection edge cases: exact-integer b (u==L), clamp at both ends
    nexp["reward"][0] = 0.0; nexp["done"][0] = 1.0          # t_z == 0 for all atoms -> b integer mid
    nexp["reward"][1] = 50.0                                  # clamps to v_max (u==L==N-1)
    nexp["reward"][2] = -50.0                                 # clamps to v_min (u==L==0)
    exp["reward"][0] = 0.0; exp["done"][0] = 1.0
    w = torch.rand(B, generator=g) * 0.9 + 0.1
    exp["weights"] = w.view(weights_shape)
    exp["idxs"] = torch.randint(0, 1000, (B, 1), generator=g)
    if driver_shapes:   # what train_off_policy actually feeds: storage[idxs [B,1]] (quirk Q2)
        nexp = {k: v.unsqueeze(1) for k, v in nexp.items()}
    exp_td = TensorDict({k: v.clone() for k, v in exp.items()}, batch_size=[B])
    nexp_td = TensorDict({k: v.clone() for k, v in nexp.items()}, batch_size=[B])

    torch.manual_seed(seed + 7)
    loss, idxs, pri = agent.learn(exp_td, n_experiences=nexp_td if n_step else None, per=True)
    torch.manual_seed(seed + 7)
    z_actor, z_target = _draw_noise(spec), _draw_noise(spec)
    actor1, target1 = sd_np(agent.actor.state_dict()), sd_np(agent.actor_target.state_dict())
    grads = {k: p.grad.detach().numpy().copy() for k, p in agent.actor.named_parameters()}
    adam = agent.optimizer.optimizer.state_dict()["state"]
    names = [k for k, _ in agent.actor.named_parameters()]
    exp_avg = {names[i]: s["exp_avg"].numpy().copy() for i, s in adam.items()}
    exp_avg_sq = {names[i]: s["exp_avg_sq"].numpy().copy() for i, s in adam.items()}

    # ---- oracle must reproduce the reference exactly (same torch CPU ops, same machine) ----
    oa = olearn.OracleAgent(spec, {k: torch.from_numpy(v) for k, v in actor0.items()},
                            {k: torch.from_numpy(v) for k, v in target0.items()},
                            batch_size=B, lr=1e-3, v_min=v_min, v_max=v_max, combined_reward=combined)
    oloss, _, opri = oa.learn_rainbow(exp, nexp if n_step else None, per=True, noise_normals=(z_actor, z_target))
    assert oloss == loss, (oloss, loss)
    assert np.array_equal(opri, pri)
    for k in actor1:
        assert np.array_equal(oa.actor[k].detach().numpy(), actor1[k]), k
        assert np.array_equal(oa.target[k].detach().numpy(), target1[k]), k
    print(f"  {name}: oracle == reference bit-exact (loss {loss:.6f})")

    out = dict(loss=np.float64(loss), priorities=pri, idxs=idxs.numpy(), z_actor=z_actor.numpy(),
               z_target=z_target.numpy(), proj_dist=oa.last_proj_dist.numpy(), B=B)
    for k, v in exp.items():
        out[f"exp_{k}"] = v.numpy()
    for k, v in nexp.items():
        out[f"nexp_{k}"] = v.numpy()
    if full:
        for tag, d in (("actor0", actor0), ("target0", target0), ("actor1", actor1), ("target1", target1),
                       ("grad", grads), ("m", exp_avg), ("v", exp_avg_sq)):
            for k, v in d.items():
                out[f"{tag}/{k}"] = v
    save(name, **out)


def gen_rainbow():
    small_cfg = {"encoder_config": {"channel_size": [8, 16], "kernel_size": [4, 3], "stride_size": [2, 1]},
                 "head_config": {"hidden_size": [32]}, "latent_dim": 16}
    def small_spec():
        return onets.rainbow_spec((3, 20, 20), 4, (8, 16), (4, 3), (2, 1), 16, (32,))
    import copy
    _rainbow_case("rainbow_small_canonical.npz", (3, 20, 20), 4, copy.deepcopy(small_cfg), small_spec(), 16,
                  weights_shape=(16,))
    _rainbow_case("rainbow_small_wcol.npz", (3, 20, 20), 4, copy.deepcopy(small_cfg), small_spec(), 16,
                  weights_shape=(16, 1), seed=1, full=False)                 # quirk Q1
    _rainbow_case("rainbow_small_driver.npz", (3, 20, 20), 4, copy.deepcopy(small_cfg), small_spec(), 16,
                  weights_shape=(16, 1), driver_shapes=True, seed=2, full=False)   # quirks Q1+Q2
    _rainbow_case("rainbow_small_combined.npz", (3, 20, 20), 4, copy.deepcopy(small_cfg), small_spec(), 16,
                  weights_shape=(16,), combined=True, seed=3, full=False)
    _rainbow_case("rainbow_small_1step.npz", (3, 20, 20), 4, copy.deepcopy(small_cfg), small_spec(), 16,
                  weights_shape=(16,), n_step=False, seed=4, full=False)
    # vector observations -> noisy MLP encoder with layer norm (q_networks.py:189-206)
    vec_cfg = {"encoder_config": {"hidden_size": [24, 24]}, "head_config": {"hidden_size": [32, 16]}, "latent_dim": 16}
    vspec = onets.rainbow_spec((5,), 3, latent_dim=16, hidden_size=(32, 16), encoder_hidden=(24, 24))
    _rainbow_case("rainbow_vector.npz", (5,), 3, vec_cfg, vspec, 8, weights_shape=(8,), seed=5)
    # the north-star architecture at B=16 (outputs only)
    ns_cfg = {"encoder_config": {"channel_size": [32, 32], "kernel_size": [8, 4], "stride_size": [4, 2]}}
    ns_spec = onets.rainbow_spec((4, 84, 84), 6)
    _rainbow_case("rainbow_northstar_b16.npz", (4, 84, 84), 6, ns_cfg, ns_spec, 16, weights_shape=(16,), seed=6,
                  full=False)


def gen_dqn():
    for double, seed in ((False, 0), (True, 1)):
        torch.manual_seed(seed)
        B, obs_shape, n_act = 16, (4,), 2
        agent = DQN(spaces.Box(-1, 1, obs_shape, np.float32), spaces.Discrete(n_act), batch_size=B, lr=1e-3,
                    double=double)
        with torch.no_grad():
            for p in agent.actor_target.parameters():
                p.add_(0.01 * torch.randn_like(p))
        actor0, target0 = sd_np(agent.actor.state_dict()), sd_np(agent.actor_target.state_dict())
        g = torch.Generator().manual_seed(seed + 50)
        exp = dict(obs=torch.randn(B, 4, generator=g), action=torch.randint(0, n_act, (B, 1), generator=g).float(),
                   reward=torch.randn(B, 1, generator=g), next_obs=torch.randn(B, 4, generator=g),
                   done=(torch.rand(B, 1, generator=g) < 0.2).float())
        loss = agent.learn(TensorDict({k: v.clone() for k, v in exp.items()}, batch_size=[B]))
        actor1, target1 = sd_np(agent.actor.state_dict()), sd_np(agent.actor_target.state_dict())
        spec = onets.q_spec(obs_shape, n_act)
        oa = olearn.OracleAgent(spec, {k: torch.from_numpy(v) for k, v in actor0.items()},
                                {k: torch.from_numpy(v) for k, v in target0.items()}, batch_size=B, lr=1e-3,
                                double=double)
        oloss = oa.learn_dqn(exp)
        assert oloss == loss, (oloss, loss)
        for k in actor1:
            assert np.array_equal(oa.actor[k].detach().numpy(), actor1[k]), k
            assert np.array_equal(oa.target[k].detach().numpy(), target1[k]), k
        print(f"  dqn double={double}: oracle == reference bit-exact (loss {loss:.6f})")
        out = dict(loss=np.float64(loss), B=B, double=double)
        for k, v in exp.items():
            out[f"exp_{k}"] = v.numpy()
        for tag, d in (("actor0", actor0), ("target0", target0), ("actor1", actor1), ("target1", target1)):
            for k, v in d.items():
                out[f"{tag}/{k}"] = v
        save(f"dqn_vector_double{int(double)}.npz", **out)


def gen_tournament():
    class A:
        algo = "DQN"
        def __init__(self, index, fitness):
            self.index, self.fitness = index, list(fitness)
        def clone(self, index=None, wrap=True):
            a = A(self.index if index is None else index, self.fitness); a.parent = getattr(self, "parent", self.index)
            a.parent = self.index
            return a
    rng = np.random.default_rng(3)
    cases = []
    for c, (pop, tsize, elit) in enumerate([(6, 2, True), (8, 3, True), (8, 4, False), (4, 2, True)]):
        fit = rng.standard_normal((pop, 5)) * 10
        idxs = rng.permutation(pop * 2)[:pop]
        agents = [A(int(i), f) for i, f in zip(idxs, fit)]
        ts = TournamentSelection(tsize, elit, pop, eval_loop=3)
        np.random.seed(100 + c)
        elite, new_pop = ts.select(agents)
        np.random.seed(100 + c)
        epos, sel = otourn.select_positions([a.fitness for a in agents], [a.index for a in agents], tsize, elit, pop, 3)
        assert agents[epos].index == elite.index
        assert [(agents[p].index, ni) for p, ni in sel] == [(a.parent, a.index) for a in new_pop]
        cases.append(dict(fit=fit, idxs=idxs, tsize=tsize, elit=elit, seed=100 + c, elite_index=elite.index,
                          parents=np.array([a.parent for a in new_pop]), new_index=np.array([a.index for a in new_pop])))
    # the reference's own known-answer case (tests/test_hpo/test_tournament.py:74-125): elite = index 4
    out = {}
    for c, d in enumerate(cases):
        for k, v in d.items():
            out[f"c{c}_{k}"] = np.asarray(v)
    out["n_cases"] = len(cases)
    save("tournament.npz", **out)
    print("  tournament: oracle == reference")


def gen_ddpg_td3():
    """SURVEY §8(f) rank 1 groundwork: DDPG / TD3 learn() of BASELINE config 3's shapes (17-dim obs, 6-dim
    action) — four consecutive learn calls (actor + targets move on calls 2 and 4), oracle == reference
    bit for bit; the fixture keeps the initial state dicts, the batches, the RNG seeds of the in-place
    target-policy noise, and the reference's losses + final parameters."""
    from agilerl.algorithms.ddpg import DDPG
    from agilerl.algorithms.td3 import TD3
    from oracle import ddpg_td3 as od
    obs_space = spaces.Box(-1, 1, (17,), np.float32)
    act_space = spaces.Box(-1, 1, (6,), np.float32)
    B, steps = 32, 4

    def batch(seed):
        g = torch.Generator().manual_seed(seed)
        return dict(obs=torch.randn(B, 17, generator=g), action=torch.rand(B, 6, generator=g) * 2 - 1,
                    reward=torch.randn(B, 1, generator=g), next_obs=torch.randn(B, 17, generator=g),
                    done=(torch.rand(B, 1, generator=g) < 0.2).float())

    for name, cls, twin in (("ddpg", DDPG, False), ("td3", TD3, True)):
        torch.manual_seed(7)
        ref = cls(obs_space, act_space, batch_size=B, device="cpu")
        crit = [ref.critic] if not twin else [ref.critic_1, ref.critic_2]
        crit_t = [ref.critic_target] if not twin else [ref.critic_target_1, ref.critic_target_2]
        a_hidden = list(ref.actor.head_net.net_config["hidden_size"])
        c_hidden = list(crit[0].head_net.net_config["hidden_size"])
        a_specs = od.actor_specs(17, 6, head_hidden=a_hidden, encoder_layer_norm=ref.actor.encoder.net_config["layer_norm"])
        c_specs = od.critic_specs(17, 6, head_hidden=c_hidden)
        out = {"B": B, "steps": steps, "twin": int(twin), "a_hidden": np.array(a_hidden), "c_hidden": np.array(c_hidden),
               "gamma": ref.gamma, "tau": ref.tau, "lr_actor": ref.lr_actor, "lr_critic": ref.lr_critic,
               "policy_freq": ref.policy_freq}
        out.update({f"actor0/{k}": v for k, v in sd_np(ref.actor.state_dict()).items()})
        out.update({f"actor_target0/{k}": v for k, v in sd_np(ref.actor_target.state_dict()).items()})
        for i, (c, t) in enumerate(zip(crit, crit_t)):
            out.update({f"critic{i}_0/{k}": v for k, v in sd_np(c.state_dict()).items()})
            out.update({f"critic_target{i}_0/{k}": v for k, v in sd_np(t.state_dict()).items()})
        orc = od.OracleDDPG(a_specs, c_specs, ref.actor.state_dict(), ref.actor_target.state_dict(),
                            [c.state_dict() for c in crit], [c.state_dict() for c in crit_t], gamma=ref.gamma, tau=ref.tau,
                            lr_actor=ref.lr_actor, lr_critic=ref.lr_critic, policy_freq=ref.policy_freq, twin=twin)
        for st in range(steps):
            e_ref, e_orc = batch(40 + st), batch(40 + st)
            for k, v in e_ref.items():
                out[f"s{st}_{k}"] = v.numpy().copy()
            out[f"s{st}_seed"] = 500 + st
            torch.manual_seed(500 + st)
            ra, rc = ref.learn(TensorDict(e_ref, batch_size=[B]))
            torch.manual_seed(500 + st)
            oa, oc = orc.learn(e_orc)
            assert ra == oa and rc == oc, (name, st, ra, oa, rc, oc)
            out[f"s{st}_noise"] = e_ref["action"].numpy().copy()          # the batch's action tensor now holds the noise
            out[f"s{st}_actor_loss"] = np.nan if ra is None else ra
            out[f"s{st}_critic_loss"] = rc
        for k, v in ref.actor.state_dict().items():
            assert torch.equal(v, orc.actor[k].data), (name, k)
        for c, ocr in zip(crit, orc.critics):
            for k, v in c.state_dict().items():
                assert torch.equal(v, ocr[k].data), (name, k)
        for c, oct_ in zip(crit_t, orc.critic_targets):
            for k, v in c.state_dict().items():
                assert torch.equal(v, oct_[k]), (name, k)
        out.update({f"actor1/{k}": v for k, v in sd_np(ref.actor.state_dict()).items()})
        out.update({f"actor_target1/{k}": v for k, v in sd_np(ref.actor_target.state_dict()).items()})
        for i, (c, t) in enumerate(zip(crit, crit_t)):
            out.update({f"critic{i}_1/{k}": v for k, v in sd_np(c.state_dict()).items()})
            out.update({f"critic_target{i}_1/{k}": v for k, v in sd_np(t.state_dict()).items()})
        save(f"{name}_vector.npz", **out)
        print(f"  {name}: oracle == reference over {steps} learn calls (losses, every parameter, targets)")


def gen_gae():
    """SURVEY §8(f) rank 2 groundwork: RolloutBuffer.compute_returns_and_advantages at BASELINE config 4's
    shape (256 vector envs, 8-dim obs), GAE and Monte-Carlo modes; oracle (oracle/gae.py) == reference bit
    for bit, fixture keeps rewards / dones / values / bootstrap inputs and the reference's outputs."""
    from agilerl.components.rollout_buffer import RolloutBuffer
    from oracle import gae
    T, E = 64, 256
    obs_space = spaces.Box(-1, 1, (8,), np.float32)
    act_space = spaces.Discrete(4)
    out = {"T": T, "E": E, "gamma": 0.99, "gae_lambda": 0.95}
    for mode, use_gae in (("gae", True), ("mc", False)):
        rng = np.random.default_rng(11 + int(use_gae))
        buf = RolloutBuffer(capacity=T, num_envs=E, observation_space=obs_space, action_space=act_space, device="cpu",
                            gae_lambda=0.95, gamma=0.99, use_gae=use_gae)
        for t in range(T):
            buf.add(obs=rng.standard_normal((E, 8)).astype(np.float32), action=rng.integers(0, 4, E),
                    reward=rng.standard_normal(E).astype(np.float32), done=rng.random(E) < 0.05,
                    value=rng.standard_normal(E).astype(np.float32), log_prob=rng.standard_normal(E).astype(np.float32))
        lv = rng.standard_normal(E).astype(np.float32)
        ld = (rng.random(E) < 0.05).astype(np.float32)
        buf.compute_returns_and_advantages(lv, ld)
        R = buf.buffer["rewards"][:T].numpy().reshape(T, E)
        D = buf.buffer["dones"][:T].numpy().reshape(T, E)
        V = buf.buffer["values"][:T].numpy().reshape(T, E)
        ra = buf.buffer["advantages"][:T].numpy().reshape(T, E)
        rr = buf.buffer["returns"][:T].numpy().reshape(T, E)
        oa, orr = gae.compute_returns_and_advantages(R, D, V, lv, ld, 0.99, 0.95, use_gae)
        assert np.array_equal(ra, oa) and np.array_equal(rr, orr), mode
        out.update({f"{mode}_rewards": R, f"{mode}_dones": D.astype(np.uint8), f"{mode}_values": V, f"{mode}_last_value": lv,
                    f"{mode}_last_done": ld, f"{mode}_advantages": ra, f"{mode}_returns": rr})
    save("gae_rollout.npz", **out)
    print("  gae: oracle == reference (GAE and Monte-Carlo)")


def gen_mutations():
    """Mutations (agilerl/hpo/mutation.py) on the UNMODIFIED reference: everything its seeded generators decide —
    which mutation each member of a population gets (``self.rng.choice``, :335-339), what
    ``_gaussian_parameter_mutation`` does to a network's state_dict (:733-827: numpy Generator for keys / rows /
    columns / branch, torch's global generator for the noise), the ``rl_hyperparam_mutation`` sequence (:413-452 ->
    registry.py:135-186, 234-241: torch.randperm + torch.rand) and the activation picked by
    ``_permutate_activation``.  (Architecture mutations draw from each module's own unseeded generator in the
    reference — only the METHOD choice, made by ``Mutations.rng``, is reproducible and recorded.)"""
    from agilerl.algorithms.core.registry import HyperparameterConfig, RLParameter
    from agilerl.hpo.mutation import Mutations
    out = {}
    obs_space, act_space = spaces.Box(0, 255, (3, 20, 20), np.uint8), spaces.Discrete(4)
    net_config = {"encoder_config": {"channel_size": [8, 16], "kernel_size": [4, 3], "stride_size": [2, 1]},
                  "head_config": {"hidden_size": [32]}, "latent_dim": 16}
    # (a) mutation choice per population member
    for c, (probs, seed) in enumerate([((0.2, 0.2, 0.2, 0.2, 0.2), 42), ((0.4, 0.0, 0.3, 0.0, 0.3), 7), ((0, 1, 1, 1, 1), 3)]):
        m = Mutations(no_mutation=probs[0], architecture=probs[1], new_layer_prob=0.5, parameters=probs[2],
                      activation=probs[3], rl_hp=probs[4], rand_seed=seed)
        names = [f.__name__ for f in m.rng.choice(m.mut_options, 12, p=m.mut_proba)]
        pre = [f.__name__ for f in m.rng.choice(m.pretraining_mut_options, 12, p=m.pretraining_mut_proba)]
        out[f"choice{c}_probs"], out[f"choice{c}_seed"] = np.array(probs, np.float64), seed
        out[f"choice{c}_names"], out[f"choice{c}_pre"] = np.array(names), np.array(pre)
    # (b) Gaussian parameter mutation of a RainbowQNetwork state_dict
    for c, seed in enumerate((11, 12)):
        torch.manual_seed(100 + seed)
        agent = RainbowDQN(obs_space, act_space, net_config=dict(net_config), batch_size=8, v_min=-10.0, v_max=10.0)
        m = Mutations(0, 0, 0.5, 1, 0, 0, mutation_sd=0.1, rand_seed=seed)
        before = sd_np(agent.actor.state_dict())
        torch.manual_seed(500 + seed)
        m._gaussian_parameter_mutation(agent.actor)
        after = sd_np(agent.actor.state_dict())
        out[f"gauss{c}_seed"] = seed
        for k, v in before.items():
            out[f"gauss{c}_before/{k}"] = v
        for k, v in after.items():
            out[f"gauss{c}_after/{k}"] = v
        n_changed = sum(int((before[k] != after[k]).sum()) for k in before)
        print(f"  gaussian mutation seed {seed}: {n_changed} weights changed")
    # (c) RL hyper-parameter mutation sequence
    hp = HyperparameterConfig(lr=RLParameter(min=1e-5, max=1e-2), batch_size=RLParameter(min=8, max=64, dtype=int),
                              learn_step=RLParameter(min=1, max=16, dtype=int, grow_factor=1.5, shrink_factor=0.75))
    torch.manual_seed(0)
    agent = RainbowDQN(obs_space, act_space, hp_config=hp, net_config=dict(net_config), batch_size=16, lr=1e-3, learn_step=4,
                       v_min=-10.0, v_max=10.0)
    m = Mutations(0, 0, 0.5, 0, 0, 1, rand_seed=5)
    torch.manual_seed(900)
    seq = []
    for _ in range(12):
        agent = m.rl_hyperparam_mutation(agent)
        seq.append((agent.mut, float(agent.lr), int(agent.batch_size), int(agent.learn_step)))
    out["rlhp_mut"] = np.array([s[0] for s in seq])
    out["rlhp_vals"] = np.array([[s[1], s[2], s[3]] for s in seq], np.float64)
    # (d) activation picks
    m = Mutations(0, 0, 0.5, 0, 1, 0, activation_selection=["ReLU", "ELU", "GELU"], rand_seed=9)
    acts = []
    for _ in range(8):
        agent = m.activation_mutation(agent)
        acts.append(agent.actor.activation)
    out["act_seq"] = np.array(acts)
    # (e) architecture: the method Mutations.rng samples for a RainbowQNetwork (names only)
    m = Mutations(0, 1, 0.5, 0, 0, 0, rand_seed=21)
    torch.manual_seed(1)
    agent = RainbowDQN(obs_space, act_space, net_config=dict(net_config), batch_size=8, v_min=-10.0, v_max=10.0)
    out["arch_methods"] = np.array(list(agent.actor.mutation_methods))
    out["arch_probs"] = np.array(agent.actor.get_mutation_probs(m.new_layer_prob), np.float64)
    picks = []
    for _ in range(16):
        picks.append(agent.actor.sample_mutation_method(m.new_layer_prob, m.rng))
    out["arch_picks"] = np.array([p if isinstance(p, str) else getattr(p, "__name__", str(p)) for p in picks])
    save("mutations.npz", **out)
    print("  mutations: reference outputs recorded")


def gen_maddpg():
    """SURVEY §8(f) rank 4: MADDPG.learn (maddpg.py:571-740) on BASELINE config 5's shapes (4 agents x 18-dim
    observations, 5-dim actions) — three consecutive learn calls of the UNMODIFIED reference, oracle == reference bit
    for bit (losses, every actor / critic / target parameter).  A NaN reward and a NaN done (an agent that was not
    alive) ride in the second batch: maddpg.py:683-694."""
    from agilerl.algorithms.maddpg import MADDPG
    from oracle import maddpg as om
    ids = [f"agent_{i}" for i in range(4)]
    obs_dims, act_dims = [18, 18, 18, 18], [5, 5, 5, 5]
    obs_spaces = [spaces.Box(-1, 1, (d,), np.float32) for d in obs_dims]
    act_spaces = [spaces.Box(-1, 1, (d,), np.float32) for d in act_dims]
    B, steps = 32, 3
    torch.manual_seed(11)
    ref = MADDPG(obs_spaces, act_spaces, agent_ids=ids, batch_size=B, device="cpu")
    a_hidden = list(ref.actors[ids[0]].head_net.net_config["hidden_size"])
    c_hidden = list(ref.critics[ids[0]].head_net.net_config["hidden_size"])
    a_specs = {a: om.actor_specs(o, d, head_hidden=a_hidden) for a, o, d in zip(ids, obs_dims, act_dims)}
    c_head = om.critic_head_spec(sum(act_dims), head_hidden=c_hidden)
    out = {"B": B, "steps": steps, "agent_ids": np.array(ids), "obs_dims": np.array(obs_dims), "act_dims": np.array(act_dims),
           "a_hidden": np.array(a_hidden), "c_hidden": np.array(c_hidden), "gamma": ref.gamma, "tau": ref.tau,
           "lr_actor": ref.lr_actor, "lr_critic": ref.lr_critic}
    groups = (("actor", ref.actors), ("actor_target", ref.actor_targets), ("critic", ref.critics),
              ("critic_target", ref.critic_targets))
    for gname, nets in groups:
        for a in ids:
            out.update({f"{gname}0/{a}/{k}": v for k, v in sd_np(nets[a].state_dict()).items()})
    orc = om.OracleMADDPG(ids, a_specs, c_head, {a: ref.actors[a].state_dict() for a in ids},
                          {a: ref.actor_targets[a].state_dict() for a in ids}, {a: ref.critics[a].state_dict() for a in ids},
                          {a: ref.critic_targets[a].state_dict() for a in ids}, gamma=ref.gamma, tau=ref.tau,
                          lr_actor=ref.lr_actor, lr_critic=ref.lr_critic)

    def batch(seed, with_nan):
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

    for s_ in range(steps):
        e_ref, e_orc = batch(70 + s_, s_ == 1), batch(70 + s_, s_ == 1)
        for fname, fd in zip(("obs", "action", "reward", "next_obs", "done"), e_ref):
            for a in ids:
                out[f"s{s_}_{fname}/{a}"] = fd[a].numpy().copy()
        r_loss = ref.learn(e_ref)
        o_loss = orc.learn(e_orc)
        for a in ids:
            assert tuple(r_loss[a]) == tuple(o_loss[a]), (s_, a, r_loss[a], o_loss[a])
            out[f"s{s_}_actor_loss/{a}"], out[f"s{s_}_critic_loss/{a}"] = r_loss[a]
        if s_ == 0:
            for k, v in orc.last_grads.items():
                out[f"s0_grad/{k}"] = v.numpy().copy()
    for gname, nets, onets_ in (("actor", ref.actors, orc.actors), ("actor_target", ref.actor_targets, orc.actor_targets),
                               ("critic", ref.critics, orc.critics), ("critic_target", ref.critic_targets, orc.critic_targets)):
        for a in ids:
            for k, v in nets[a].state_dict().items():
                assert torch.equal(v, onets_[a][k].data), (gname, a, k)
            out.update({f"{gname}1/{a}/{k}": v for k, v in sd_np(nets[a].state_dict()).items()})
    save("maddpg_vector.npz", **out)
    print(f"  maddpg: oracle == reference over {steps} learn calls (losses, every parameter, targets)")


def gen_ma_replay():
    """MultiAgentReplayBuffer (multi_agent_replay_buffer.py:30-242) of the UNMODIFIED reference: vectorised and
    single-env saves into a 50-slot buffer until it has wrapped, then seeded ``random.sample`` batches; the oracle
    ring reproduces every sampled tensor bit for bit."""
    import random
    from agilerl.components.multi_agent_replay_buffer import MultiAgentReplayBuffer
    from oracle import maddpg as om
    ids = ["agent_0", "agent_1", "agent_2"]
    fields = ["obs", "action", "reward", "next_obs", "done"]
    dims = {"agent_0": (6, 2), "agent_1": (4, 3), "agent_2": (6, 2)}
    cap, E = 50, 4
    ref, orc = MultiAgentReplayBuffer(cap, fields, ids, device="cpu"), om.OracleMAReplay(cap, fields, ids)
    rng = np.random.default_rng(5)
    out = {"cap": cap, "E": E, "agent_ids": np.array(ids), "fields": np.array(fields),
           "obs_dims": np.array([dims[a][0] for a in ids]), "act_dims": np.array([dims[a][1] for a in ids])}
    n_steps = 0
    for t in range(20):
        vect = t % 5 != 4                      # every fifth step comes from a single (un-vectorised) environment
        lead = (E,) if vect else ()
        obs = {a: rng.standard_normal(lead + (dims[a][0],)).astype(np.float32) for a in ids}
        act = {a: rng.uniform(-1, 1, lead + (dims[a][1],)).astype(np.float32) for a in ids}
        rew = {a: (rng.standard_normal(E) if vect else float(rng.standard_normal())) for a in ids}
        nobs = {a: rng.standard_normal(lead + (dims[a][0],)).astype(np.float32) for a in ids}
        done = {a: ((rng.uniform(size=E) < 0.3) if vect else bool(rng.uniform() < 0.3)) for a in ids}
        if t == 17:                            # an agent that was not alive: NaN reward / done (float arrays)
            rew["agent_1"] = np.array(rew["agent_1"], dtype=np.float64); rew["agent_1"][1] = np.nan
            done["agent_1"] = np.array(done["agent_1"], dtype=np.float64); done["agent_1"][1] = np.nan
        ref.save_to_memory(obs, act, rew, nobs, done, is_vectorised=vect)
        orc.save_to_memory(obs, act, rew, nobs, done, is_vectorised=vect)
        out[f"t{t}_vect"] = int(vect)
        for fname, fd in zip(fields, (obs, act, rew, nobs, done)):
            for a in ids:
                out[f"t{t}_{fname}/{a}"] = np.asarray(fd[a])
        n_steps += 1
        assert len(ref) == len(orc) and ref.counter == orc.counter
    out["n_steps"], out["final_len"], out["final_counter"] = n_steps, len(ref), ref.counter
    for c, (seed, B) in enumerate([(1, 8), (2, 16), (3, 50)]):
        random.seed(seed)
        r = ref.sample(B)
        random.seed(seed)
        o = orc.sample(B)
        for fname, rd, od_ in zip(fields, r, o):
            for a in ids:
                assert rd[a].dtype == od_[a].dtype == torch.float32 and rd[a].shape == od_[a].shape, (fname, a)
                assert torch.equal(torch.nan_to_num(rd[a], nan=-7.0), torch.nan_to_num(od_[a], nan=-7.0)), (c, fname, a)
                out[f"sample{c}_{fname}/{a}"] = rd[a].numpy().copy()
        out[f"sample{c}_seed"], out[f"sample{c}_B"] = seed, B
    out["n_samples"] = 3
    save("ma_replay.npz", **out)
    print("  multi-agent replay: oracle == reference on every sampled leaf (3 seeded batches, wrapped buffer)")


def gen_api_surface():
    """The reference's public signatures that tests/test_api_surface_cpu.py holds this package to: constructor parameters
    (in order) of every replaced class, the defaults of the learners' constructors, the driver's parameters and the
    multi-agent replay's method parameters."""
    import inspect
    import json

    import agilerl.algorithms.maddpg as r_ma
    import agilerl.components.multi_agent_replay_buffer as r_mb
    import agilerl.hpo.mutation as r_mut
    import agilerl.training.train_off_policy as r_train

    def params(fn):
        return [p for p in inspect.signature(fn).parameters if p != "self"]

    def defaults(cls):
        return {n: p.default for n, p in inspect.signature(cls.__init__).parameters.items()
                if n not in ("self", "device") and p.default is not inspect.Parameter.empty}

    classes = dict(ReplayBuffer=ReplayBuffer, MultiStepReplayBuffer=MultiStepReplayBuffer,
                   PrioritizedReplayBuffer=PrioritizedReplayBuffer, RainbowDQN=RainbowDQN, DQN=DQN,
                   TournamentSelection=TournamentSelection, Mutations=r_mut.Mutations, SumSegmentTree=SumSegmentTree,
                   MinSegmentTree=MinSegmentTree, MADDPG=r_ma.MADDPG, MultiAgentReplayBuffer=r_mb.MultiAgentReplayBuffer)
    out = {"ctor": {k: params(c.__init__) for k, c in classes.items()},
           "defaults": {k: defaults(classes[k]) for k in ("RainbowDQN", "DQN", "MADDPG")},
           "train_off_policy": params(r_train.train_off_policy),
           "multi_agent_buffer_methods": {m: params(getattr(r_mb.MultiAgentReplayBuffer, m)) for m in
                                          ("save_to_memory", "save_to_memory_single_env", "save_to_memory_vect_envs", "sample")}}
    with open(os.path.join(HERE, "api_surface.json"), "w") as f:
        json.dump(out, f, indent=1, sort_keys=True)
    print("wrote api_surface.json")


def gen_driver_equivalence():
    """The reference's unchanged drivers on the seeded runs of tests/_driver_equivalence_standin.py (our restated driver is
    checked against each run while recording)."""
    import json
    import subprocess

    out = {}
    for mode in ("DQN", "TD3", "RAINBOW", "MADDPG"):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "_driver_equivalence_standin.py"), mode, "--record"],
                           capture_output=True, text=True, check=True)
        lines = dict(l.split(" ", 1) for l in p.stdout.splitlines() if l.startswith(("REFERENCE ", "RESULT ")))
        assert json.loads(lines["RESULT"])["equal"], (mode, lines["RESULT"])
        out[mode] = json.loads(lines["REFERENCE"])
    with open(os.path.join(HERE, "driver_equivalence.json"), "w") as f:
        json.dump(out, f, sort_keys=True)
    print("wrote driver_equivalence.json: our restated drivers == the reference's")


def gen_maddpg_host():
    """The reference's ``MADDPG.test`` and ``get_action`` on the cases of tests/test_multi_agent_host_cpu.py."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import test_multi_agent_host_cpu as t
    save("maddpg_host.npz", **t.reference_test_loop_outputs(), **t.reference_get_action_outputs())


if __name__ == "__main__":
    torch.set_num_threads(1)   # deterministic CPU reductions while generating
    if len(sys.argv) > 1 and sys.argv[1] == "api_surface":
        gen_api_surface()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "drivers":
        gen_driver_equivalence()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "maddpg_host":
        gen_maddpg_host()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "mutations":
        gen_mutations()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "ddpg_td3":
        gen_ddpg_td3()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "maddpg":
        gen_maddpg()
        gen_ma_replay()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "gae":
        gen_gae()
        sys.exit(0)
    gen_tree()
    gen_replay()
    gen_rainbow()
    gen_dqn()
    gen_tournament()
    gen_ddpg_td3()
    gen_gae()
    gen_mutations()
    gen_maddpg()
    gen_ma_replay()
    gen_api_surface()
    gen_driver_equivalence()
    gen_maddpg_host()
