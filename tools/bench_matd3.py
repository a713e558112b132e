"""MATD3 and MADDPG learn throughput in one run, at BASELINE config 5's shapes (4 agents x 18-dim observations, 5-dim
continuous actions, one shared 100k-step HBM replay, pop = 16 on one GPU) with the MADDPG arm's hyper-parameters of
bench.py (batch 64, lr 1e-4 / 1e-3, tau 1e-3, gamma 0.95) and policy_freq = 2 (the reference's matd3.yaml).

    python tools/bench_matd3.py [--steps 20] [--warmup 3]

Prints one JSON line shaped like ``bench.py --workload maddpg``'s: ``value`` is MATD3's device-resident population
gradient-steps/s (position draw + gather into the captured buffers + graph replay per member, members overlapped), median
of repeats; ``maddpg`` holds the same loop for MADDPG members; ``e2e`` the reference-shaped ``learn()`` path for both;
``cpu_baseline`` the oracle restatement of the reference's MATD3.learn on the host; ``graph_kernels`` the kernel nodes of
the two captured MATD3 calls and of the MADDPG call; ``gpu`` the device name and power limit read in the same run.
Writes nothing."""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import ClockSampler, time_region  # noqa: E402


def gpu_info(index: int = 0) -> dict:
    out = {"name": torch.cuda.get_device_name(index)}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        out["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
        out["power_default_limit_w"] = pynvml.nvmlDeviceGetPowerManagementDefaultLimit(h) / 1000.0
    except Exception as e:  # noqa: BLE001 - reported, not hidden
        out["power_limit_w"] = None
        out["power_error"] = repr(e)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    from agilerl_b200 import _lib
    from agilerl_b200.algorithms import MADDPG, MATD3
    from agilerl_b200.compat import spaces
    from agilerl_b200.components import MultiAgentReplayBuffer
    from agilerl_b200.training.population import multi_agent_population_learn
    from oracle import maddpg as om
    from oracle.matd3 import OracleMATD3
    device, BT, N, NA, OD, AD, POPM, PF = "cuda:0", 64, 100_000, 4, 18, 5, 16, 2
    torch.cuda.set_device(0)
    lib = _lib.load(require_cuda=True)
    ids = [f"agent_{i}" for i in range(NA)]
    obs_sp = [spaces.Box(-np.inf, np.inf, (OD,), np.float32) for _ in ids]
    act_sp = [spaces.Box(-1.0, 1.0, (AD,), np.float32) for _ in ids]
    hp = dict(agent_ids=ids, batch_size=BT, lr_actor=1e-4, lr_critic=1e-3, tau=1e-3, gamma=0.95, device=device)
    pops = {}
    for name, cls, kw in (("MATD3", MATD3, {"policy_freq": PF}), ("MADDPG", MADDPG, {})):
        pops[name] = []
        for a in range(POPM):
            torch.manual_seed(a)
            pops[name].append(cls(obs_sp, act_sp, index=a, **hp, **kw))
    fields = ["obs", "action", "reward", "next_obs", "done"]
    mem = MultiAgentReplayBuffer(N, fields, ids, device=device)
    rng = np.random.default_rng(0)
    chunk = 20_000
    for _ in range(N // chunk):
        mem.save_to_memory({a: rng.standard_normal((chunk, OD), dtype=np.float32) for a in ids},
                           {a: rng.uniform(-1, 1, (chunk, AD)).astype(np.float32) for a in ids},
                           {a: rng.standard_normal(chunk, dtype=np.float32) for a in ids},
                           {a: rng.standard_normal((chunk, OD), dtype=np.float32) for a in ids},
                           {a: rng.uniform(size=chunk) < 0.01 for a in ids}, is_vectorised=True)
    torch.cuda.synchronize()

    res = {}
    sampler = ClockSampler(0)
    sampler.start()
    for name, pop in pops.items():
        dev_step = lambda pop=pop: multi_agent_population_learn(pop, mem, BT)[-1]

        def api_step(pop=pop):
            out = None
            for agent in pop:
                out = agent.learn(mem.sample(BT))
            return out
        for _ in range(max(args.warmup, 3)):
            dev_step()
        api_step()
        torch.cuda.synchronize()
        l0 = lib.b2rl_launch_count()
        ms, ms_all = time_region(dev_step, args.steps, False)
        launches = (lib.b2rl_launch_count() - l0) // len(ms_all)
        e2e_steps = max(1, min(args.steps, 50))
        ms_e2e, ms_e2e_all = time_region(api_step, e2e_steps, False, repeats=3)
        kernels = {}
        for kind, g in pop[0]._plans[BT].graphs.items():
            c = ctypes.c_int(0)
            _lib.check(lib.b2rl_graph_kernel_count(g, ctypes.byref(c)))
            kernels["critic_only" if kind else "full"] = c.value
        res[name] = {"value": POPM * args.steps / (ms / 1e3), "unit": "steps/s", "ms_per_step": ms / args.steps,
                     "ms_repeats": [round(x, 3) for x in ms_all], "gpu_launches_per_step": int(launches),
                     "graph_kernels": kernels,
                     "e2e": {"value": POPM * e2e_steps / (ms_e2e / 1e3), "unit": "steps/s", "ms_per_step": ms_e2e / e2e_steps,
                             "steps": e2e_steps, "ms_repeats": [round(x, 3) for x in ms_e2e_all]}}
    clocks = sampler.stop()
    # CPU arm: the oracle restatement of the reference's MATD3.learn, one member, batches sampled like the reference
    a0 = pops["MATD3"][0]
    cpu = lambda net: {k: v.cpu().clone() for k, v in net.state_dict().items()}
    sd = lambda attr: {a: cpu(getattr(a0, attr)[a]) for a in ids}
    orc = OracleMATD3(ids, {a: om.actor_specs(OD, AD, head_hidden=[64]) for a in ids}, om.critic_head_spec(NA * AD, head_hidden=[64]),
                      sd("actors"), sd("actor_targets"), sd("critics_1"), sd("critic_targets_1"), sd("critics_2"),
                      sd("critic_targets_2"), gamma=0.95, tau=1e-3, lr_actor=1e-4, lr_critic=1e-3, policy_freq=PF)
    omem = om.OracleMAReplay(20_000, fields, ids)
    for _ in range(20_000):
        omem._add({a: rng.standard_normal(OD, dtype=np.float32) for a in ids}, {a: rng.uniform(-1, 1, AD).astype(np.float32) for a in ids},
                  {a: float(rng.standard_normal()) for a in ids}, {a: rng.standard_normal(OD, dtype=np.float32) for a in ids},
                  {a: bool(rng.uniform() < 0.01) for a in ids})
    t0, n_cpu = time.perf_counter(), 0
    while time.perf_counter() - t0 < 10.0:
        orc.learn(omem.sample(BT))
        n_cpu += 1
    cpu_val = n_cpu / (time.perf_counter() - t0)
    m, d = res["MATD3"], res["MADDPG"]
    line = {"metric": "population gradient-steps/sec (MATD3 pop=16, 4 agents)", "value": m["value"], "unit": "steps/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "MATD3 learn step (policy_freq 2), 4 agents x 18-dim obs / 5-dim act, batch 64, 100k-step shared "
                                   "HBM replay, pop=16 on one GPU (BASELINE configs[4] shapes; bench.py's MADDPG hyper-parameters)",
                       "pop": POPM, "batch": BT, "buffer": N, "agents": NA, "policy_freq": PF,
                       "net": "actors: LayerNorm MLP [64,64]->32 -> head [64] Tanh; critics (x2 for MATD3): final_dense 72->32 "
                              "ReLU, cat(latent, 20 actions) -> [64] -> 1"},
            "timing": {"repeats": len(m["ms_repeats"]), "stat": "median", "ms_repeats": m["ms_repeats"]},
            "gpu_launches": m["gpu_launches_per_step"], "clocks": clocks, "gpu": gpu_info(0),
            "graph_kernels": {"MATD3": m["graph_kernels"], "MADDPG": d["graph_kernels"]},
            "e2e": m["e2e"],
            "maddpg": {"value": d["value"], "unit": "steps/s", "ms_per_step": d["ms_per_step"], "ms_repeats": d["ms_repeats"],
                       "gpu_launches": d["gpu_launches_per_step"], "e2e": d["e2e"]},
            "matd3_over_maddpg": m["value"] / d["value"],
            "cpu_baseline": {"value": cpu_val, "unit": "steps/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": "10 s of oracle MATD3.learn (bit-exact restatement of the reference) incl. random.sample "
                                       "over a 20k-step deque and the per-agent stacking, one member of the 16"}}
    print(json.dumps(line))


if __name__ == "__main__":
    main()
