#!/usr/bin/env python
"""bench.py — population gradient-steps/sec, Rainbow-DQN pop=8 (BASELINE.json metric, config 2).

    python bench.py --gpus N --steps K --warmup W              # our CUDA path (one rank per GPU)
    python bench.py --impl reference --steps K --warmup W      # the oracle port on host cores
    python bench.py --steps K --warmup W --dump-outputs DIR    # + what the last timed step computed, as DIR/*.npy

One *gradient step* of one agent = PER sample(B, beta) + n-step gather + RainbowDQN.learn
(3 forwards, C51 projection, backward, clip, Adam, Polyak, noise reset) + update_priorities
(SURVEY §8d).  A bench "step" = one such gradient step for EVERY agent of the population
(pop=8, sharded pop/N agents per GPU; total work fixed -> "strong" scaling).

  value : replay resident in HBM, fused device path (no host round trip), CUDA-event timed.
  e2e   : same metric through the reference-shaped Python API with HOST buffers: every step
          H2D-copies one env-step of transitions from pinned memory (memory.add), samples,
          learns, D2H-reads loss + priorities and writes priorities back (update_priorities).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# --- workload constants (BASELINE.md §4, SURVEY §8d) ------------------------------------------------
POP = int(os.environ.get("B2RL_BENCH_POP", "8"))   # BASELINE configs[1]: pop=8 (override only for experiments)
B = 256
OBS = (4, 84, 84)
N_ACT = 6
N_ATOMS = 51
BUFFER = 100_000
ALPHA, BETA, N_STEP, GAMMA = 0.6, 0.4, 3, 0.99
V_MIN, V_MAX = -10.0, 10.0
LR, TAU, PRIOR_EPS = 1e-4, 1e-3, 1e-6
NUM_ENVS = 4                                  # env-steps ingested per e2e step
ALG_BYTES_PER_STEP = 22_954_544               # SURVEY §8d table
ALG_FLOPS_PER_STEP = 12_067_307_520
# dram__bytes_read.sum + dram__bytes_write.sum of one conv_fwd_i8_kernel<8,8> launch (profiles/r2_conv1_i8_single.txt,
# ncu --set full): 7.29 MB read (the 7.2 MB of uint8 frames + weights) + 0 written -- the 13.1 MB of fp32 activations stay
# in the 126 MB L2 for the next layer, so DRAM traffic is BELOW the algorithmic bytes, i.e. no re-reads.
TRAFFIC_CONV1 = 7287808


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return d.get("hbm_gbs", 6650.0), d.get("bf16_tflops", 1590.0), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region: an NVML polling thread (5 ms period, so
    even a 10 ms region is covered); falls back to `nvidia-smi -lms 20` when pynvml cannot be initialised."""
    NAMES = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.thread = None
        self.samples: list = []
        self.reasons: set = set()
        self.max_mhz = None
        self._stop = False
        self.how = None

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            if not uuid.startswith("GPU-"):
                uuid = "GPU-" + uuid
            return pynvml, pynvml.nvmlDeviceGetHandleByUUID(uuid)
        except Exception:
            return pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)

    def _poll(self, nv, h):
        while not self._stop:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
                for bit, name in self.NAMES.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        import threading
        try:
            nv, h = self._nvml_handle()
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, args=(nv, h), daemon=True)
            self.thread.start()
            self.how = "nvml thread, 5 ms"
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.how = "nvidia-smi -lms 20"
        except OSError:
            self.proc = None

    def stop(self) -> dict:
        if self.thread is not None:
            self._stop = True
            self.thread.join(timeout=1.0)
            sm = self.samples
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.max_mhz,
                    "reasons": sorted(self.reasons), "samples": len(sm), "how": self.how}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "how": self.how}


# ---------------------------------------------------------------------------------------------------
def build_rank(device, n_agents, seed0):
    from agilerl_b200.algorithms import RainbowDQN
    from agilerl_b200.compat import TensorDict, spaces
    from agilerl_b200.components import MultiStepReplayBuffer, PrioritizedReplayBuffer

    obs_space = spaces.Box(0, 255, OBS, np.uint8)
    act_space = spaces.Discrete(N_ACT)
    net_config = {"encoder_config": {"channel_size": [32, 32], "kernel_size": [8, 4], "stride_size": [4, 2]},
                  "head_config": {"hidden_size": [64]}, "latent_dim": 32}
    agents = []
    for a in range(n_agents):
        torch.manual_seed(seed0 + a)
        agents.append(RainbowDQN(obs_space, act_space, index=seed0 + a, net_config=dict(net_config), batch_size=B, lr=LR,
                                 gamma=GAMMA, tau=TAU, beta=BETA, prior_eps=PRIOR_EPS, num_atoms=N_ATOMS, v_min=V_MIN,
                                 v_max=V_MAX, n_step=N_STEP, device=device))
    engines = agents
    # one replay pair per rank, shared by the rank's agents (reference: one buffer per process, Q15)
    mem = PrioritizedReplayBuffer(BUFFER, ALPHA, device=device)
    nmem = MultiStepReplayBuffer(BUFFER, N_STEP, GAMMA, device=device)
    mem.device_rng = True
    g = torch.Generator(device=device).manual_seed(seed0)
    chunk = 10_000
    for s in range(0, BUFFER, chunk):          # synthetic 84x84x4 uint8 frames, filled through add()
        n = min(chunk, BUFFER - s)
        for buf in (nmem, mem):
            td = TensorDict({
                "obs": torch.randint(0, 256, (n, *OBS), dtype=torch.uint8, device=device, generator=g),
                "action": torch.randint(0, N_ACT, (n,), device=device, generator=g).float(),
                "next_obs": torch.randint(0, 256, (n, *OBS), dtype=torch.uint8, device=device, generator=g),
                "reward": torch.randn(n, device=device, generator=g),
                "done": (torch.rand(n, device=device, generator=g) < 0.01).float(),
            }, batch_size=[n])
            if buf is nmem:
                from agilerl_b200.components.replay_buffer import ReplayBuffer
                ReplayBuffer.add(nmem, td)      # already-rolled synthetic n-step transitions
                nmem.done_key = "done"
            else:
                buf.add(td)
    # priorities initialised by one pass of |N(0,1)| + 1e-6 (BASELINE.md §4)
    for s in range(0, BUFFER, 4096):
        n = min(4096, BUFFER - s)
        idx = torch.arange(s, s + n, device=device)
        pri = torch.randn(n, device=device, generator=g).abs() + 1e-6
        mem.update_priorities_device(idx, pri)
    torch.cuda.synchronize(device)
    return engines, mem, nmem


def hp():
    return dict(v_min=V_MIN, v_max=V_MAX, delta_z=(V_MAX - V_MIN) / (N_ATOMS - 1), lr=LR, tau=TAU, prior_eps=PRIOR_EPS)


OVERLAP = os.environ.get("B2RL_BENCH_OVERLAP", "1") != "0"


def fused_population_step(agents, mem, nmem, support=None):
    """One learn step of every local agent against the shared HBM replay (agilerl_b200.training.
    population_learn).  The tree is read and written in agent order on one high-priority stream (the
    reference's sequential semantics); each agent's backward + optimiser runs on its own stream under
    the next agents' forwards.  Tails are joined once, at the end of the timed region.  Returns every
    local agent's loss (device tensors)."""
    from agilerl_b200.training.population import population_learn
    return population_learn(agents, mem, nmem, overlap=OVERLAP, join=False)


def api_population_step(agents, mem, nmem, support, host_tr):
    """The public-API path with host buffers — exactly what train_off_policy.py:327-412 does per
    learn step: Transition -> n_step_memory.add -> memory.add -> sampler.sample ->
    n_step_sampler.sample -> agent.learn -> memory.update_priorities."""
    from agilerl_b200.components import Transition
    out = None
    for agent in agents:
        td = Transition(obs=host_tr["obs"], action=host_tr["action"], reward=host_tr["reward"],
                        next_obs=host_tr["next_obs"], done=host_tr["done"], batch_size=[NUM_ENVS]).to_tensordict()
        one = nmem.add(td)                      # H2D + n-step roll + ring write
        if one is not None:
            mem.add(one)                        # ring write + tree leaves
        exp = mem.sample(agent.batch_size, agent.beta)          # tree sample + gather (materialised batch)
        nexp = nmem.sample_from_indices(exp["idxs"].squeeze(1))
        exp["weights"] = exp["weights"].squeeze(1)              # canonical shapes (quirks Q1/Q2 off)
        loss_f, idxs, pri_np = agent.learn(exp, n_experiences=nexp, per=True)   # float + np.ndarray: 2 D2H reads
        mem.update_priorities(idxs, pri_np)
        out = loss_f
    return out


REPEATS = int(os.environ.get("B2RL_BENCH_REPEATS", "5"))
DUMP_BYTES = 48 << 20                         # --dump-outputs budget over the whole population (limit: 64 MB)


def dump_outputs(out_dir, agents, losses):
    """What the last timed step handed back and left behind, per agent: its loss and its online and target
    parameters after the step (float32; a fixed, seeded sample of the parameters where the population's
    would exceed DUMP_BYTES).  Two builds run with the same arguments see the same inputs, so their dumps
    compare array for array."""
    os.makedirs(out_dir, exist_ok=True)
    max_elems = DUMP_BYTES // (2 * POP * 4)
    for agent, loss in zip(agents, losses):
        arrays = {"loss": loss.detach().reshape(-1), "actor_params": agent.actor.buffers.params.detach(),
                  "target_params": agent.actor_target.buffers.params.detach()}
        for name, t in arrays.items():
            a = t.float().cpu().numpy().reshape(-1)
            if a.size > max_elems:
                a = a[np.sort(np.random.default_rng(0).choice(a.size, max_elems, replace=False))]
            np.save(os.path.join(out_dir, f"agent{agent.index}_{name}.npy"), a)


def time_region(fn, steps, dist_on, finish=None, repeats=None):
    """EXACTLY ``steps`` steps between a barrier + synchronize on both sides, CUDA events on the launching
    stream, MAX over ranks — repeated ``repeats`` times; returns (median ms, [ms of every repeat]).
    ``finish`` joins work left on side streams (overlapped learn tails) into the timed stream before the
    closing event, so the region covers every kernel of the K steps."""
    import torch.distributed as dist
    out = []
    for _ in range(repeats or REPEATS):
        if dist_on:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        if finish is not None:
            finish()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if dist_on:
            t = torch.tensor([ms], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
            dist.barrier()
        out.append(ms)
    return statistics.median(out), out


def conv1_roofline(eng, nmem, device):
    """Dominant kernel = first conv layer of the online forward (igemm_kernel<128,32,...>): timed
    alone with CUDA events on the launch stream; inputs are B random ring rows (ring >> L2)."""
    from agilerl_b200 import _lib
    lib = _lib.load()
    desc = eng.layout.desc
    L = desc.enc[0]
    out = torch.empty(B * L.out_c * L.out_h * L.out_w, dtype=torch.float32, device=device)
    ws = torch.empty(64 << 20, dtype=torch.uint8, device=device)
    frames = nmem._fields[("obs",)]
    flops = 2.0 * B * L.out_h * L.out_w * L.out_c * L.in_c * L.ksize * L.ksize
    alg_bytes = B * desc.obs_elems + out.numel() * 4 + (L.out_c * L.in_c * L.ksize * L.ksize + L.out_c) * 4
    stream = _lib.stream_ptr(torch.device(device))

    def launch(idx, reuse):
        _lib.check(lib.b2rl_encoder_layer_forward(ctypes.byref(desc), 0, eng.actor.params.data_ptr(), frames.data_ptr(),
                                                  idx.data_ptr(), B, out.data_ptr(), ws.data_ptr(), ws.numel(), int(reuse),
                                                  stream))
    # the first call splits the weights into digit planes (weight_digits_kernel: once per step in the real loop); the
    # timed launches are the convolution kernel alone, 20 back to back between one pair of events (each on B fresh
    # random rows of the 2.8 GB frame ring, so nothing is L2-resident), which amortises the event/launch latency
    # that would otherwise dominate a ~10 us kernel
    per_batch = 20
    idxs = [torch.randint(0, BUFFER, (B,), device=device) for _ in range(per_batch)]
    launch(idxs[0], False)
    torch.cuda.synchronize()
    times = []
    for it in range(8):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for idx in idxs:
            launch(idx, True)
        e1.record()
        torch.cuda.synchronize()
        if it >= 2:
            times.append(e0.elapsed_time(e1) / per_batch)
    ms = statistics.mean(times)
    desc = {"kernel": "conv_fwd_i8_kernel<8, 8> (digit planes split once per step by weight_digits_kernel, not in the timed launch): conv1 forward (4->32, k8 s4) of B=256 frames gathered "
                      "from the replay ring; persistent warp-specialised kernel, tcgen05.mma kind::i8 over the raw frame bytes "
                      "against four int8 digit planes of the fp32 weights (exact int32 accumulation in TMEM), fp32 "
                      "recombination + bias + ReLU in the epilogue",
            "operand": "int8", "peak_vs_bf16": 2.0, "mmas_per_product": 4,
            # dram__bytes_read.sum + dram__bytes_write.sum per launch, ncu --set full (cold L2): profiles/r2_conv1_i8_*.txt
            "traffic": TRAFFIC_CONV1,
            "note": "uint8 frames read once + fp32 activations written once + weights; fp32-equivalent FLOPs 2*M*N*K, each "
                    "multiply-add costing 4 int8 tensor-core products (one per weight digit plane); nominal int8 dense rate = "
                    "2x bf16"}
    return flops, alg_bytes, ms, desc


# ---------------------------------------------------------------------------------------------------
FRAME_SLOTS = 4096      # distinct frame rows the CPU arm keeps in host RAM (0.46 GB); see cpu_reference


def cpu_reference(steps, warmup, cores):
    """The reference's CPU implementation of one gradient step, as restated by the oracle (pure-Python list
    segment trees like the reference + torch-CPU learn) on the STATED configuration: replay of BUFFER =
    100 000 transitions — trees of capacity 2^17 with every one of the 100 000 leaves set, indices sampled over
    the full range, 17-level descents and write-backs.  Only the frame payload is bounded: row i's frames are
    those of slot i mod 4096 (0.46 GB of host RAM instead of 11.3 GB; the gather still copies B full rows)."""
    from oracle import learn as olearn, nets as onets, replay as oreplay
    from oracle.segtree import PySegTree
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    spec = onets.rainbow_spec(OBS, N_ACT)
    from agilerl_b200.networks.init import init_state_dict
    from agilerl_b200.networks.spec import FlatLayout, rainbow_spec
    layout = FlatLayout(rainbow_spec(OBS, N_ACT, channel_size=(32, 32), kernel_size=(8, 4), stride_size=(4, 2),
                                     obs_low=0.0, obs_high=255.0, obs_u8=True))
    sd = init_state_dict(layout)
    for k, e in layout.entries.items():
        if e.buf == "eps":
            sd[k] = torch.zeros(e.shape)
    agent = olearn.OracleAgent(spec, sd, sd, batch_size=B, lr=LR, v_min=V_MIN, v_max=V_MAX)
    agent.reset_noise()

    class WindowedFrames:
        """gather(idx) over the full index space; frames come from slot idx mod FRAME_SLOTS."""
        def gather(self, idx):
            return {k: v[idx % FRAME_SLOTS] for k, v in self.storage.items()}

    class PER(WindowedFrames, oreplay.OraclePER):
        pass

    class NStep(WindowedFrames, oreplay.OracleReplay):
        pass

    g = torch.Generator().manual_seed(0)
    mem, nmem = PER(BUFFER, ALPHA, tree_cls=PySegTree), NStep(BUFFER)
    for buf in (mem, nmem):
        buf.storage = dict(obs=torch.randint(0, 256, (FRAME_SLOTS, *OBS), dtype=torch.uint8, generator=g),
                           action=torch.randint(0, N_ACT, (FRAME_SLOTS, 1), generator=g).float(),
                           next_obs=torch.randint(0, 256, (FRAME_SLOTS, *OBS), dtype=torch.uint8, generator=g),
                           reward=torch.randn(FRAME_SLOTS, 1, generator=g),
                           done=(torch.rand(FRAME_SLOTS, 1, generator=g) < 0.01).float())
        buf.size = buf.counter = BUFFER
    # priorities |N(0,1)| + 1e-6 on all 100 000 leaves (BASELINE.md section 4), trees built bottom-up in fp64
    cap = mem.sum_tree.capacity
    assert cap == 1 << 17
    pa = np.zeros(cap)
    pri = np.abs(torch.randn(BUFFER, generator=g).numpy().astype(np.float64)) + 1e-6
    pa[:BUFFER] = np.maximum(pri, 1e-5) ** ALPHA
    sums, mins = [pa], [np.where(np.arange(cap) < BUFFER, pa, np.inf)]
    while len(sums[-1]) > 1:
        sums.append(sums[-1][0::2] + sums[-1][1::2])
        mins.append(np.minimum(mins[-1][0::2], mins[-1][1::2]))
    mem.sum_tree.tree = [0.0] + np.concatenate(sums[::-1]).tolist()
    mem.min_tree.tree = [float("inf")] + np.concatenate(mins[::-1]).tolist()
    mem.max_priority = float(pri.max())

    def one_step():
        t0 = time.perf_counter()
        exp = mem.sample(B, BETA)
        nexp = nmem.gather(exp["idxs"].squeeze(1))
        exp["weights"] = exp["weights"].squeeze(1)
        loss, idxs, pri = agent.learn_rainbow(exp, nexp, per=True)
        mem.update_priorities(idxs, pri)
        return time.perf_counter() - t0

    # the host's best thread count for this workload (oversubscribing a many-core box slows torch's CPU
    # convolutions down): one probe step per candidate, keep the fastest
    one_step()
    cands = sorted({c for c in (cores, cores // 2, cores // 4, 32, 16) if 1 <= c <= cores}, reverse=True)
    best, best_t = cores, None
    for c in cands:
        torch.set_num_threads(c)
        dt = one_step()
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    torch.set_num_threads(best)
    times = []
    for it in range(warmup + steps):
        dt = one_step()
        if it >= warmup:
            times.append(dt)
    return times, best


CPU_SAMPLE = ("gradient steps of ONE agent of the 8 (B=256; replay of 100 000 transitions: trees of capacity 2^17 with all "
              "leaves set, full index space; frame payload of row i taken from slot i mod 4096 to bound host RAM), "
              "pure-Python segment trees + torch-CPU learn at the fastest probed torch thread count (oracle restatement "
              "of the reference; a Python reference cannot be installed on the box)")


def config_for(world: int) -> dict:
    n_local = POP // world
    return {"workload": "Rainbow-DQN learn step, synthetic 84x84x4 uint8, batch 256, PER+3-step+C51, pop=8 "
                        "(BASELINE configs[1])", "pop": POP, "batch": B, "buffer": BUFFER, "n_actions": N_ACT,
            "atoms": N_ATOMS, "net": "conv[32,32] k[8,4] s[4,2] -> 2592 -> latent 32 -> noisy dueling head [64]",
            "shapes": "canonical ([B] weights, [B,1] reward/done); quirks Q1/Q2 off",
            "parallelism": f"pop{POP}/dp{world} ({n_local} agents per GPU, no data-path collective)",
            "l2": "inputs larger than L2: 11.3 GB replay ring per rank, fresh random rows every step"}


def tournament_generation(agents, world, rank, device):
    """Two generations of TournamentSelection.select on the sharded population (hpo/tournament.py:41-119 with the
    checkpoint transport of utils/utils.py:756-782 replaced by NCCL): per generation one all-gather of (fitness,
    index), identical plan on every rank (asserted), winners moved point to point.  The first generation pays
    NCCL's lazy point-to-point channel set-up; the second is the steady state.  Timed with CUDA events + wall
    clock, max over ranks; OUTSIDE the timed learn region."""
    import torch.distributed as dist
    from agilerl_b200.hpo import TournamentSelection
    n_local = len(agents)
    ts = TournamentSelection(2, True, POP, 1, seed=1)
    gens = []
    for gen in range(2):
        for a in agents:
            a.synchronize()
            a.fitness = [float(((a.index + 3 * gen) * 37) % 11)]      # synthetic evaluation scores
        dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        elite, agents = ts.select(agents)
        e1.record()
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1e3
        elite_pos, slots = ts.last_plan
        plans = [None] * world
        dist.all_gather_object(plans, [elite_pos, [list(x) for x in slots]])
        assert all(p == plans[0] for p in plans), "ranks derived different tournament plans"
        assert len(agents) == n_local and all(a is not None for a in agents)
        moved = sum(1 for slot, (parent, _) in enumerate(slots) if slot // n_local != parent // n_local)
        eng = agents[0].engine
        per_agent = 4 * (2 * eng.actor.params.numel() + 2 * eng.actor.eps.numel() + 2 * eng.exp_avg.numel())
        t = torch.tensor([e0.elapsed_time(e1), wall], device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        gens.append({"ms_device": float(t[0].item()), "ms_wall": float(t[1].item()), "moved_agents": moved,
                     "bytes_moved": moved * per_agent, "elite_index": int(slots[0][1])})
    out = dict(gens[1], bytes_allgather=world * n_local * 16, plans_identical=True, generations=gens,
               note="ms of generation 2 (steady state); winners move by broadcast from their owner over the communicator the "
                    "fitness all_gather uses (no per-pair channel set-up); generation 1 includes NCCL's first-collective set-up")
    return out, agents


def ppo_workload(args):
    """BASELINE configs[3]: PPO, 256 vector envs x 8-dim observations, pop = 8 — the rollout post-processing the
    reference runs on the host after every collection (RolloutBuffer.compute_returns_and_advantages,
    rollout_buffer.py:413-481: D2H, a NumPy loop over T, H2D) plus the global advantage normalisation of
    PPO.learn (ppo.py:831-834).  One "step" = that post-processing for every agent of the population
    (b2rl_gae_scan_normalize: one launch per agent).  T = learn_step / num_envs = 2048 / 256 = 8 (reference
    defaults); B2RL_PPO_T overrides the horizon."""
    from agilerl_b200 import _lib
    from agilerl_b200.components.rollout import compute_returns_and_normalized_advantages
    from oracle import gae as ogae
    E, T = 256, int(os.environ.get("B2RL_PPO_T", "8"))
    device = "cuda:0"
    torch.cuda.set_device(0)
    lib = _lib.load(require_cuda=True)
    rng = np.random.default_rng(0)
    host = [dict(r=rng.standard_normal((T, E)).astype(np.float32), v=rng.standard_normal((T, E)).astype(np.float32),
                 d=rng.random((T, E)) < 0.02, lv=rng.standard_normal(E).astype(np.float32),
                 ld=(rng.random(E) < 0.02).astype(np.float32)) for _ in range(POP)]
    dev = [{k: torch.from_numpy(np.ascontiguousarray(x)).to(device) for k, x in h.items()} for h in host]
    pin = [{k: torch.from_numpy(np.ascontiguousarray(x)).pin_memory() for k, x in h.items()} for h in host]

    def dev_step():
        for a in dev:
            compute_returns_and_normalized_advantages(a["r"], a["d"], a["v"], a["lv"], a["ld"], 0.99, 0.95, True)

    def e2e_step():
        outs = []
        for a in pin:
            adv, ret, nrm = compute_returns_and_normalized_advantages(
                a["r"].to(device, non_blocking=True), a["d"].to(device, non_blocking=True), a["v"].to(device, non_blocking=True),
                a["lv"].to(device, non_blocking=True), a["ld"].to(device, non_blocking=True), 0.99, 0.95, True)
            outs.append((ret.cpu(), nrm.cpu()))                 # the minibatch loop reads returns + normalised advantages
        return outs

    for _ in range(max(args.warmup, 3)):
        dev_step(); e2e_step()
    l0 = lib.b2rl_launch_count()
    ms, ms_all = time_region(dev_step, args.steps, False)
    launches = (lib.b2rl_launch_count() - l0) // len(ms_all)
    ms_e2e, _ = time_region(e2e_step, args.steps, False, repeats=3)
    value = POP * args.steps / (ms / 1e3)
    # the oracle: the reference's NumPy loop + torch normalisation on the host (its own path: the data is already there)
    t0 = time.perf_counter()
    n_cpu = 0
    while time.perf_counter() - t0 < 2.0:
        for h in host:
            adv, ret = ogae.compute_returns_and_advantages(h["r"], h["d"], h["v"], h["lv"], h["ld"], 0.99, 0.95, True)
            ogae.normalize_advantages(adv)
            n_cpu += 1
    cpu_val = n_cpu / (time.perf_counter() - t0)
    hbm_peak, _, peak_kind = peaks()
    alg = T * E * (4 + 1 + 4 + 4 + 4) + T * E * 4 * 3          # scan: r, d, v in, adv, ret out; normalisation: 2 reads + 1 write
    per_launch_ms = ms / args.steps / POP
    line = {"metric": "PPO rollout post-processing (GAE scan + advantage normalisation), rollouts/sec, pop=8",
            "value": value, "unit": "rollouts/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": f"PPO GAE + advantage normalisation, {E} vector envs x T={T} steps per rollout, pop={POP} "
                                   "(BASELINE configs[3])", "pop": POP, "envs": E, "T": T,
                       "l2": "inputs are a few KB: latency-bound by T dependent float64 steps, not by HBM"},
            "timing": {"repeats": len(ms_all), "stat": "median", "ms_repeats": [round(x, 4) for x in ms_all]},
            "gpu_launches": int(launches),
            "roofline": {"kernel": "gae_fused_kernel (one CTA: thread e walks environment e backwards in float64, the CTA then "
                                   "normalises the T x E advantages)", "bound": "hbm",
                         "achieved": alg / (per_launch_ms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                         "frac": alg / (per_launch_ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
                         "alg_bytes_per_launch": alg, "ms_per_launch": per_launch_ms,
                         "note": "timed inside the population loop incl. the host call; a serial recurrence of T dependent fp64 "
                                 "steps per environment — latency-bound by construction (SURVEY 8f-2)"},
            "e2e": {"value": POP * args.steps / (ms_e2e / 1e3), "unit": "rollouts/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": POP * (T * E * 9 + E * 8), "d2h_bytes_per_step": POP * T * E * 8},
            "cpu_baseline": {"value": cpu_val, "unit": "rollouts/s", "cores": 1, "kind": "port",
                             "sample": "2 s of oracle.gae (the reference's NumPy loop, bit-exact restatement) + torch normalisation "
                                       "per rollout, host arrays in place (no copies counted)"}}
    print(json.dumps(line))


def td3_workload(args):
    """BASELINE configs[2]: TD3, 17-dim observations / 6-dim actions, batch 512, 1M-transition HBM replay, pop = 8.
    One "step" = one learn call of every agent of the population against the shared uniform replay.
      value : device-resident loop — distinct uniform indices drawn on device, one multi-field gather, b2rl_ddpg_learn,
              losses left on the device;
      e2e   : the reference-shaped API with host numbers — ReplayBuffer.sample (torch.randperm(1M) on the host: the
              reference's own sampling cost, replay_buffer.py:125), agent.learn -> Python floats."""
    from agilerl_b200 import _lib
    from agilerl_b200.algorithms import TD3
    from agilerl_b200.compat import TensorDict, spaces
    from agilerl_b200.components import ReplayBuffer
    from oracle import ddpg_td3 as od
    device, BT, N, OD, AD = "cuda:0", 512, 1_000_000, 17, 6
    torch.cuda.set_device(0)
    lib = _lib.load(require_cuda=True)
    obs_space, act_space = spaces.Box(-np.inf, np.inf, (OD,), np.float32), spaces.Box(-1.0, 1.0, (AD,), np.float32)
    agents = []
    for a in range(POP):
        torch.manual_seed(a)
        agents.append(TD3(obs_space, act_space, index=a, batch_size=BT, lr_actor=1e-4, lr_critic=1e-3, device=device))
    mem = ReplayBuffer(N, device=device)
    g = torch.Generator(device=device).manual_seed(0)
    for s0 in range(0, N, 250_000):
        n = min(250_000, N - s0)
        mem.add(TensorDict({"obs": torch.randn(n, OD, device=device, generator=g),
                            "action": torch.rand(n, AD, device=device, generator=g) * 2 - 1,
                            "reward": torch.randn(n, device=device, generator=g),
                            "next_obs": torch.randn(n, OD, device=device, generator=g),
                            "done": (torch.rand(n, device=device, generator=g) < 0.01).float()}, batch_size=[n]))
    torch.cuda.synchronize()

    def dev_step():
        out = None
        for agent in agents:
            out, _ = agent.learn_device(mem.sample_device(BT))
        return out

    def api_step():
        out = None
        for agent in agents:
            out = agent.learn(mem.sample(BT))
        return out

    for _ in range(max(args.warmup, 3)):
        dev_step()
    api_step()
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    l0 = lib.b2rl_launch_count()
    ms, ms_all = time_region(dev_step, args.steps, False)
    launches = (lib.b2rl_launch_count() - l0) // len(ms_all)
    clocks = sampler.stop()
    value = POP * args.steps / (ms / 1e3)
    e2e_steps = max(1, min(args.steps, 20))                  # ~8 ms of host randperm(1M) per agent-step
    ms_e2e, ms_e2e_all = time_region(api_step, e2e_steps, False, repeats=3)
    # CPU arm: the oracle (bit-exact restatement of the reference's TD3.learn) + the reference's host sampling
    cpu = lambda net: {k: v.cpu().clone() for k, v in net.state_dict().items()}
    a0 = agents[0]
    orc = od.OracleDDPG(od.actor_specs(OD, AD, head_hidden=[32]), od.critic_specs(OD, AD, head_hidden=[64]), cpu(a0.actor),
                        cpu(a0.actor_target), [cpu(c) for c in a0._critics()], [cpu(t) for t in a0._targets()], gamma=0.99,
                        tau=0.005, lr_actor=1e-4, lr_critic=1e-3, policy_freq=2, twin=True)
    host_store = {k: v[:200_000].cpu() for k, v in mem._fields.items()}
    t0, n_cpu = time.perf_counter(), 0
    while time.perf_counter() - t0 < 10.0:
        idx = torch.randperm(N)[:BT] % 200_000
        exp = {k[0]: v[idx].clone() for k, v in host_store.items()}
        orc.learn(exp)
        n_cpu += 1
    cpu_val = n_cpu / (time.perf_counter() - t0)
    hbm_peak, _, peak_kind = peaks()
    n_par = sum(n.layout.n_param_elems for n in (a0.actor, a0.critic_1, a0.critic_2))
    alg = BT * (2 * OD + AD + 2) * 4 + 12 * n_par * 4       # gathered rows + (read/grad/Adam/Polyak) parameter traffic
    per_call_ms = ms / args.steps / POP
    line = {"metric": "population gradient-steps/sec (TD3 pop=8)", "value": value, "unit": "steps/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "TD3 learn step, 17-dim obs / 6-dim act, batch 512, 1M-transition HBM replay, pop=8 "
                                   "(BASELINE configs[2])", "pop": POP, "batch": BT, "buffer": N,
                       "net": "MLP encoder [64,64]->32 (no LayerNorm); actor head [32] Tanh; twin critics cat(latent, action) -> [64] -> 1",
                       "l2": "168 MB replay: random 168-byte rows; the step is launch/latency-bound, not HBM-bound"},
            "timing": {"repeats": len(ms_all), "stat": "median", "ms_repeats": [round(x, 3) for x in ms_all]},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"kernel": "whole b2rl_ddpg_learn call (26 launches: fused chain forward / backward / weight-gradient "
                                   "kernels over 64-wide MLPs)", "bound": "hbm", "achieved": alg / (per_call_ms * 1e-3) / 1e9,
                         "peak": hbm_peak, "unit": "GB/s", "frac": alg / (per_call_ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
                         "alg_bytes_per_launch": alg, "ms_per_launch": per_call_ms,
                         "note": "tiny networks (28 k parameters in the three learning nets): bound by ~26 dependent launches"},
            "e2e": {"value": POP * e2e_steps / (ms_e2e / 1e3), "unit": "steps/s", "ms_per_step": ms_e2e / e2e_steps,
                    "h2d_bytes_per_step": POP * BT * 8, "d2h_bytes_per_step": POP * 8, "steps": e2e_steps,
                    "ms_repeats": [round(x, 3) for x in ms_e2e_all]},
            "cpu_baseline": {"value": cpu_val, "unit": "steps/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": "10 s of oracle TD3.learn (bit-exact restatement of the reference) incl. torch.randperm(1M) "
                                       "sampling and the row gather, one agent of the 8"}}
    print(json.dumps(line))


def maddpg_workload(args):
    """BASELINE configs[4]: MADDPG, 4 agents x 18-dim observations (5-dim continuous actions), ONE shared replay,
    pop = 16, hyper-parameters of the reference's configs/training/multi_agent/maddpg.yaml (batch 64, 100 k-step memory,
    lr 1e-4 / 1e-3, tau 1e-3, gamma 0.95).  One "step" = one learn call of every member of the population.
      value : device-resident loop — distinct uniform positions drawn on device, one gather launch over the five field
              rings (agents side by side), b2rl_maddpg_learn, losses left on the device;
      e2e   : the reference-shaped API with host numbers — MultiAgentReplayBuffer.sample (Python random.sample, indices
              H2D), MADDPG.learn -> {agent: (float, float)};
      plus one mutation sweep: Gaussian parameter mutation of the whole population on the device."""
    from agilerl_b200 import _lib
    from agilerl_b200.algorithms import MADDPG
    from agilerl_b200.compat import spaces
    from agilerl_b200.components import MultiAgentReplayBuffer
    from agilerl_b200.hpo import Mutations
    from oracle import maddpg as om
    device, BT, N, NA, OD, AD, POPM = "cuda:0", 64, 100_000, 4, 18, 5, 16
    torch.cuda.set_device(0)
    lib = _lib.load(require_cuda=True)
    ids = [f"agent_{i}" for i in range(NA)]
    obs_sp = [spaces.Box(-np.inf, np.inf, (OD,), np.float32) for _ in ids]
    act_sp = [spaces.Box(-1.0, 1.0, (AD,), np.float32) for _ in ids]
    agents = []
    for a in range(POPM):
        torch.manual_seed(a)
        agents.append(MADDPG(obs_sp, act_sp, agent_ids=ids, index=a, batch_size=BT, lr_actor=1e-4, lr_critic=1e-3, tau=1e-3,
                             gamma=0.95, device=device))
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
    assert len(mem) == N

    from agilerl_b200.training.population import multi_agent_population_learn
    overlap = [True]

    def dev_step():                    # per member: position draw + gather into the buffers its captured learn call reads + graph
        return multi_agent_population_learn(agents, mem, BT, overlap=overlap[0])[-1]

    def api_step():
        out = None
        for agent in agents:
            out = agent.learn(mem.sample(BT))
        return out

    for _ in range(max(args.warmup, 3)):
        dev_step()
    api_step()
    torch.cuda.synchronize()
    sampler = ClockSampler(0)
    sampler.start()
    l0 = lib.b2rl_launch_count()
    ms, ms_all = time_region(dev_step, args.steps, False)
    launches = (lib.b2rl_launch_count() - l0) // len(ms_all)
    clocks = sampler.stop()
    value = POPM * args.steps / (ms / 1e3)
    variants = {}                      # the same loop with members one after another / without the graph / without agent streams
    for name, (ov, gr, fan) in {"members serial, graph+agent streams": (False, True, True),
                                "members serial, eager+agent streams": (False, False, True),
                                "members serial, eager, agents serial": (False, False, False),
                                "members overlapped, graph, agents serial": (True, True, False)}.items():
        overlap[0] = ov
        for a in agents:
            a.use_graph, a.concurrent_agents = gr, fan
        dev_step(); dev_step()
        ms_v, _ = time_region(dev_step, args.steps, False, repeats=3)
        variants[name] = POPM * args.steps / (ms_v / 1e3)
    overlap[0] = True
    for a in agents:
        a.use_graph, a.concurrent_agents = True, True
    dev_step()
    e2e_steps = max(1, min(args.steps, 50))
    ms_e2e, ms_e2e_all = time_region(api_step, e2e_steps, False, repeats=3)
    # mutation sweep on the device: every member's four actors (index_put of 10 % of the chosen matrices)
    mut = Mutations(0, 0, 0.5, 1, 0, 0, rand_seed=0, device=device)
    mut.device_parameter_mutation = True
    clones = [a.clone() for a in agents]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    mut.mutation(clones)
    torch.cuda.synchronize()
    sweep_ms = (time.perf_counter() - t0) * 1e3
    # CPU arm: the oracle (bit-exact restatement of the reference's MADDPG.learn) + the reference's deque sampling cost
    a0 = agents[0]
    cpu = lambda net: {k: v.cpu().clone() for k, v in net.state_dict().items()}
    orc = om.OracleMADDPG(ids, {a: om.actor_specs(OD, AD, head_hidden=[64]) for a in ids}, om.critic_head_spec(NA * AD, head_hidden=[64]),
                          {a: cpu(a0.actors[a]) for a in ids}, {a: cpu(a0.actor_targets[a]) for a in ids},
                          {a: cpu(a0.critics[a]) for a in ids}, {a: cpu(a0.critic_targets[a]) for a in ids}, gamma=0.95, tau=1e-3,
                          lr_actor=1e-4, lr_critic=1e-3)
    omem = om.OracleMAReplay(20_000, fields, ids)
    for i in range(20_000):
        omem._add({a: rng.standard_normal(OD, dtype=np.float32) for a in ids}, {a: rng.uniform(-1, 1, AD).astype(np.float32) for a in ids},
                  {a: float(rng.standard_normal()) for a in ids}, {a: rng.standard_normal(OD, dtype=np.float32) for a in ids},
                  {a: bool(rng.uniform() < 0.01) for a in ids})
    t0, n_cpu = time.perf_counter(), 0
    while time.perf_counter() - t0 < 10.0:
        orc.learn(omem.sample(BT))
        n_cpu += 1
    cpu_val = n_cpu / (time.perf_counter() - t0)
    hbm_peak, _, peak_kind = peaks()
    n_par = sum(a0.actors[a].layout.n_param_elems + a0.critics[a].layout.n_param_elems for a in ids)
    alg = BT * (2 * NA * OD + NA * AD + 2 * NA) * 4 + 12 * n_par * 4     # gathered rows + (read/grad/Adam/Polyak) parameter traffic
    per_call_ms = ms / args.steps / POPM
    line = {"metric": "population gradient-steps/sec (MADDPG pop=16, 4 agents)", "value": value, "unit": "steps/s", "n_gpus": 1,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": "MADDPG learn step, 4 agents x 18-dim obs / 5-dim act, batch 64, 100k-step shared HBM replay, "
                                   "pop=16 on one GPU (BASELINE configs[4]; hyper-parameters of the reference's maddpg.yaml)",
                       "pop": POPM, "batch": BT, "buffer": N, "agents": NA,
                       "net": "actors: LayerNorm MLP [64,64]->32 -> head [64] Tanh; critics: final_dense 72->32 ReLU, "
                              "cat(latent, 20 actions) -> [64] -> 1",
                       "l2": "69 MB replay (fits L2): the step is launch/latency-bound (128 kernels in four concurrent per-agent chains, "
                             "replayed as one CUDA graph per member), not HBM-bound"},
            "timing": {"repeats": len(ms_all), "stat": "median", "ms_repeats": [round(x, 3) for x in ms_all]},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"kernel": "whole b2rl_maddpg_learn call (fused chain forward / backward / weight-gradient kernels over "
                                   "18..72-wide MLPs)", "bound": "hbm", "achieved": alg / (per_call_ms * 1e-3) / 1e9,
                         "peak": hbm_peak, "unit": "GB/s", "frac": alg / (per_call_ms * 1e-3) / 1e9 / hbm_peak, "traffic": None,
                         "alg_bytes_per_launch": alg, "ms_per_launch": per_call_ms,
                         "note": "eight tiny networks per member: bound by the chain of dependent launches"},
            "e2e": {"value": POPM * e2e_steps / (ms_e2e / 1e3), "unit": "steps/s", "ms_per_step": ms_e2e / e2e_steps,
                    "h2d_bytes_per_step": POPM * BT * 8, "d2h_bytes_per_step": POPM * NA * 8, "steps": e2e_steps,
                    "ms_repeats": [round(x, 3) for x in ms_e2e_all]},
            "variants_steps_per_s": variants,
            "mutation_sweep": {"ms": sweep_ms, "members": POPM, "networks": POPM * NA,
                               "what": "Mutations.parameter_mutation with device_parameter_mutation on every member"},
            "cpu_baseline": {"value": cpu_val, "unit": "steps/s", "cores": torch.get_num_threads(), "kind": "port",
                             "sample": "10 s of oracle MADDPG.learn (bit-exact restatement of the reference) incl. random.sample "
                                       "over a 20k-step deque and the per-agent stacking, one member of the 16"}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--workload", default="rainbow", choices=["rainbow", "ppo", "td3", "maddpg"],
                    help="rainbow: BASELINE configs[1] (the metric line the driver reads); td3: configs[2]; ppo: configs[3] "
                         "post-processing")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (each agent's loss and updated online "
                         "and target parameters) as DIR/agent<i>_<name>.npy; rainbow workload, --impl ours")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "rainbow" or args.impl != "ours"):
        ap.error("--dump-outputs is implemented for the rainbow workload with --impl ours")
    if args.workload == "ppo":
        return ppo_workload(args)
    if args.workload == "td3":
        return td3_workload(args)
    if args.workload == "maddpg":
        return maddpg_workload(args)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cores = os.cpu_count() or 1

    if args.impl == "reference":
        if rank != 0:
            return
        # a "step" of this arm = a bounded sample of the population step: ONE agent's gradient step (1/8)
        times, cores = cpu_reference(args.steps, args.warmup, cores)
        per_step = statistics.median(times)
        val = 1.0 / per_step                     # gradient-steps/s of ONE agent == population rate on one host
        line = {"metric": "population gradient-steps/sec (Rainbow-DQN pop=8)", "value": val, "unit": "steps/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step * 1e3 * POP,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "impl": "reference", "config": config_for(max(1, args.gpus)),
                "cpu_baseline": {"value": val, "unit": "steps/s", "cores": cores, "kind": "port",
                                 "sample": f"{args.steps} timed " + CPU_SAMPLE,
                                 "ms_p10_p50_p90": [float(np.percentile(times, q)) * 1e3 for q in (10, 50, 90)]},
                "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    device = f"cuda:{local_rank}"
    dist_on = world > 1
    if dist_on:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(device))
    from agilerl_b200 import _lib
    lib = _lib.load(require_cuda=True)

    assert POP % world == 0, "population of 8 must divide over the ranks"
    n_local = POP // world
    engines, mem, nmem = build_rank(device, n_local, seed0=rank * n_local)
    support = torch.linspace(V_MIN, V_MAX, N_ATOMS).to(device)

    # ---- value: fused device path ------------------------------------------------------------
    last = {}

    def step_fn():
        last["losses"] = fused_population_step(engines, mem, nmem, support)

    for _ in range(max(args.warmup, 3)):
        step_fn()
    for a in engines:
        a.synchronize()
    torch.cuda.synchronize()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = lib.b2rl_launch_count()
    join_all = lambda: [a.synchronize() for a in engines]
    prof = os.environ.get("B2RL_PROFILE_REGION") == "1"      # `ncu --profile-from-start off`: only the timed region
    if prof:
        torch.cuda.profiler.start()
    ms, ms_all = time_region(step_fn, args.steps, dist_on, finish=join_all)
    if prof:
        torch.cuda.profiler.stop()
    launches = (lib.b2rl_launch_count() - l0) // len(ms_all)
    clocks = sampler.stop() if rank == 0 else None
    value = POP * args.steps / (ms / 1e3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, engines, last["losses"])

    # ---- e2e: public API with host buffers ----------------------------------------------------
    e2e = None
    if not args.no_e2e:
        g = torch.Generator().manual_seed(123 + rank)
        host_tr = {
            "obs": torch.randint(0, 256, (NUM_ENVS, *OBS), dtype=torch.uint8, generator=g).pin_memory(),
            "action": torch.randint(0, N_ACT, (NUM_ENVS,), generator=g).float().pin_memory(),
            "next_obs": torch.randint(0, 256, (NUM_ENVS, *OBS), dtype=torch.uint8, generator=g).pin_memory(),
            "reward": torch.randn(NUM_ENVS, generator=g).pin_memory(),
            "done": (torch.rand(NUM_ENVS, generator=g) < 0.01).float().pin_memory(),
        }
        mem.device_rng = False                   # API path consumes torch's CPU RNG like the reference
        api_fn = lambda: api_population_step(engines, mem, nmem, support, host_tr)
        for _ in range(max(args.warmup, 3)):
            api_fn()
        ms_e2e, ms_e2e_all = time_region(api_fn, args.steps, dist_on, repeats=3)
        h2d = sum(v.numel() * v.element_size() for v in host_tr.values()) + B * 4 + B * 8      # + uniforms + p_alpha
        d2h = 4 + B * 4
        e2e = {"value": POP * args.steps / (ms_e2e / 1e3), "unit": "steps/s", "ms_per_step": ms_e2e / args.steps,
               "h2d_bytes_per_step": h2d * n_local, "d2h_bytes_per_step": d2h * n_local,
               "ms_repeats": [round(x, 3) for x in ms_e2e_all]}

    # ---- per-generation exchange (N > 1): one tournament on the sharded population -------------
    tournament = None
    if dist_on:
        tournament, engines = tournament_generation(engines, world, rank, device)

    if rank != 0:
        if dist_on:
            torch.distributed.destroy_process_group()
        return

    hbm_peak, tf_peak, peak_kind = peaks()
    flops, kbytes, kms, kdesc = conv1_roofline(engines[0].engine, nmem, device)
    achieved_tf = flops / (kms / 1e3) / 1e12
    # tensor roof of this kernel: fp32-equivalent FLOPs, each multiply-add costing `mmas_per_product` tensor-core
    # products of the operand type used (peak of that type = measured cuBLAS bf16 peak x the nominal type ratio)
    type_peak = tf_peak * kdesc["peak_vs_bf16"]
    tensor_peak_eq = type_peak / kdesc["mmas_per_product"]
    line = {
        "metric": "population gradient-steps/sec (Rainbow-DQN pop=8)", "value": value, "unit": "steps/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": config_for(world),
        "timing": {"repeats": len(ms_all), "stat": "median", "ms_repeats": [round(x, 3) for x in ms_all]},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "step_hbm": {"alg_bytes_per_grad_step": ALG_BYTES_PER_STEP,
                     "achieved_gbs_per_gpu": ALG_BYTES_PER_STEP * value / world / 1e9,
                     "frac_of_peak": ALG_BYTES_PER_STEP * value / world / 1e9 / hbm_peak, "peak_gbs": hbm_peak,
                     "peak": peak_kind},
        # conv1 forward: 1.68 GFLOP over 20.4 MB of algorithmic traffic = 82 FLOP/B, left of the B200 ridge
        # (measured 1678 TFLOP/s / 6.59 TB/s = 255 FLOP/B): the roof that bounds it is HBM; the tensor roof is
        # reported beside it
        "roofline": {"kernel": kdesc["kernel"],
                     "bound": "hbm", "achieved": kbytes / (kms * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                     "frac": kbytes / (kms * 1e-3) / 1e9 / hbm_peak,
                     "traffic": kdesc["traffic"], "peak_kind": peak_kind + " (copy bandwidth, burst)",
                     "alg_bytes_per_launch": kbytes, "flops_per_launch": flops, "ms_per_launch": kms,
                     "tensor": {"achieved": achieved_tf, "unit": "TFLOP/s fp32-equivalent", "peak": tensor_peak_eq,
                                "frac": achieved_tf / tensor_peak_eq, "operand": kdesc["operand"],
                                "mmas_per_product": kdesc["mmas_per_product"],
                                "peak_kind": f"{peak_kind} bf16 cuBLAS peak x {kdesc['peak_vs_bf16']} (nominal "
                                             f"{kdesc['operand']}:bf16 ratio) / {kdesc['mmas_per_product']}"},
                     "note": kdesc["note"],
                     # NOT live: shares and durations from the committed ncu launch list of this command
                     # (profiles/r2_launches_warm_final.txt, 33 kernels / 386 us of kernel time per agent-step) and the
                     # per-kernel table of DESIGN.md par. 5.  The kernel timed live above is the one the round-1 review named
                     # (first-layer forward); after this round's work the LARGEST share of the step is conv2's forward.
                     "step_shares_from_profiles": [
                         {"kernel": "conv_fwd_tc_kernel (conv2 forward 32->32 k4 s2, 3xTF32 gather, 2 launches/step)",
                          "share_of_step_kernel_time": 0.151, "us_per_launch": 39.0, "alg_mbytes_per_launch": 31.6,
                          "frac_of_hbm_peak": 0.12},
                         {"kernel": "conv_fwd_i8_kernel (conv1 forward, the three passes of a step in one launch)",
                          "share_of_step_kernel_time": 0.061, "us_per_launch": 23.2, "alg_mbytes_per_launch": 53.8,
                          "frac_of_hbm_peak": 0.35},
                         {"kernel": "conv_wgrad_tc_kernel (conv2 weight gradient)", "share_of_step_kernel_time": 0.076,
                          "us_per_launch": 29.4, "alg_mbytes_per_launch": 15.8, "frac_of_hbm_peak": 0.07}]},
    }
    if e2e is not None:
        line["e2e"] = e2e
    if tournament is not None:
        line["tournament"] = tournament
    if not args.no_cpu_baseline and world == 1:
        t, used = cpu_reference(5, 1, cores)
        per = statistics.median(t)
        line["cpu_baseline"] = {"value": 1.0 / per, "unit": "steps/s", "cores": used, "kind": "port",
                                "sample": "5 timed " + CPU_SAMPLE}
    print(json.dumps(line))
    if dist_on:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
