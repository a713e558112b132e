"""Population-level fused learn step.

The reference learns the population agent by agent against ONE shared replay
(train_off_policy.py:399-412: sample -> learn -> update_priorities per agent), so agent i+1's sampler
must see the priorities agent i just wrote.  That ordering is kept exactly: sample, forward, loss and
the priority write-back of all agents form one chain on a single (high-priority) stream.  What does
not feed that chain — each agent's backward, optimiser step, Polyak update and noise reset — is left
running on the agent's own stream underneath the following agents' forwards.
"""
from __future__ import annotations

import torch

_HI: dict = {}


def _hi_priority_stream(device) -> "torch.cuda.Stream":
    key = torch.device(device)
    if key not in _HI:
        _HI[key] = torch.cuda.Stream(device=key, priority=-1)
    return _HI[key]


def population_learn(pop, memory, n_step_memory, overlap: bool = True, join: bool = True) -> list:
    """One ``learn_from_buffers`` step for every agent of ``pop`` (all on one device) against the shared
    HBM-resident buffers.  Returns the per-agent losses as device tensors (no host sync).

    ``join=True`` makes the caller's stream wait for every overlapped tail before returning control —
    required before anything writes the buffers (env ingest) or reads parameters through torch
    (evaluation, tournament, mutation).  Loops that call this back to back pass ``join=False`` and
    join once at the end (``agent.synchronize()``)."""
    if not pop:
        return []
    if not overlap:
        return [agent.learn_from_buffers(memory, n_step_memory) for agent in pop]
    device = pop[0]._dev
    cur = torch.cuda.current_stream(device)
    hi = _hi_priority_stream(device)
    hi.wait_stream(cur)
    with torch.cuda.stream(hi):
        # with few local agents the GPU still has room for each backward's weight gradients on a side stream
        # (a lone agent still gains: its priority write-back runs beside its own backward)
        side = 3 if len(pop) <= 2 else 1
        losses = [agent.learn_from_buffers(memory, n_step_memory, overlap=True, side_streams=side) for agent in pop]
    cur.wait_stream(hi)
    for loss in losses:
        loss.record_stream(cur)
    if join:
        for agent in pop:
            agent.synchronize()
    return losses


_MEMBER_STREAMS: dict = {}


def multi_agent_population_learn(pop, memory, batch_size: int | None = None, overlap: bool = True) -> list:
    """One learn call of every member of a MADDPG or MATD3 population (all on one device) against the shared HBM replay
    (train_multi_agent_off_policy: ``experiences = memory.sample(agent.batch_size); agent.learn(experiences)`` per
    member).  The members share nothing that a learn call writes — the replay is only read — so each member's position
    draw, gather (straight into the buffers its captured learn call reads) and graph launch go to the member's own
    stream and overlap; the caller's stream waits for all of them before the function returns.  Returns the members'
    ``[n_agents, 2]`` loss tensors on the device (no host sync)."""
    if not pop:
        return []
    device = pop[0]._dev
    if not overlap:
        return [m.learn_device(memory.sample_device(batch_size or m.batch_size, out=m.batch_buffers(batch_size or m.batch_size),
                                                    packed_only=True)) for m in pop]
    cur = torch.cuda.current_stream(device)
    streams = _MEMBER_STREAMS.setdefault(torch.device(device), [])
    while len(streams) < len(pop):
        streams.append(torch.cuda.Stream(device=device))
    losses = []
    for m, st in zip(pop, streams):
        B = batch_size or m.batch_size
        st.wait_stream(cur)
        if m.graph_ready(B):       # steady state: two C calls + one graph launch on the member's stream, no torch state touched
            sp = st.cuda_stream
            losses.append(m.learn_device(memory.sample_device(B, out=m.batch_buffers(B), packed_only=True, stream=sp), stream=sp))
        else:                      # first call of this member / batch size: allocations and the capture follow torch's current stream
            with torch.cuda.stream(st):
                losses.append(m.learn_device(memory.sample_device(B, out=m.batch_buffers(B), packed_only=True)))
    for st in streams[:len(pop)]:
        cur.wait_stream(st)
    return losses


def share_transitions(transition, device=None, group=None):
    """The reference trains the WHOLE population against one replay buffer (train_off_policy.py:327-345,
    docs/off_policy/index.rst:103): every agent's environment steps land in it.  With the population sharded one
    process per GPU each rank only sees its own agents' steps, so before ingest the ranks exchange them: every
    leaf of the transition is packed into one byte block, ONE all-gather moves the blocks (NCCL on the device,
    gloo on the host), and the result is the transition of all ranks concatenated along the environment
    dimension in rank order — identical on every rank, so every rank's buffer holds the population's experience
    exactly as a single process stepping ``world_size * num_envs`` environments would.  Without an initialised
    process group (or world size 1) the transition is returned unchanged."""
    import torch.distributed as dist
    from ..compat import TensorDict
    from ..components.replay_buffer import _leaf_items, _unflatten
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return transition
    world = dist.get_world_size(group)
    use_cuda = dist.get_backend(group) != "gloo"
    dev = torch.device(device) if (device is not None and use_cuda) else (
        torch.device("cuda", torch.cuda.current_device()) if use_cuda else torch.device("cpu"))
    leaves = [(p, v if isinstance(v, torch.Tensor) else torch.as_tensor(v)) for p, v in _leaf_items(transition)]
    plan, off = [], 0
    for path, v in leaves:
        nb = v.numel() * v.element_size()
        plan.append((path, off, nb, v.dtype, tuple(v.shape)))
        off = (off + nb + 255) & ~255
    total = max(off, 256)
    block = torch.zeros(total, dtype=torch.uint8, device=dev)
    for (path, o, nb, dt, shape), (_, v) in zip(plan, leaves):
        block[o:o + nb].view(dt).view(shape).copy_(v.contiguous(), non_blocking=True)
    gathered = torch.empty(world * total, dtype=torch.uint8, device=dev)
    dist.all_gather_into_tensor(gathered, block, group=group)          # the single exchange of an environment step
    out = {}
    for path, o, nb, dt, shape in plan:
        parts = [gathered[r * total + o:r * total + o + nb].view(dt).view(shape) for r in range(world)]
        out[path] = torch.cat(parts, dim=0)
    n = next(iter(out.values())).shape[0]
    return _unflatten(out, (n,))
