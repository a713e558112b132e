"""Python stand-in for ``b2rl_maddpg_learn`` when it is handed a MATD3 call (test-only; the product has no CPU path):
records the ``twin`` / ``critic_only`` flags, the bias corrections and the critic_2 / actor step-state pointers of every
call, and writes losses the way the library does (the actor column NaN on a critic-only call)."""
import ctypes

import numpy as np

from test_multi_agent_host_cpu import StandIn, _f32


class Matd3StandIn(StandIn):
    def __init__(self):
        super().__init__()
        self.calls = []

    def b2rl_maddpg_workspace_bytes_cfg(self, actors, critics, cfg, out):
        out._obj.value = 8192 if cfg._obj.twin else 4096
        return 0

    def b2rl_maddpg_learn(self, actors, critics, cfg, bufs, stream):
        c, b = cfg._obj, bufs._obj
        n = c.n_agents
        rec = {f[0]: getattr(c, f[0]) for f in c._fields_}
        rec["critic2"] = [b.critic2[i] for i in range(n)]
        rec["critic2_target"] = [b.critic2_target[i] for i in range(n)]
        rec["critic2_m"] = [b.critic2_m[i] for i in range(n)]
        rec["step_state"], rec["actor_step_state"] = b.step_state, b.actor_step_state
        self.calls.append(rec)
        losses = _f32(b.losses, 2 * n).reshape(n, 2)
        losses[:, 1] = np.arange(n) + 0.5
        losses[:, 0] = np.nan if c.critic_only else -np.arange(n) - 1.0
        return 0
