// maddpg.cuh — MADDPG learn() and the on-device Gaussian parameter mutation (SURVEY 8f-4, BASELINE configs[4]);
// included by nn.cu after ddpg.cuh, whose chain helpers and elementwise kernels it reuses.
//
// Replaces agilerl/algorithms/maddpg.py:571-740 (learn / _learn_individual / soft_update) for vector observations
// and continuous actions, with the networks MADDPG.__init__ builds (maddpg.py:272-350):
//   actor_i  = DeterministicActor: LayerNorm MLP encoder -> LayerNorm MLP head, Tanh        (networks/actors.py:78-210)
//   critic_i = ContinuousQNetwork over ALL agents' observations: EvolvableMultiInput without feature nets, i.e.
//              final_dense Linear(sum obs -> latent) + ReLU over the concatenated raw vectors
//              (modules/multi_input.py:404-465), cat(latent, ALL agents' actions) -> LayerNorm MLP head -> 1
//              (networks/q_networks.py:424-425)
// The host hands over the batch as three row-major matrices — obs / next_obs [B, sum obs] and action [B, sum act],
// the agents' columns side by side in agent order (exactly the operands the reference's torch.cat builds) — plus
// reward / done [B, n_agents].  Per learn call, in the reference's order:
//   (0) next actions of EVERY agent from the target actors (before any update of this call)
//   per agent i: (1) Q_i(obs, act), Q'_i(next_obs, next_act)  (2) NaN reward -> 0, NaN done -> 1 (uint8), TD target,
//   MSE  (3) critic backward + Adam (its Polyak update rides in the same launch: critic_target_i is not read again
//   in this call)  (4) a_i = actor_i(obs_i) replaces agent i's columns of the action matrix; -mean Q_i through the
//   UPDATED critic; dQ/da_i columns -> actor backward + Adam (+ Polyak).
// The per-agent steps (1)-(4) are independent of each other and run on one library side stream per agent.
// Same regime as DDPG/TD3: chains of 18..72-wide layers, launch/latency-bound; every chain is one fused launch forward
// and two backward (head_fused.cuh).  4 agents: 128 kernels + 4 device copies per learn call
// (profiles/r2_maddpg_launches_*.txt), replayed as one CUDA graph with a branch per agent (algorithms/maddpg.py).
#pragma once

namespace b2rl {

// dst[r][col0 : col0+n] = src[r][0:n]
__global__ void maddpg_put_cols_kernel(const float *__restrict__ src, int n, float *__restrict__ dst, int ld, int col0, int64_t B) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < B * n; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / n;
        dst[r * ld + col0 + (int)(e - r * n)] = src[e];
    }
}

// maddpg.py:683-700: rewards NaN -> 0; dones NaN -> 1, .to(uint8); y = r + (1 - d) * gamma * Q'; MSE (mean);
// seed dL/dq = 2 (q - y) / B.  One CTA, fixed-order sums.
__global__ void maddpg_td_loss_kernel(const float *__restrict__ q, const float *__restrict__ qn, const float *__restrict__ reward,
                                      const float *__restrict__ done, int ld, float gamma, int64_t B, float *__restrict__ g,
                                      float *__restrict__ loss) {
    __shared__ float red[32];
    float s = 0.f;
    for (int64_t i = threadIdx.x; i < B; i += blockDim.x) {
        float r = reward[i * ld], d = done[i * ld];       // column `agent` of the [B, n_agents] matrices
        r = isnan(r) ? 0.f : r;
        d = isnan(d) ? 1.f : d;
        const unsigned d8 = __float2uint_rz(fminf(fmaxf(d, 0.f), 255.f)) & 0xFFu;      // .to(torch.uint8)
        const float omd = (float)((1u - d8) & 0xFFu);                                   // (1 - dones) in uint8
        const float y = __fadd_rn(r, __fmul_rn(__fmul_rn(omd, gamma), qn[i]));
        const float df = q[i] - y;
        s += df * df;
        g[i] = 2.0f * df / (float)B;
    }
    s = block_reduce_sum(s, red);
    if (threadIdx.x == 0) *loss = s / (float)B;
}

// matd3.py:769-788, the twin-critic TD step: y = r + (1 - d) * gamma * min(Q'1, Q'2) with maddpg_td_loss_kernel's
// NaN handling; critic_loss = MSE(Q1, y) + MSE(Q2, y); seeds dL/dQk = 2 (Qk - y) / B.  One CTA, fixed-order sums.
// actor_loss != NULL (a critic-only call, no actor step): NaN there, so a device-side reader never sees a stale value.
__global__ void matd3_td_loss_kernel(const float *__restrict__ q1, const float *__restrict__ q2, const float *__restrict__ qn1,
                                     const float *__restrict__ qn2, const float *__restrict__ reward, const float *__restrict__ done,
                                     int ld, float gamma, int64_t B, float *__restrict__ g1, float *__restrict__ g2,
                                     float *__restrict__ loss, float *__restrict__ actor_loss) {
    __shared__ float red[32];
    float s1 = 0.f, s2 = 0.f;
    for (int64_t i = threadIdx.x; i < B; i += blockDim.x) {
        float r = reward[i * ld], d = done[i * ld];
        r = isnan(r) ? 0.f : r;
        d = isnan(d) ? 1.f : d;
        const unsigned d8 = __float2uint_rz(fminf(fmaxf(d, 0.f), 255.f)) & 0xFFu;      // .to(torch.uint8)
        const float omd = (float)((1u - d8) & 0xFFu);
        const float a = qn1[i], b = qn2[i];
        const float qn = (isnan(a) || a < b) ? a : b;                                   // torch.min: NaN propagates
        const float y = __fadd_rn(r, __fmul_rn(__fmul_rn(omd, gamma), qn));
        const float d1 = q1[i] - y, d2 = q2[i] - y;
        s1 += d1 * d1;
        s2 += d2 * d2;
        g1[i] = 2.0f * d1 / (float)B;
        g2[i] = 2.0f * d2 / (float)B;
    }
    s1 = block_reduce_sum(s1, red);
    s2 = block_reduce_sum(s2, red);
    if (threadIdx.x == 0) {
        *loss = s1 / (float)B + s2 / (float)B;
        if (actor_loss) *actor_loss = __int_as_float(0x7fc00000);
    }
}

// hpo/mutation.py:733-827 on the device: slot j mutates W[rows[j]][cols[j]] (host-drawn positions and branch
// uniforms, the reference's numpy stream).  branch: u < 0.05 -> w + |10 w| z; u < 0.10 -> z; else w + |sd w| z;
// clamp(+-1e6).  keep[j] == 0 marks a slot whose position is written again by a later slot (index_put_: last writer
// wins); every slot reads the ORIGINAL value (the reference gathers before it scatters): a kept slot is the only
// writer of its element.  z: injected standard normals (parity tests) or the Philox stream.
__global__ void gaussian_mutate_kernel(float *__restrict__ W, int64_t ld, const int64_t *__restrict__ rows,
                                       const int64_t *__restrict__ cols, const float *__restrict__ u,
                                       const uint8_t *__restrict__ keep, const float *__restrict__ z_in, uint64_t seed,
                                       uint64_t offset, float mut_sd, int64_t n) {
    for (int64_t j = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) {
        if (keep && !keep[j]) continue;
        const float z = z_in ? z_in[j] : philox_normal(seed, offset + (uint64_t)j, 0x4D555441ull /* "MUTA" */);
        float *p = W + rows[j] * ld + cols[j];
        const float w = *p, uj = u[j];
        float v;
        if (uj < 0.05f) v = __fadd_rn(w, __fmul_rn(fabsf(__fmul_rn(10.0f, w)), z));
        else if (uj < 0.1f) v = z;
        else v = __fadd_rn(w, __fmul_rn(fabsf(__fmul_rn(mut_sd, w)), z));
        *p = fminf(fmaxf(v, -1000000.0f), 1000000.0f);
    }
}

// torch.optim.Adam (no clipping) + the Polyak update of the target, one flat parameter buffer (tgt == NULL: Adam only, a
// MATD3 call without soft updates).  state != NULL (a captured learn call): this step's bias corrections come from the device block the graph's first node rewrites —
// the same double arithmetic as the host's (lr / bc1, sqrt(bc2)), so a replay is bit-identical to the eager call.
__global__ void ma_adam_polyak_kernel(float *__restrict__ p, const float *__restrict__ g, float *__restrict__ m,
                                      float *__restrict__ v, float *__restrict__ tgt, int64_t n, AdamCfg c, double lr,
                                      const b2rl_step_state *__restrict__ state) {
    if (state) {
        c.neg_step = (float)(-__ddiv_rn(lr, state->bias_correction1));
        c.bc2_sqrt = (float)__dsqrt_rn(state->bias_correction2);
    }
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float gi = g[i];
        float mi = m[i], vi = v[i];
        mi = fmaf(c.w1, gi - mi, mi);                        // exp_avg.lerp_(grad, 1-beta1)
        vi = vi * c.beta2 + c.w2 * gi * gi;                  // mul_(beta2).addcmul_(g, g, 1-beta2)
        m[i] = mi; v[i] = vi;
        const float denom = sqrtf(vi) / c.bc2_sqrt + c.eps;
        const float pi = p[i] + (c.neg_step * mi) / denom;   // addcdiv_(exp_avg, denom, value=-step_size)
        p[i] = pi;
        if (tgt) tgt[i] = __fadd_rn(__fmul_rn(c.tau, pi), __fmul_rn(c.one_minus_tau, tgt[i]));   // soft_update (maddpg.py:733-746)
    }
}
static int ma_adam(float *p, float *g, float *m, float *v, float *tgt, int64_t n, double lr, double bc1, double bc2,
                   const b2rl_maddpg_cfg &cfg, const b2rl_step_state *state, cudaStream_t s) {
    AdamCfg c;
    c.clip = 0; c.max_norm = 0.f;
    c.w1 = (float)(1.0 - cfg.beta1); c.beta2 = (float)cfg.beta2; c.w2 = (float)(1.0 - cfg.beta2);
    c.neg_step = (float)(-(lr / bc1)); c.bc2_sqrt = (float)sqrt(bc2); c.eps = (float)cfg.adam_eps;
    c.tau = (float)cfg.tau; c.one_minus_tau = (float)(1.0 - cfg.tau);
    int blocks = (int)((n + 255) / 256);
    if (blocks > sm_count() * 4) blocks = sm_count() * 4;
    ma_adam_polyak_kernel<<<blocks, 256, 0, s>>>(p, g, m, v, tgt, n, c, lr, state);
    B2RL_LAUNCH_CHECK();
    return B2RL_OK;
}

// One side stream per agent: after the target actions (every agent needs every agent's), the agents' critic / actor
// steps are independent of each other — own networks, own optimiser state, own scratch — so they run concurrently
// and the call's critical path is one agent's chain instead of n.  Library-owned, created once per process; forked
// from and joined back into the caller's stream with events, which a stream capture turns into graph edges.
// A twin call (MATD3) gives every agent a second stream, s[B2RL_MAX_AGENTS + i], for its critic_2 chains: forwards,
// backward and Adam of critic_2 depend on critic_1's only through the TD step, and the actor step reads critic_1 alone.
struct MaStreams {
    cudaStream_t s[2 * B2RL_MAX_AGENTS] = {};
    cudaEvent_t fork = nullptr, ta[B2RL_MAX_AGENTS] = {}, join[B2RL_MAX_AGENTS] = {};
    // twin: fork2 (agent stream -> critic_2 stream), q2 (critic_2's Q values are ready for the TD step), td (its
    // gradient seed is written), join2 (critic_2 stepped)
    cudaEvent_t fork2[B2RL_MAX_AGENTS] = {}, q2[B2RL_MAX_AGENTS] = {}, td[B2RL_MAX_AGENTS] = {}, join2[B2RL_MAX_AGENTS] = {};
    bool ready = false;
};
static int ma_streams(MaStreams **out) {
    static MaStreams ms;
    if (!ms.ready) {
        B2RL_CUDA(cudaEventCreateWithFlags(&ms.fork, cudaEventDisableTiming));
        for (int i = 0; i < B2RL_MAX_AGENTS; ++i) {
            B2RL_CUDA(cudaStreamCreateWithFlags(&ms.s[i], cudaStreamNonBlocking));
            B2RL_CUDA(cudaStreamCreateWithFlags(&ms.s[B2RL_MAX_AGENTS + i], cudaStreamNonBlocking));
            for (cudaEvent_t *e : {&ms.ta[i], &ms.join[i], &ms.fork2[i], &ms.q2[i], &ms.td[i], &ms.join2[i]})
                B2RL_CUDA(cudaEventCreateWithFlags(e, cudaEventDisableTiming));
        }
        ms.ready = true;
    }
    *out = &ms;
    return B2RL_OK;
}

struct MaAgentWS {
    // critic passes: [0] critic(obs, act) with gradients; [1] critic_target(next_obs, next_act); [2] the updated critic
    // on (obs, act with agent i's columns replaced by actor_i(obs_i)) with gradients w.r.t. its input only
    LayerBuf c_enc[3][B2RL_MAX_ENC], c_head[3][B2RL_MAX_HEAD];
    float *cat[3], *g_cat[3];
    LayerBuf a_enc[2][B2RL_MAX_ENC], a_head[2][B2RL_MAX_HEAD];   // [0] actor_i(obs_i) with gradients, [1] actor_target_i(next_obs_i)
    float *obs_i, *nobs_i;           // contiguous copies of agent i's observation columns
    float *act_mod;                  // [B, sum act] the batch's actions with agent i's columns replaced
    float *g_obs;                    // dL/d(input) scratch of the first chains (unused result)
    float *lnpart;                   // LayerNorm-affine partial sums of this agent's backward passes
    // twin only (carved after everything above, so a MADDPG workspace is unchanged): critic_2 passes [0] critic_2(obs, act)
    // with gradients, [1] critic_2_target(next_obs, next_act); own dL/d(input) and LayerNorm scratch (its own stream)
    LayerBuf c2_enc[2][B2RL_MAX_ENC], c2_head[2][B2RL_MAX_HEAD];
    float *cat2[2], *g_cat2, *g_obs2, *lnpart2;
};
struct MaWS {
    MaAgentWS ag[B2RL_MAX_AGENTS];
    float *next_act;                 // [B, sum act] every agent's target action, side by side
    size_t lnpart_floats;
    size_t bytes;
};

struct MaShape { int n; int o_off[B2RL_MAX_AGENTS + 1], a_off[B2RL_MAX_AGENTS + 1]; int L; };

static int ma_shape(const b2rl_net_desc *const *actors, const b2rl_net_desc *const *critics, int n, MaShape &sh) {
    B2RL_CHECK_ARG(actors && critics && n >= 1 && n <= B2RL_MAX_AGENTS, "between 1 and %d agents", B2RL_MAX_AGENTS);
    sh.n = n; sh.o_off[0] = sh.a_off[0] = 0;
    int rc;
    for (int i = 0; i < n; ++i) {
        B2RL_CHECK_ARG(actors[i] && critics[i], "NULL network description");
        const b2rl_net_desc &a = *actors[i];
        if ((rc = chain_check(enc_chain(a))) != B2RL_OK || (rc = chain_check(val_chain(a))) != B2RL_OK ||
            (rc = chain_check(enc_chain(*critics[i]))) != B2RL_OK || (rc = chain_check(val_chain(*critics[i]))) != B2RL_OK)
            return rc;
        B2RL_CHECK_ARG(a.val[0].in_c == a.enc[a.n_enc - 1].out_c, "actor head does not fit its encoder");
        sh.o_off[i + 1] = sh.o_off[i] + a.enc[0].in_c;
        sh.a_off[i + 1] = sh.a_off[i] + a.val[a.n_val - 1].out_c;
    }
    sh.L = critics[0]->enc[critics[0]->n_enc - 1].out_c;
    for (int i = 0; i < n; ++i) {
        const b2rl_net_desc &c = *critics[i];
        B2RL_CHECK_ARG(c.enc[0].in_c == sh.o_off[n], "critic encoder must take every agent's observation (%d inputs, got %d)",
                       sh.o_off[n], c.enc[0].in_c);
        B2RL_CHECK_ARG(c.enc[c.n_enc - 1].out_c == sh.L && c.val[0].in_c == sh.L + sh.a_off[n],
                       "critic head must take cat(latent, every agent's action)");
        B2RL_CHECK_ARG(c.val[c.n_val - 1].out_c == 1, "critic head must end in one value");
    }
    return B2RL_OK;
}

static void carve_maddpg(const b2rl_net_desc *const *actors, const b2rl_net_desc *const *critics, const MaShape &sh, int64_t B,
                         bool twin, void *base, MaWS &ws) {
    Bump b(base);
    const int SO = sh.o_off[sh.n], SA = sh.a_off[sh.n];
    ws.next_act = b.take<float>(B * SA);
    const int64_t tiles = (B + kHeadRows - 1) / kHeadRows;
    ws.lnpart_floats = (size_t)tiles * 2 * kHeadWgMaxIn * 4;
    for (int i = 0; i < sh.n; ++i) {
        MaAgentWS &w = ws.ag[i];
        w.act_mod = b.take<float>(B * SA);
        w.g_obs = b.take<float>(B * SO);
        w.lnpart = b.take<float>(ws.lnpart_floats);
        const b2rl_net_desc &a = *actors[i], &c = *critics[i];
        for (int p = 0; p < 3; ++p) {
            const bool grad = p != 1;
            carve_layers(b, c.enc, c.n_enc, w.c_enc[p], B, grad ? B : 0);
            carve_layers(b, c.val, c.n_val, w.c_head[p], B, grad ? B : 0);
            w.cat[p] = b.take<float>(B * (sh.L + SA));
            w.g_cat[p] = grad ? b.take<float>(B * (sh.L + SA)) : nullptr;
        }
        for (int p = 0; p < 2; ++p) {
            carve_layers(b, a.enc, a.n_enc, w.a_enc[p], B, p == 0 ? B : 0);
            carve_layers(b, a.val, a.n_val, w.a_head[p], B, p == 0 ? B : 0);
        }
        w.obs_i = b.take<float>(B * a.enc[0].in_c);
        w.nobs_i = b.take<float>(B * a.enc[0].in_c);
    }
    for (int i = 0; twin && i < sh.n; ++i) {     // critic_2 shares critic_1's description (same architecture)
        MaAgentWS &w = ws.ag[i];
        const b2rl_net_desc &c = *critics[i];
        for (int p = 0; p < 2; ++p) {
            carve_layers(b, c.enc, c.n_enc, w.c2_enc[p], B, p == 0 ? B : 0);
            carve_layers(b, c.val, c.n_val, w.c2_head[p], B, p == 0 ? B : 0);
            w.cat2[p] = b.take<float>(B * (sh.L + SA));
        }
        w.g_cat2 = b.take<float>(B * (sh.L + SA));
        w.g_obs2 = b.take<float>(B * SO);
        w.lnpart2 = b.take<float>(ws.lnpart_floats);
    }
    ws.bytes = b.off + 256;
}

// enc(obs) -> cat(latent, action) -> head
static int ma_critic_forward(const b2rl_net_desc &critic, const float *params, const float *obs, const float *action, int64_t B,
                             const LayerBuf *enc_bufs, const LayerBuf *head_bufs, float *cat, int L, int SA, cudaStream_t s) {
    int rc = chain_forward(enc_chain(critic), params, obs, B, enc_bufs, s);
    if (rc != B2RL_OK) return rc;
    ddpg_concat_kernel<<<ew_blocks(B * (L + SA)), 256, 0, s>>>(enc_bufs[critic.n_enc - 1].a, L, action, SA, B, cat);
    B2RL_LAUNCH_CHECK();
    return chain_forward(val_chain(critic), params, cat, B, head_bufs, s);
}

}  // namespace b2rl

using namespace b2rl;

extern "C" {

static int maddpg_workspace_bytes(const b2rl_net_desc *const *actors_host, const b2rl_net_desc *const *critics_host, int n_agents,
                                  int64_t batch, bool twin, size_t *out_host) {
    B2RL_CHECK_ARG(out_host && batch >= 1, "bad arguments");
    MaShape sh;
    int rc = ma_shape(actors_host, critics_host, n_agents, sh);
    if (rc != B2RL_OK) return rc;
    MaWS ws;
    carve_maddpg(actors_host, critics_host, sh, batch, twin, nullptr, ws);
    *out_host = ws.bytes;
    MaStreams *ms;                       // everything a later stream capture must not create: side streams, events,
    if ((rc = ma_streams(&ms)) != B2RL_OK) return rc;     // kernel attributes
    return head_kernels_ready();
}

int b2rl_maddpg_workspace_bytes(const b2rl_net_desc *const *actors_host, const b2rl_net_desc *const *critics_host, int n_agents,
                                int64_t batch, size_t *out_host) {
    return maddpg_workspace_bytes(actors_host, critics_host, n_agents, batch, false, out_host);
}

int b2rl_maddpg_workspace_bytes_cfg(const b2rl_net_desc *const *actors_host, const b2rl_net_desc *const *critics_host,
                                    const b2rl_maddpg_cfg *cfg_host, size_t *out_host) {
    B2RL_CHECK_ARG(cfg_host, "NULL descriptor");
    return maddpg_workspace_bytes(actors_host, critics_host, cfg_host->n_agents, cfg_host->batch, cfg_host->twin != 0, out_host);
}

int b2rl_maddpg_learn(const b2rl_net_desc *const *actors_host, const b2rl_net_desc *const *critics_host,
                      const b2rl_maddpg_cfg *cfg_host, const b2rl_maddpg_bufs *bufs_host, void *stream) {
    B2RL_CHECK_ARG(cfg_host && bufs_host, "NULL descriptor");
    const b2rl_maddpg_cfg &cfg = *cfg_host;
    const b2rl_maddpg_bufs &bf = *bufs_host;
    const int64_t B = cfg.batch;
    const int n = cfg.n_agents;
    const bool twin = cfg.twin != 0, critic_only = cfg.critic_only != 0;
    B2RL_CHECK_ARG(B >= 1, "Batch size must be greater than or equal to one.");
    MaShape sh;
    int rc = ma_shape(actors_host, critics_host, n, sh);
    if (rc != B2RL_OK) return rc;
    B2RL_CHECK_ARG(bf.obs && bf.next_obs && bf.action && bf.reward && bf.done && bf.losses, "NULL batch buffer");
    for (int i = 0; i < n; ++i) {
        B2RL_CHECK_ARG(bf.actor[i] && bf.actor_target[i] && bf.actor_grads[i] && bf.actor_m[i] && bf.actor_v[i] && bf.critic[i] &&
                           bf.critic_target[i] && bf.critic_grads[i] && bf.critic_m[i] && bf.critic_v[i],
                       "NULL network buffer of agent %d", i);
        B2RL_CHECK_ARG(!twin || (bf.critic2[i] && bf.critic2_target[i] && bf.critic2_grads[i] && bf.critic2_m[i] && bf.critic2_v[i]),
                       "NULL critic_2 buffer of agent %d", i);
    }
    MaWS ws;
    carve_maddpg(actors_host, critics_host, sh, B, twin, bf.workspace, ws);
    B2RL_CHECK_ARG(bf.workspace && bf.workspace_bytes >= ws.bytes, "workspace too small: need %zu bytes, got %zu", ws.bytes,
                   bf.workspace_bytes);
    cudaStream_t s = as_stream(stream);
    const int SO = sh.o_off[n], SA = sh.a_off[n], L = sh.L;
    const b2rl_step_state *state = static_cast<const b2rl_step_state *>(bf.step_state);
    const b2rl_step_state *actor_state = bf.actor_step_state ? static_cast<const b2rl_step_state *>(bf.actor_step_state) : state;
    const bool fan = !cfg.serial && n > 1;
    const bool fan2 = !cfg.serial && twin;
    MaStreams *ms = nullptr;
    if (fan || fan2) {
        if ((rc = ma_streams(&ms)) != B2RL_OK) return rc;
        if (fan) B2RL_CUDA(cudaEventRecord(ms->fork, s));
    }

    // (0) next actions of every agent from the target actors (maddpg.py:600-609), side by side like torch.cat(dim=1)
    for (int j = 0; j < n; ++j) {
        const b2rl_net_desc &a = *actors_host[j];
        MaAgentWS &w = ws.ag[j];
        cudaStream_t sj = fan ? ms->s[j] : s;
        if (fan) B2RL_CUDA(cudaStreamWaitEvent(sj, ms->fork, 0));
        const int o = sh.o_off[j + 1] - sh.o_off[j], ad = sh.a_off[j + 1] - sh.a_off[j];
        ddpg_slice_kernel<<<ew_blocks(B * o), 256, 0, sj>>>(bf.next_obs, SO, sh.o_off[j], o, B, w.nobs_i);
        B2RL_LAUNCH_CHECK();
        if ((rc = chain_forward(enc_chain(a), bf.actor_target[j], w.nobs_i, B, w.a_enc[1], sj)) != B2RL_OK) return rc;
        if ((rc = chain_forward(val_chain(a), bf.actor_target[j], w.a_enc[1][a.n_enc - 1].a, B, w.a_head[1], sj)) != B2RL_OK) return rc;
        maddpg_put_cols_kernel<<<ew_blocks(B * ad), 256, 0, sj>>>(w.a_head[1][a.n_val - 1].a, ad, ws.next_act, SA, sh.a_off[j], B);
        B2RL_LAUNCH_CHECK();
        if (fan) B2RL_CUDA(cudaEventRecord(ms->ta[j], sj));
    }
    for (int i = 0; i < n; ++i) {
        const b2rl_net_desc &a = *actors_host[i], &c = *critics_host[i];
        MaAgentWS &w = ws.ag[i];
        cudaStream_t si = fan ? ms->s[i] : s;
        if (fan)
            for (int j = 0; j < n; ++j)
                if (j != i) B2RL_CUDA(cudaStreamWaitEvent(si, ms->ta[j], 0));
        const Chain ae = enc_chain(a), ah = val_chain(a), ce = enc_chain(c), ch = val_chain(c);
        const int o = sh.o_off[i + 1] - sh.o_off[i], ad = sh.a_off[i + 1] - sh.a_off[i];
        cudaStream_t s2 = fan2 ? ms->s[B2RL_MAX_AGENTS + i] : si;
        if (fan2) {
            B2RL_CUDA(cudaEventRecord(ms->fork2[i], si));
            B2RL_CUDA(cudaStreamWaitEvent(s2, ms->fork2[i], 0));
        }
        // (1) Q_i(obs, act) and the target Q'_i(next_obs, next_act) (twin: the same two passes of critic_2 on s2)
        if (twin) {
            if ((rc = ma_critic_forward(c, bf.critic2[i], bf.obs, bf.action, B, w.c2_enc[0], w.c2_head[0], w.cat2[0], L, SA, s2)) != B2RL_OK)
                return rc;
            if ((rc = ma_critic_forward(c, bf.critic2_target[i], bf.next_obs, ws.next_act, B, w.c2_enc[1], w.c2_head[1], w.cat2[1], L, SA,
                                        s2)) != B2RL_OK)
                return rc;
            if (fan2) B2RL_CUDA(cudaEventRecord(ms->q2[i], s2));
        }
        if ((rc = ma_critic_forward(c, bf.critic[i], bf.obs, bf.action, B, w.c_enc[0], w.c_head[0], w.cat[0], L, SA, si)) != B2RL_OK) return rc;
        if ((rc = ma_critic_forward(c, bf.critic_target[i], bf.next_obs, ws.next_act, B, w.c_enc[1], w.c_head[1], w.cat[1], L, SA, si)) != B2RL_OK)
            return rc;
        // (2) TD target, MSE, dL/dq seed
        if (twin) {
            if (fan2) B2RL_CUDA(cudaStreamWaitEvent(si, ms->q2[i], 0));
            matd3_td_loss_kernel<<<1, 512, 0, si>>>(w.c_head[0][c.n_val - 1].a, w.c2_head[0][c.n_val - 1].a, w.c_head[1][c.n_val - 1].a,
                                                    w.c2_head[1][c.n_val - 1].a, bf.reward + i, bf.done + i, n, (float)cfg.gamma, B,
                                                    w.c_head[0][c.n_val - 1].g, w.c2_head[0][c.n_val - 1].g, bf.losses + 2 * i + 1,
                                                    critic_only ? bf.losses + 2 * i : nullptr);
            B2RL_LAUNCH_CHECK();
            if (fan2) {
                B2RL_CUDA(cudaEventRecord(ms->td[i], si));
                B2RL_CUDA(cudaStreamWaitEvent(s2, ms->td[i], 0));
            }
        } else {
            maddpg_td_loss_kernel<<<1, 512, 0, si>>>(w.c_head[0][c.n_val - 1].a, w.c_head[1][c.n_val - 1].a, bf.reward + i, bf.done + i, n,
                                                     (float)cfg.gamma, B, w.c_head[0][c.n_val - 1].g, bf.losses + 2 * i + 1);
            B2RL_LAUNCH_CHECK();
            if (critic_only) B2RL_CUDA(cudaMemsetAsync(bf.losses + 2 * i, 0xFF, sizeof(float), si));     // all-ones bits: a NaN
        }
        // (3) critic backward + Adam (+ Polyak unless critic-only); twin: critic_2's on s2, beside critic_1's
        if (twin) {
            if ((rc = chain_backward(ch, bf.critic2[i], w.cat2[0], B, w.c2_head[0], w.g_cat2, bf.critic2_grads[i], w.lnpart2,
                                     ws.lnpart_floats, s2)) != B2RL_OK)
                return rc;
            ddpg_slice_kernel<<<ew_blocks(B * L), 256, 0, s2>>>(w.g_cat2, L + SA, 0, L, B, w.c2_enc[0][c.n_enc - 1].g);
            B2RL_LAUNCH_CHECK();
            if ((rc = chain_backward(ce, bf.critic2[i], bf.obs, B, w.c2_enc[0], w.g_obs2, bf.critic2_grads[i], w.lnpart2, ws.lnpart_floats,
                                     s2)) != B2RL_OK)
                return rc;
            if ((rc = ma_adam(bf.critic2[i], bf.critic2_grads[i], bf.critic2_m[i], bf.critic2_v[i], critic_only ? nullptr : bf.critic2_target[i],
                              c.n_params, cfg.lr_critic, cfg.bc1_critic, cfg.bc2_critic, cfg, state, s2)) != B2RL_OK)
                return rc;
            if (fan2) B2RL_CUDA(cudaEventRecord(ms->join2[i], s2));
        }
        if ((rc = chain_backward(ch, bf.critic[i], w.cat[0], B, w.c_head[0], w.g_cat[0], bf.critic_grads[i], w.lnpart,
                                 ws.lnpart_floats, si)) != B2RL_OK)
            return rc;
        ddpg_slice_kernel<<<ew_blocks(B * L), 256, 0, si>>>(w.g_cat[0], L + SA, 0, L, B, w.c_enc[0][c.n_enc - 1].g);
        B2RL_LAUNCH_CHECK();
        if ((rc = chain_backward(ce, bf.critic[i], bf.obs, B, w.c_enc[0], w.g_obs, bf.critic_grads[i], w.lnpart, ws.lnpart_floats,
                                 si)) != B2RL_OK)
            return rc;
        if ((rc = ma_adam(bf.critic[i], bf.critic_grads[i], bf.critic_m[i], bf.critic_v[i], critic_only ? nullptr : bf.critic_target[i],
                          c.n_params, cfg.lr_critic, cfg.bc1_critic, cfg.bc2_critic, cfg, state, si)) != B2RL_OK)
            return rc;
        // (4) actor step through the UPDATED critic_i: -mean Q_i(obs, [act_0 .. actor_i(obs_i) .. act_n-1])
        if (!critic_only) {
            ddpg_slice_kernel<<<ew_blocks(B * o), 256, 0, si>>>(bf.obs, SO, sh.o_off[i], o, B, w.obs_i);
            B2RL_LAUNCH_CHECK();
            if ((rc = chain_forward(ae, bf.actor[i], w.obs_i, B, w.a_enc[0], si)) != B2RL_OK) return rc;
            if ((rc = chain_forward(ah, bf.actor[i], w.a_enc[0][a.n_enc - 1].a, B, w.a_head[0], si)) != B2RL_OK) return rc;
            B2RL_CUDA(cudaMemcpyAsync(w.act_mod, bf.action, sizeof(float) * B * SA, cudaMemcpyDeviceToDevice, si));
            maddpg_put_cols_kernel<<<ew_blocks(B * ad), 256, 0, si>>>(w.a_head[0][a.n_val - 1].a, ad, w.act_mod, SA, sh.a_off[i], B);
            B2RL_LAUNCH_CHECK();
            if ((rc = ma_critic_forward(c, bf.critic[i], bf.obs, w.act_mod, B, w.c_enc[2], w.c_head[2], w.cat[2], L, SA, si)) != B2RL_OK)
                return rc;
            ddpg_actor_loss_kernel<<<1, 512, 0, si>>>(w.c_head[2][c.n_val - 1].a, B, w.c_head[2][c.n_val - 1].g, bf.losses + 2 * i);
            B2RL_LAUNCH_CHECK();
            if ((rc = chain_backward(ch, bf.critic[i], w.cat[2], B, w.c_head[2], w.g_cat[2], nullptr, w.lnpart, ws.lnpart_floats, si)) !=
                B2RL_OK)
                return rc;
            ddpg_slice_kernel<<<ew_blocks(B * ad), 256, 0, si>>>(w.g_cat[2], L + SA, L + sh.a_off[i], ad, B, w.a_head[0][a.n_val - 1].g);
            B2RL_LAUNCH_CHECK();
            if ((rc = chain_backward(ah, bf.actor[i], w.a_enc[0][a.n_enc - 1].a, B, w.a_head[0], w.a_enc[0][a.n_enc - 1].g,
                                     bf.actor_grads[i], w.lnpart, ws.lnpart_floats, si)) != B2RL_OK)
                return rc;
            if ((rc = chain_backward(ae, bf.actor[i], w.obs_i, B, w.a_enc[0], w.g_obs, bf.actor_grads[i], w.lnpart, ws.lnpart_floats,
                                     si)) != B2RL_OK)
                return rc;
            if ((rc = ma_adam(bf.actor[i], bf.actor_grads[i], bf.actor_m[i], bf.actor_v[i], bf.actor_target[i], a.n_params,
                              cfg.lr_actor, cfg.bc1_actor, cfg.bc2_actor, cfg, actor_state, si)) != B2RL_OK)
                return rc;
        }
        if (fan2) B2RL_CUDA(cudaStreamWaitEvent(si, ms->join2[i], 0));
        if (fan) B2RL_CUDA(cudaEventRecord(ms->join[i], si));
    }
    if (fan)
        for (int i = 0; i < n; ++i) B2RL_CUDA(cudaStreamWaitEvent(s, ms->join[i], 0));
    return B2RL_OK;
}

int b2rl_gaussian_mutate(float *weights, int64_t n_rows, int64_t n_cols, const int64_t *rows, const int64_t *cols,
                         const float *branch_uniforms, const uint8_t *keep, const float *normals, uint64_t seed, uint64_t offset,
                         double mutation_sd, int64_t n, void *stream) {
    B2RL_CHECK_ARG(weights && rows && cols && branch_uniforms && n_rows >= 1 && n_cols >= 1 && n >= 0, "bad arguments");
    if (n == 0) return B2RL_OK;
    gaussian_mutate_kernel<<<ew_blocks(n), 256, 0, as_stream(stream)>>>(weights, n_cols, rows, cols, branch_uniforms, keep, normals,
                                                                        seed, offset, (float)mutation_sd, n);
    B2RL_LAUNCH_CHECK();
    return B2RL_OK;
}

}  // extern "C"
