/* b2rl.h — C ABI of libb2rl.so: the B200 (sm_100a) hot path behind AgileRL's off-policy learn().
 *
 * The reference (AgileRL 2.6.1) is pure Python and has NO FFI / plugin interface: its boundary
 * for this path is the Python class surface (SURVEY.md §8b).  This header is therefore the new
 * seam a maintainer would bind from those classes (ctypes stub in INTEGRATION.md).  Every entry
 * point cites the reference routine it replaces.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes; no torch / C++ types.  All pointers are DEVICE
 *     pointers unless the name ends in _host.  `stream` is a cudaStream_t passed as void*.
 *   - every function returns 0 on success, a negative B2RL_E* code on failure;
 *     b2rl_last_error() returns a thread-local message.  Nothing here synchronises the stream
 *     unless documented; nothing allocates device memory (the caller owns every buffer).
 *   - integer / index / priority-tree work is bit-exact w.r.t. the reference's Python-double
 *     arithmetic (IEEE fp64, no FMA contraction); fp32 network math follows torch op order where
 *     it matters (projection, noise composition, Polyak) and is within 1e-5 elsewhere.
 */
#ifndef B2RL_H_
#define B2RL_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2RL_OK 0
#define B2RL_EINVAL (-1)   /* bad argument (maps to AssertionError / ValueError in the wrappers) */
#define B2RL_ECUDA (-2)    /* CUDA runtime error (RuntimeError) */
#define B2RL_EUNSUPPORTED (-3) /* architecture/activation outside what the kernels implement */

int b2rl_version(void);
const char *b2rl_last_error(void);
/* Number of CUDA kernels this library has launched in this process (bench.py: gpu_launches). */
unsigned long long b2rl_launch_count(void);
/* How many convolution launches took each forward path so far (tests assert the intended kernel ran, not a fallback):
 * path 0 = gather tf32 kernel (conv_tc.cuh), 1 = int8 digit planes over uint8 frames (conv_i8.cuh),
 * 2 = TMA-staged receptive fields (conv_st.cuh); anything else returns 0. */
unsigned long long b2rl_conv_path_count(int path);
/* Which convolution passes take the TMA-staged kernels (conv_st / conv_wst / conv_dst): bit 0 forward, bit 1 weight
 * gradient, bit 2 input gradient.  mask >= 0 sets it, mask < 0 only queries; returns the previous mask.  The default comes
 * from the environment variable B2RL_ST (letters f, w, d; "d" when unset). */
int b2rl_conv_staged_paths(int mask);
/* Device properties the host side sizes grids with (SM count, etc.). */
int b2rl_device_sm_count(int device, int *out_host);

/* Per-step scalars of a CUDA-graph-replayed gradient step: everything the host changes from one step to the next
 * (the driver-annealed beta, len(memory), Philox offsets, Adam's bias corrections / lr).  A captured step reads them
 * from a DEVICE copy of this struct; b2rl_graph_launch rewrites that copy through the graph's first node, so the
 * host's double arithmetic (CPython's `1 - beta**step`, `lr / bias_correction1`) stays the source of the values. */
typedef struct b2rl_step_state {
    double beta;                        /* PER importance exponent (train_off_policy.py:346-351 anneals it) */
    int64_t size;                       /* len(memory) */
    uint64_t sample_offset;             /* Philox offset of the B sampling uniforms */
    uint64_t noise_offset[2];           /* Philox offsets of the actor / target noise reset */
    double lr, bias_correction1, bias_correction2;   /* torch.optim.Adam scalars of this step */
} b2rl_step_state;

/* ------------------------------------------------------------------------------------------
 * Priority trees — agilerl/components/segment_tree.py (SumSegmentTree / MinSegmentTree).
 * Layout: array heap of 2*cap fp64 per tree, node i has children 2i, 2i+1, leaf j at cap+j,
 * root at 1 (tree[0] unused, holds the init value like the reference list).
 * ------------------------------------------------------------------------------------------ */

/* SegmentTree.__init__ (segment_tree.py:19-26): sum tree <- 0.0, min tree <- +inf. */
int b2rl_tree_init(double *sum_tree, double *min_tree, int64_t cap, void *stream);

/* n x SegmentTree.__setitem__ (segment_tree.py:81-95) on BOTH trees, sequential semantics:
 * duplicate indices resolve to the LAST writer; every touched ancestor is recomputed bottom-up
 * as op(tree[2i], tree[2i+1]).  leaf values are the already-exponentiated p**alpha
 * (PrioritizedReplayBuffer._update_priority, replay_buffer.py:311-329).  idx in [0, cap).
 * Either tree pointer may be NULL to update only the other one (SegmentTree.__setitem__). */
int b2rl_tree_set(double *sum_tree, double *min_tree, int64_t cap, const int64_t *idx,
                  const double *p_alpha, int64_t n, void *stream);

/* PrioritizedReplayBuffer.add's priority loop (replay_buffer.py:306-309): n consecutive slots
 * starting at tree_ptr, wrapping modulo max_size (not cap — quirk Q7), all set to p_alpha. */
int b2rl_tree_set_range(double *sum_tree, double *min_tree, int64_t cap, int64_t tree_ptr,
                        int64_t n, int64_t max_size, double p_alpha, void *stream);
/* Same (replay_buffer.py:306-309), for a loop that keeps its running maximum on the device (b2rl_tree_set_from_priorities folds into
 * *max_priority_dev): leaf = pow(max(host_max, *max_priority_dev), alpha) computed on device — no host read of the
 * device scalar between an update and the next add (device pow: <= 1 ulp from glibc, like the update it follows). */
int b2rl_tree_set_range_devmax(double *sum_tree, double *min_tree, int64_t cap, int64_t tree_ptr, int64_t n,
                               int64_t max_size, double host_max, const double *max_priority_dev, double alpha,
                               void *stream);

/* PrioritizedReplayBuffer.update_priorities (replay_buffer.py:411-428) as a device-only call, used by the fused path:
 * leaf = pow(max(priority, floor), alpha) computed ON
 * DEVICE (<= 1 ulp from glibc pow: leaves are NOT guaranteed bit-identical to the reference;
 * the tree arithmetic above them is).  Also folds max(priority) into *max_priority (fp64). */
int b2rl_tree_set_from_priorities(double *sum_tree, double *min_tree, int64_t cap,
                                  const int64_t *idx, const float *priority, int64_t n,
                                  double alpha, double floor_, double *max_priority, void *stream);

/* SumSegmentTree.retrieve (segment_tree.py:136-156) for n upper bounds. */
int b2rl_tree_retrieve(const double *sum_tree, int64_t cap, const double *upperbound, int64_t n,
                       int64_t *out_idx, void *stream);

/* PrioritizedReplayBuffer._sample_proportional + _calculate_weights
 * (replay_buffer.py:357-409): stratified proportional sample from B float32 uniforms and the
 * importance weights ((p_i*size)^-beta / (p_min*size)^-beta), fp64 then cast to f32.
 * out_idx int64[B], out_w float[B]. */
int b2rl_per_sample(const double *sum_tree, const double *min_tree, int64_t cap,
                    const float *uniforms, int64_t B, double beta, int64_t size, int64_t *out_idx,
                    float *out_w, void *stream);
/* Same (replay_buffer.py:357-409), drawing the uniforms on device from Philox(seed, offset) instead of the B
 * torch.rand(1) draws of replay_buffer.py:377 (production path). */
int b2rl_per_sample_philox(const double *sum_tree, const double *min_tree, int64_t cap,
                           uint64_t seed, uint64_t offset, int64_t B, double beta, int64_t size,
                           int64_t *out_idx, float *out_w, void *stream);

/* The fused sample step of the HBM-resident path (north star K1): one kernel does the sum-tree
 * descent, the importance weights AND the gather of the sampled slots' n-step action / reward /
 * done from the (ingest-rolled, replay_buffer.py:206-258) n-step ring.  Frames are not copied:
 * the encoder's first-layer loader reads them from the ring through out_idx.  uniforms == NULL
 * draws them from Philox(seed, offset).  *_ring are float32 [max_size] (the [max_size,1]
 * storage columns). */
int b2rl_per_sample_fused(const double *sum_tree, const double *min_tree, int64_t cap,
                          const float *uniforms, uint64_t seed, uint64_t offset, int64_t B,
                          double beta, int64_t size, const float *action_ring,
                          const float *reward_ring, const float *done_ring, int64_t *out_idx,
                          float *out_w, float *out_action, float *out_reward, float *out_done,
                          void *stream);
/* Same (replay_buffer.py:331-355 + :196-204), with beta / size / the Philox offset read on device from *state
 * (graph-replayed steps; Philox only). */
int b2rl_per_sample_fused_state(const double *sum_tree, const double *min_tree, int64_t cap, uint64_t seed,
                                const b2rl_step_state *state, int64_t B, const float *action_ring,
                                const float *reward_ring, const float *done_ring, int64_t *out_idx, float *out_w,
                                float *out_action, float *out_reward, float *out_done, void *stream);

/* No reference counterpart (the reference draws from torch's CPU generator: replay_buffer.py:377,
 * custom_components.py:118-119).  Read-back of the device random streams (parity tests hand them to the oracle): the B float32 uniforms
 * b2rl_per_sample_philox / b2rl_per_sample_fused(uniforms = NULL) consume at (seed, offset), and the
 * standard normals b2rl_noise_reset_philox consumes at (seed, offset) in b2rl_noise_reset_from_normals' layout. */
int b2rl_philox_uniforms(uint64_t seed, uint64_t offset, int64_t n, float *out, void *stream);
int b2rl_philox_normals(uint64_t seed, uint64_t offset, int64_t n, float *out, void *stream);

/* ------------------------------------------------------------------------------------------
 * Ring storage — ReplayBuffer.add / storage[indices] (replay_buffer.py:72-112, :126, :204, :345).
 * One call per field (SoA); rows are opaque byte strings of row_bytes.
 * ------------------------------------------------------------------------------------------ */

/* storage[start:start+n] (with wrap split at max_size) <- src[0:n]. */
int b2rl_ring_write(void *storage, const void *src, int64_t row_bytes, int64_t start, int64_t n,
                    int64_t max_size, void *stream);
/* dst[i] <- storage[idx[i]], i < n (idx int64 on device, values in [0, max_size)). */
int b2rl_gather_rows(void *dst, const void *storage, const int64_t *idx, int64_t row_bytes,
                     int64_t n, void *stream);
/* The same for up to 8 fields of a transition in one launch (host arrays of n_fields device pointers /
 * row sizes): what ReplayBuffer.add and storage[indices] do over every key of the TensorDict. */
int b2rl_ring_write_multi(int n_fields, void *const *storage, const void *const *src, const int64_t *row_bytes,
                          int64_t start, int64_t n, int64_t max_size, void *stream);
int b2rl_gather_rows_multi(int n_fields, void *const *dst, const void *const *storage, const int64_t *row_bytes,
                           const int64_t *idx, int64_t n, void *stream);

/* ReplayBuffer.sample's index draw on device (replay_buffer.py:114-131, quirk Q12: uniform WITHOUT replacement):
 * B distinct indices uniform over [0, N) from Philox(seed, offset), B <= 1024, deterministic.  The API path keeps
 * torch.randperm on the host (same RNG stream as the reference); this serves the HBM-resident loop. */
int b2rl_sample_uniform_distinct(uint64_t seed, uint64_t offset, int64_t N, int64_t B, int64_t *out_idx, void *stream);

/* HOST helper (no device work): PrioritizedReplayBuffer.update_priorities' per-priority arithmetic
 * (replay_buffer.py:411-428, :311-329) — q = max((double)p, floor); out[i] = pow(q, alpha) with the C library's pow,
 * which is what CPython's `priority ** alpha` evaluates, so the leaves are bit-identical to the reference's; *max_host
 * (in/out, nullable) accumulates max(q) (max_priority, :329). */
int b2rl_host_priority_pow(const float *priority_host, int64_t n, double alpha, double floor_, double *out_host,
                           double *max_host);

/* HOST helper (no device work): ReplayBuffer.sample's index draw (replay_buffer.py:126: `torch.randperm(self.size)[:batch_size]`)
 * without materialising the permutation.  rng_state_host = the bytes of torch.get_rng_state() (CPU generator, mt19937),
 * updated in place to the state torch.randperm(n) leaves; out_host[0:B] = torch.randperm(n)[:B] (n < UINT32_MAX / 20:
 * torch's 32-bit Fisher-Yates shuffle, of which entry i is final after iteration i).  Same indices and same generator
 * stream as the reference; the wrapper verifies that against torch.randperm once per process. */
int b2rl_host_randperm_prefix(uint8_t *rng_state_host, int64_t state_bytes, int64_t n, int64_t B, int64_t *out_host);

/* MultiStepReplayBuffer._get_n_step_info (replay_buffer.py:206-258) over a device window of n
 * per-env batches (oldest first): reward_out[e] = sum_i gamma^i r_i[e] (fp32 accumulate, gamma^i a
 * double rounded to f32 like torch scalar mul), stop after the first step i>=1 where ANY env is
 * done; last_step_out (int32, 1 element) = index of the step whose next_obs/done are carried. */
int b2rl_nstep_fold(const float *const *reward_steps, const float *const *done_steps, int n_step,
                    int64_t num_envs, double gamma, float *reward_out, int32_t *last_step_out,
                    void *stream);

/* MultiStepReplayBuffer.add in ONE launch (replay_buffer.py:173-194 -> :206-258 -> :72-112): fold the window of n_step
 * per-env batches and write the resulting n-step transition straight into the ring rows [cursor, cursor+num_envs) (mod
 * max_size).  Field i: ring[i] (storage base), src[i*n_step + k] (step k's [num_envs, ...] batch of that field),
 * row_bytes[i], role[i] = 0 take step 0 (obs, action ...), 1 take the step the fold stopped at (next_obs, done),
 * 2 the folded float32 reward.  reward_steps / done_steps: float32 [num_envs] per step.  All arrays HOST arrays of
 * device pointers. */
int b2rl_nstep_ingest(int n_fields, void *const *ring, const void *const *src, const int64_t *row_bytes, const int32_t *role,
                      const float *const *reward_steps, const float *const *done_steps, int n_step, int64_t num_envs,
                      double gamma, int64_t cursor, int64_t max_size, void *stream);

/* dst[0:bytes] <- srcs[*which][0:bytes]: carries next_obs/done of the step the fold stopped
 * at (replay_buffer.py:249-250) without a host round trip.  srcs_host: HOST array of n_srcs
 * device pointers; which: DEVICE int32. */
int b2rl_select_copy(void *dst, const void *const *srcs_host, int n_srcs, const int32_t *which,
                     int64_t bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * Networks — RainbowQNetwork / QNetwork forward+backward, RainbowDQN/DQN learn tail.
 * A network is a flat fp32 parameter buffer plus a layer table.
 * ------------------------------------------------------------------------------------------ */
enum { B2RL_ACT_NONE = 0, B2RL_ACT_RELU = 1, B2RL_ACT_ELU = 2, B2RL_ACT_GELU = 3, B2RL_ACT_TANH = 4 };
enum { B2RL_LAYER_CONV = 0, B2RL_LAYER_LINEAR = 1 };
enum { B2RL_LN_NONE = 0, B2RL_LN_AFFINE = 1, B2RL_LN_PLAIN = 2 };
enum { B2RL_NET_Q = 0, B2RL_NET_RAINBOW = 1 };

typedef struct b2rl_layer {
    int32_t kind;                       /* B2RL_LAYER_* */
    int32_t in_c, in_h, in_w;           /* conv input  (linear: in_c = in_features, h=w=1) */
    int32_t out_c, out_h, out_w;        /* conv output (linear: out_c = out_features) */
    int32_t ksize, stride;
    int32_t act;                        /* activation applied after (LN if any) */
    int32_t ln;                         /* B2RL_LN_* applied between linear and activation */
    int32_t noisy;                      /* NoisyLinear: W = mu + sigma*eps */
    int64_t w_off, b_off;               /* offsets (floats) into the parameter buffer (mu) */
    int64_t ws_off, bs_off;             /* sigma offsets (noisy only) */
    int64_t we_off, be_off;             /* epsilon offsets into the eps buffer (noisy only) */
    int64_t lnw_off, lnb_off;           /* LayerNorm affine (B2RL_LN_AFFINE only) */
} b2rl_layer;

#define B2RL_MAX_ENC 12
#define B2RL_MAX_HEAD 6

typedef struct b2rl_net_desc {
    int32_t kind;                       /* B2RL_NET_* */
    int32_t n_enc, n_val, n_adv;        /* layer counts (n_adv = 0 for B2RL_NET_Q) */
    b2rl_layer enc[B2RL_MAX_ENC];       /* encoder: convs then linears (flatten is implicit) */
    b2rl_layer val[B2RL_MAX_HEAD];      /* value head / plain Q head */
    b2rl_layer adv[B2RL_MAX_HEAD];      /* advantage head (rainbow) */
    int32_t n_actions, n_atoms;
    int32_t obs_u8;                     /* observations are uint8 (else float32) */
    int32_t normalize;                  /* (x-low)/(high-low), algo_utils.py:1131-1180 */
    float obs_low, obs_high;
    int64_t obs_elems;                  /* elements per observation row */
    int64_t n_params, n_eps;            /* sizes of the flat parameter / epsilon buffers */
} b2rl_net_desc;

/* Bytes of scratch a forward/learn call needs for `rows` observation rows. */
int b2rl_net_workspace_bytes(const b2rl_net_desc *net_host, int64_t rows, int with_backward,
                             size_t *out_host);

/* NoisyLinear.reset_noise for every noisy layer in traversal order
 * (custom_components.py:116-131): eps_W = f(e_out) (x) f(e_in), eps_b = f(e_out),
 * f(x) = sign(x) sqrt|x|.  `normals` holds, per noisy layer, randn(in) then randn(out). */
int b2rl_noise_reset_from_normals(const b2rl_net_desc *net_host, float *eps, const float *normals,
                                  void *stream);
/* Same with normals drawn on device: Philox4x32-10(seed, subsequence = layer, offset). */
int b2rl_noise_reset_philox(const b2rl_net_desc *net_host, float *eps, uint64_t seed,
                            uint64_t offset, void *stream);
/* Same, offset = state->noise_offset[which] read on device (which: 0 actor, 1 target). */
int b2rl_noise_reset_state(const b2rl_net_desc *net_host, float *eps, uint64_t seed, const b2rl_step_state *state,
                           int which, void *stream);
/* The two resets of a learn step (actor: noise_offset[0], target: noise_offset[1]; dqn_rainbow.py:484-485) in ONE launch —
 * same values as two b2rl_noise_reset_state calls with which = 0 and 1. */
int b2rl_noise_reset_state_pair(const b2rl_net_desc *net_host, float *eps_actor, float *eps_target, uint64_t seed,
                                const b2rl_step_state *state, void *stream);
/* Number of standard normals one reset consumes. */
int b2rl_noise_count(const b2rl_net_desc *net_host, int64_t *out_host);

/* Forward only (get_action path: dqn_rainbow.py:239-282, dqn.py:262-264).
 * obs: rows x obs_elems (uint8 or f32); row_idx (nullable) gathers rows from a ring.
 * q_out: rows x n_actions expected values; argmax_out (nullable): int64 rows.
 * use_noise: train-mode NoisyLinear (Rainbow acts in train mode).  support: n_atoms C51 atoms
 * (rainbow; NULL for Q nets). */
int b2rl_net_forward_q(const b2rl_net_desc *net_host, const float *params, const float *eps,
                       int use_noise, const float *support, const void *obs,
                       const int64_t *row_idx, int64_t rows, float *q_out, int64_t *argmax_out,
                       void *workspace, size_t workspace_bytes, void *stream);

/* RainbowQNetwork.forward(obs, q=False, log=log_probs) (q_networks.py:265-284 -> custom_modules.py:127-162):
 * per-atom distributions, dist_out: rows x n_actions x n_atoms — softmax then clamp(min=1e-3), or log_softmax
 * (unclamped) when log_probs != 0. */
int b2rl_net_forward_dist(const b2rl_net_desc *net_host, const float *params, const float *eps, int use_noise,
                          const void *obs, const int64_t *row_idx, int64_t rows, int log_probs, float *dist_out,
                          void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * PPO return / advantage recurrence — RolloutBuffer.compute_returns_and_advantages
 * (agilerl/components/rollout_buffer.py:413-481).  rewards / values float32 [T, E], dones bool (1 byte) [T, E],
 * last_value float64 [E] (the reference widens it: last_value.astype(float)), last_done float32 [E]; advantages / returns float32 [T, E] out.  use_gae = 0: Monte-Carlo returns.
 * Bit-identical to the reference's NumPy loop (float64 carry, float32 stores).
 * ------------------------------------------------------------------------------------------ */
int b2rl_gae_scan(const float *rewards, const uint8_t *dones, const float *values, const double *last_value,
                  const float *last_done, int64_t T, int64_t E, double gamma, double gae_lambda, int use_gae,
                  float *advantages, float *returns, void *stream);
/* PPO's global advantage normalisation (agilerl/algorithms/ppo.py:831-834, :935-944): out = (a - mean(a)) /
 * (std(a) + 1e-8), unbiased std; reductions in float64, fixed order (deterministic; within 1e-6 of torch's float32
 * statistics).  n = T*E elements, one launch. */
int b2rl_advantage_normalize(const float *advantages, int64_t n, float *out, void *stream);
/* Both in ONE launch when E <= 1024 (one CTA: thread e scans environment e, then the CTA normalises): returns,
 * raw advantages and normalised advantages of a rollout without leaving the device. */
int b2rl_gae_scan_normalize(const float *rewards, const uint8_t *dones, const float *values, const double *last_value,
                            const float *last_done, int64_t T, int64_t E, double gamma, double gae_lambda, int use_gae,
                            float *advantages, float *returns, float *adv_norm, void *stream);

/* Diagnostics: with B2RL_TC_DBG=<cta> in the environment the tensor-core forward convolution records
 * clock64() stamps of that CTA's producer warp 0 (slots 0..63) and MMA lane (slots 64..127); this copies the
 * first n (<= 128) to the host after a device synchronize.  Fails when diagnostics are off. */
int b2rl_debug_read(long long *out_host, int n);

/* Forward of ONE encoder layer (profiling / roofline hook: lets bench.py time the dominant
 * contraction alone with CUDA events).  layer 0 reads observations (obs/row_idx as above), layer
 * i>0 reads `input` = the previous layer's [rows, ...] fp32 activations.  out: rows x out elems.
 * reuse_split != 0: the workspace still holds this layer's pre-split weights (digit planes / tf32 hi-lo tiles) from the
 * previous call with the same parameters — only the convolution kernel itself is launched. */
int b2rl_encoder_layer_forward(const b2rl_net_desc *net_host, int layer, const float *params,
                               const void *input, const int64_t *row_idx, int64_t rows, float *out,
                               void *workspace, size_t workspace_bytes, int reuse_split, void *stream);

/* Test / profiling hook: weight and bias gradient of encoder layer `layer` alone.  g_out [rows, out...] is the gradient at the
 * layer's pre-activation output; input as in b2rl_encoder_layer_forward; the gradients are written (not accumulated) at the
 * layer's w_off / b_off of the flat buffer `grads` [n_params]. */
int b2rl_encoder_layer_wgrad(const b2rl_net_desc *net_host, int layer, const void *input, const int64_t *row_idx,
                             int64_t rows, const float *g_out, float *grads, void *workspace, size_t workspace_bytes,
                             void *stream);

/* Test / profiling hook: input gradient of convolutional encoder layer `layer` >= 1 alone: g_in [rows, in_c, in_h, in_w]
 * (overwritten) from g_out, the gradient at the layer's pre-activation output. */
int b2rl_encoder_layer_dgrad(const b2rl_net_desc *net_host, int layer, const float *params, const float *g_out, int64_t rows,
                             float *g_in, void *workspace, size_t workspace_bytes, void *stream);

/* Scalars of one learn step (doubles are the Python floats of the reference, rounded to f32
 * inside the kernels exactly where torch rounds them). */
typedef struct b2rl_learn_cfg {
    int64_t batch;                      /* B (== agent.batch_size, quirk Q17) */
    double gamma;                       /* discount used in the target (gamma**n_step for n-step) */
    double v_min, v_max;                /* C51 support bounds (rainbow) */
    double delta_z;                     /* (v_max - v_min)/(n_atoms-1) */
    int32_t weights_mode;               /* 0: no PER (mean l); 1: weights [B] -> mean(l*w);
                                           2: weights [B,1] -> mean(l)*mean(w)  (quirk Q1) */
    int32_t driver_shapes;              /* 1: reward/done arrived [B,1,1] (quirk Q2 semantics) */
    int32_t double_dqn;                 /* DQN only */
    int32_t clip;                       /* 1: clip_grad_norm_(max_grad_norm) (rainbow), 0: none */
    double max_grad_norm;
    double lr, beta1, beta2, adam_eps;
    double bias_correction1, bias_correction2; /* 1-beta^step */
    double tau;
    double prior_eps;
    int32_t accumulate;                 /* 1: second pass of combined_reward — add this pass's
                                           per-sample loss / gradients to the first pass's */
    int32_t use_noise;                  /* NoisyLinear in train mode (always 1 in learn) */
    int32_t side_streams;               /* 1: b2rl_rainbow_loss may run the target forward, and
                                           b2rl_rainbow_backward the weight gradients, on library-owned
                                           side streams (joined before the call's work is complete in the
                                           caller's stream order); 0: everything on `stream` */
    int32_t reserved_;                  /* bit 0: b2rl_rainbow_prep was enqueued for this pass (rainbow loss only) */
} b2rl_learn_cfg;

/* Device buffers of one learn step (all fp32 unless stated). */
typedef struct b2rl_learn_bufs {
    float *actor_params, *target_params;     /* n_params each */
    float *actor_eps, *target_eps;           /* n_eps each */
    float *grads, *exp_avg, *exp_avg_sq;     /* n_params each */
    const void *obs, *next_obs;              /* batch rows, or ring bases when row_idx != NULL */
    const int64_t *row_idx;                  /* nullable: B ring rows */
    const float *action, *reward, *done;     /* B each */
    const float *weights;                    /* B (PER) or NULL */
    const float *support;                    /* n_atoms (rainbow) */
    float *loss_elem;                        /* out: B per-sample loss */
    float *priorities;                       /* out: B, loss_elem + prior_eps (nullable) */
    float *loss_scalar;                      /* out: 1, the scalar loss that was back-propagated */
    float *proj_dist;                        /* out (nullable): B x n_atoms projected target */
    void *workspace; size_t workspace_bytes;
    const b2rl_step_state *step_state;       /* nullable DEVICE pointer: when set, b2rl_optim_step takes lr and the bias
                                                corrections from it instead of cfg (graph-replayed steps) */
} b2rl_learn_bufs;

/* RainbowDQN._dqn_loss (dqn_rainbow.py:284-367): three forwards, C51 projection, cross-entropy;
 * writes per-sample loss, leaves dL/dlogits staged in the workspace.  Does not touch grads. */
int b2rl_rainbow_loss(const b2rl_net_desc *net_host, const b2rl_learn_cfg *cfg_host,
                      const b2rl_learn_bufs *bufs_host, void *stream);
/* Optional: enqueue everything of the next b2rl_rainbow_loss that depends on the parameters only (noisy-layer weight
 * composition, the first layer's int8 digit planes for both networks, the tf32 split of the later convolutions) on a
 * library-owned side stream forked from `stream`, so that it overlaps whatever the caller enqueues next on `stream`
 * (the sampler).  The following b2rl_rainbow_loss on the same stream must then be called with cfg.reserved_ = 1: it joins
 * the side stream and skips those launches.  Same workspace, same buffers as the loss call. */
int b2rl_rainbow_prep(const b2rl_net_desc *net_host, const b2rl_learn_cfg *cfg_host, const b2rl_learn_bufs *bufs_host,
                      void *stream);
/* Back-propagate mean(loss*w) of the staged loss(es) into `grads` (loss.backward()).
 * n_passes = 1, or 2 when combined_reward staged two losses. */
int b2rl_rainbow_backward(const b2rl_net_desc *net_host, const b2rl_learn_cfg *cfg_host,
                          const b2rl_learn_bufs *bufs_host, void *stream);
/* Tail of learn (dqn_rainbow.py:473-488): clip_grad_norm_, Adam, soft_update. */
int b2rl_optim_step(const b2rl_net_desc *net_host, const b2rl_learn_cfg *cfg_host,
                    const b2rl_learn_bufs *bufs_host, void *stream);
/* DQN.update + learn (dqn.py:274-347): (double) Q target, MSE, backward, Adam, soft update. */
int b2rl_dqn_learn(const b2rl_net_desc *net_host, const b2rl_learn_cfg *cfg_host,
                   const b2rl_learn_bufs *bufs_host, void *stream);
/* Whole Rainbow learn step for the common case (one loss pass): loss + backward + optim. */
int b2rl_rainbow_learn(const b2rl_net_desc *net_host, const b2rl_learn_cfg *cfg_host,
                       const b2rl_learn_bufs *bufs_host, void *stream);

/* ------------------------------------------------------------------------------------------
 * DDPG / TD3 learn() — agilerl/algorithms/ddpg.py:422-500, td3.py:459-551 (SURVEY 8f-1, BASELINE configs[2]).
 * Networks are b2rl_net_desc chains: actor = enc[] (MLP encoder) -> val[] (head, Tanh output, n_actions = action dim);
 * critic = enc[] -> cat(latent, action) -> val[] (val[0].in_c = latent + action dim, output 1)
 * (networks/actors.py:78-210, networks/q_networks.py:302-443).  One flat parameter buffer per network.
 * ------------------------------------------------------------------------------------------ */
typedef struct b2rl_ddpg_cfg {
    int64_t batch;
    int32_t twin;                       /* 1: TD3 (two critics, min target, summed MSE), 0: DDPG */
    int32_t policy_update;              /* this call also steps the actor and soft-updates every target
                                           (learn_counter % policy_freq == 0, td3.py:520) */
    double gamma, tau, noise_clip, policy_noise;
    double lr_actor, lr_critic, beta1, beta2, adam_eps;
    double bc1_actor, bc2_actor, bc1_critic, bc2_critic;   /* 1 - beta^step of each optimiser */
    uint64_t noise_seed, noise_offset;  /* Philox stream of the target-policy noise when bufs.noise == NULL */
} b2rl_ddpg_cfg;

typedef struct b2rl_ddpg_bufs {
    float *actor, *actor_target, *actor_grads, *actor_m, *actor_v;
    float *critic[2], *critic_target[2], *critic_grads[2], *critic_m[2], *critic_v[2];
    const float *obs, *next_obs;        /* [B, obs_dim] float32 */
    float *action;                      /* [B, act_dim] IN/OUT: overwritten with the raw target-policy noise
                                           (actions.data.normal_(0, policy_noise), td3.py:497 — the reference's quirk) */
    const float *reward, *done;         /* [B] */
    const float *noise;                 /* nullable [B, act_dim]: injected N(0, policy_noise) draws (parity tests) */
    const float *action_low, *action_high;   /* [act_dim] */
    float *critic_loss, *actor_loss;    /* out: scalars (actor_loss written on policy steps only) */
    void *workspace; size_t workspace_bytes;
} b2rl_ddpg_bufs;

int b2rl_ddpg_workspace_bytes(const b2rl_net_desc *actor_host, const b2rl_net_desc *critic_host, int64_t batch,
                              size_t *out_host);
int b2rl_ddpg_learn(const b2rl_net_desc *actor_host, const b2rl_net_desc *critic_host, const b2rl_ddpg_cfg *cfg_host,
                    const b2rl_ddpg_bufs *bufs_host, void *stream);
/* DeterministicActor.forward (actors.py:188-210): out [rows, act_dim]. */
int b2rl_actor_workspace_bytes(const b2rl_net_desc *actor_host, int64_t rows, size_t *out_host);
int b2rl_actor_forward(const b2rl_net_desc *actor_host, const float *params, const float *obs, int64_t rows, float *out,
                       void *workspace, size_t workspace_bytes, void *stream);

/* ------------------------------------------------------------------------------------------
 * MADDPG learn() — agilerl/algorithms/maddpg.py:571-740 (SURVEY 8f-4, BASELINE configs[4]: 4 agents x 18-dim
 * observations, shared replay) for vector observations and continuous actions.
 * actor_i = b2rl_net_desc chain enc[] (LayerNorm MLP encoder over agent i's observation) -> val[] (head, Tanh);
 * critic_i = enc[] over the concatenation of EVERY agent's observation (EvolvableMultiInput's final_dense + ReLU,
 * modules/multi_input.py:404-465) -> cat(latent, EVERY agent's action) -> val[] (-> 1).
 * The batch arrives as row-major matrices with the agents' columns side by side in agent order — what the
 * reference's torch.cat(..., dim=1) builds — so the replay gather can write them directly.
 * ------------------------------------------------------------------------------------------ */
#define B2RL_MAX_AGENTS 8
typedef struct b2rl_maddpg_cfg {
    int64_t batch;
    int32_t n_agents;
    int32_t serial;                     /* 1: the agents' steps one after another on the caller's stream; 0: concurrently
                                           on one library side stream per agent (forked from / joined into `stream`) */
    double gamma, tau;
    double lr_actor, lr_critic, beta1, beta2, adam_eps;
    double bc1_actor, bc2_actor, bc1_critic, bc2_critic;   /* 1 - beta^step of the actor / critic optimisers */
    /* MATD3 (agilerl/algorithms/matd3.py:630-831).  Both zero: the MADDPG call above. */
    int32_t twin;                       /* 1: a second critic set (bufs.critic2*): y = r + (1 - d) gamma min(Q'1, Q'2),
                                           critic_loss = MSE(Q1, y) + MSE(Q2, y), both critics step; the actor step
                                           reads critic_1 only.  No target-policy smoothing noise (unlike TD3). */
    int32_t critic_only;                /* 1: critic TD steps only — no actor forward / backward / Adam and no Polyak
                                           update of any target (a MATD3 call where learn_counter % policy_freq != 0);
                                           losses[i][0] is written NaN */
} b2rl_maddpg_cfg;

typedef struct b2rl_maddpg_bufs {
    float *actor[B2RL_MAX_AGENTS], *actor_target[B2RL_MAX_AGENTS], *actor_grads[B2RL_MAX_AGENTS], *actor_m[B2RL_MAX_AGENTS],
          *actor_v[B2RL_MAX_AGENTS];
    float *critic[B2RL_MAX_AGENTS], *critic_target[B2RL_MAX_AGENTS], *critic_grads[B2RL_MAX_AGENTS], *critic_m[B2RL_MAX_AGENTS],
          *critic_v[B2RL_MAX_AGENTS];
    const float *obs, *next_obs;        /* [B, sum of observation dims] */
    const float *action;                /* [B, sum of action dims] */
    const float *reward, *done;         /* [B, n_agents]; NaN reward -> 0, NaN done -> 1 (maddpg.py:683-694) */
    float *losses;                      /* out [n_agents, 2]: actor_loss, critic_loss of each agent */
    void *workspace; size_t workspace_bytes;
    const b2rl_step_state *step_state;  /* nullable (device): a captured call reads this step's Adam bias corrections
                                           (bias_correction1 / 2; every optimiser steps once per call) from here */
    /* twin only: critic_2 of every agent, its target, gradients and Adam moments (critic_1's architecture) */
    float *critic2[B2RL_MAX_AGENTS], *critic2_target[B2RL_MAX_AGENTS], *critic2_grads[B2RL_MAX_AGENTS],
          *critic2_m[B2RL_MAX_AGENTS], *critic2_v[B2RL_MAX_AGENTS];
    const b2rl_step_state *actor_step_state;   /* nullable (device): the ACTOR optimisers' bias corrections of a captured
                                                  call whose actors and critics have stepped different numbers of times
                                                  (MATD3); NULL: the actors read step_state too */
} b2rl_maddpg_bufs;

int b2rl_maddpg_workspace_bytes(const b2rl_net_desc *const *actors_host, const b2rl_net_desc *const *critics_host, int n_agents,
                                int64_t batch, size_t *out_host);
/* The same for the call cfg_host describes (batch, n_agents, twin): a twin call needs room for the critic_2 passes. */
int b2rl_maddpg_workspace_bytes_cfg(const b2rl_net_desc *const *actors_host, const b2rl_net_desc *const *critics_host,
                                    const b2rl_maddpg_cfg *cfg_host, size_t *out_host);
/* One learn call of every agent, then every soft update (fused into the optimiser launches: no target is read after its
 * network stepped).  actors_host / critics_host: n_agents pointers to the (host) layer tables (critic_2 of a twin call
 * shares critic_1's table).  Side streams (serial == 0): one per agent, plus one per agent for critic_2's chains. */
int b2rl_maddpg_learn(const b2rl_net_desc *const *actors_host, const b2rl_net_desc *const *critics_host,
                      const b2rl_maddpg_cfg *cfg_host, const b2rl_maddpg_bufs *bufs_host, void *stream);

/* Mutations._gaussian_parameter_mutation (hpo/mutation.py:733-827) applied on the device to one weight matrix
 * [n_rows, n_cols] (row-major, leading dimension n_cols) of a flat parameter buffer: slot j rewrites
 * W[rows[j]][cols[j]] — branch_uniforms[j] < 0.05: w + |10 w| z; < 0.1: z; else w + |mutation_sd w| z; clamp(+-1e6).
 * rows / cols / branch_uniforms are the reference's host-drawn numpy values (device copies); keep (nullable, uint8)
 * marks the last writer of each position (index_put_ semantics); normals (nullable) injects z, else the Philox
 * stream (seed, offset + j). */
int b2rl_gaussian_mutate(float *weights, int64_t n_rows, int64_t n_cols, const int64_t *rows, const int64_t *cols,
                         const float *branch_uniforms, const uint8_t *keep, const float *normals, uint64_t seed, uint64_t offset,
                         double mutation_sd, int64_t n, void *stream);

/* ------------------------------------------------------------------------------------------
 * CUDA graphs: the ~40 dependent launches of a gradient step captured once and replayed per step.
 * b2rl_graph_begin puts `stream` into capture (relaxed mode; library-owned side streams fork from and join back
 * into it); every b2rl_* call made on it until b2rl_graph_end is recorded instead of executed.  If the captured
 * work starts with b2rl_step_state_write, b2rl_graph_launch patches that node's by-value argument with
 * *state_host before launching, which is how a replay sees this step's scalars.
 * ------------------------------------------------------------------------------------------ */
typedef struct b2rl_graph b2rl_graph;
/* *state_dev <- *state_host (one tiny kernel; the struct travels by value in the launch). */
int b2rl_step_state_write(const b2rl_step_state *state_host, b2rl_step_state *state_dev, void *stream);
/* Asynchronous device -> pinned-host copy on `stream` (capturable: the loss / priority read-back of a replayed step). */
int b2rl_copy_d2h(void *dst_pinned_host, const void *src, size_t bytes, void *stream);
int b2rl_graph_begin(void *stream);
int b2rl_graph_end(void *stream, b2rl_graph **out_host);
/* state_host may be NULL when the graph holds no b2rl_step_state_write node. */
int b2rl_graph_launch(b2rl_graph *g, const b2rl_step_state *state_host, void *stream);
/* For a graph with several b2rl_step_state_write nodes (e.g. a MATD3 policy call: critic and actor bias corrections):
 * the node that writes states_dev[k] gets *states_host[k], k < n; every state_dev given must have a node in the graph,
 * nodes not named keep their last value. */
int b2rl_graph_launch_states(b2rl_graph *g, const b2rl_step_state *const *states_host, b2rl_step_state *const *states_dev, int n,
                             void *stream);
/* kernel nodes in the graph (what one replay adds to b2rl_launch_count) */
int b2rl_graph_kernel_count(const b2rl_graph *g, int *out_host);
int b2rl_graph_destroy(b2rl_graph *g);

#ifdef __cplusplus
}
#endif
#endif /* B2RL_H_ */
