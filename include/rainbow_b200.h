/*
 * rainbow_b200.h -- C ABI of the B200-native Rainbow learner hot path.
 *
 * The reference (Kaixhin/Rainbow @ 1745b184) has no FFI/plugin layer: its hot
 * path is Python (memory.py, agent.py, model.py).  This header is the drop-in
 * boundary a maintainer of the reference would bind with ctypes/cffi from
 * those three files (INTEGRATION.md shows the stubs).  Each entry point names
 * the reference lines it replaces.
 *
 * Conventions
 *   - C linkage, plain pointers and sizes, no torch / C++ types.
 *   - Every pointer is a DEVICE pointer owned by the caller (e.g.
 *     tensor.data_ptr()) unless a parameter is documented "host".
 *   - Every call enqueues work on `stream` (a cudaStream_t passed as void*)
 *     and returns immediately; nothing synchronises, allocates or frees.
 *     All calls are CUDA-graph capturable.
 *   - Return value: RB_OK (0) or a negative errno-style code; the text of the
 *     last error of the calling thread is available from rb_last_error().
 *   - Device-side conditions (rejected sample batch, bad index) are reported
 *     through the `status` words written by the kernel, never by a sync.
 *
 * Data layout in HBM (structure of arrays; reference Transition_dtype is an
 * array of 7069-byte structs, memory.py:7):
 *   tree         float32[tree_start + size]   heap order, root at tree[0],
 *                children 2i+1 / 2i+2, leaves from tree_start = 2^ceil(log2 size)-1
 *                (memory.py:17-18).  For 128-byte-aligned level loads allocate
 *                one pad float in front so that (tree - 1) is 128 B aligned.
 *   frames       uint8[size][7056]            last frame of each transition
 *   timestep     int32[size]                  in-episode step (0 = episode start)
 *   action       int32[size]
 *   reward       float32[size]
 *   nonterminal  uint8[size]
 *   ring_state   int64[5]  {head (next write slot), full (0/1), t_episode, appended_total, launch ticket of
 *                          rb_append_batch (zero between launches)}
 *   running_max  float32[1] largest exponentiated priority seen (memory.py:20,48)
 *   rng_counter  uint64[1]  Philox draw counter, advanced by the kernels themselves
 *                           (so a replayed CUDA graph draws fresh numbers)
 */
#ifndef RAINBOW_B200_H
#define RAINBOW_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RB_ABI_VERSION 2

#define RB_OK 0
#define RB_ERR_INVAL (-22)       /* bad argument (EINVAL) */
#define RB_ERR_RANGE (-34)       /* size outside supported range (ERANGE) */
#define RB_ERR_CUDA (-5)         /* CUDA runtime reported an error (EIO) */

#define RB_FRAME_BYTES 7056      /* 84*84 */
#define RB_MAX_WINDOW 64         /* history + multi_step */
#define RB_MAX_ATOMS 128
#define RB_MAX_NOISY_LAYERS 8
#define RB_MAX_PEERS 8           /* ranks of one NVLink domain handled by rb_peer_clip_adam */
#define RB_APPEND_BATCH 8        /* transitions per rb_append_batch launch */

/* status words written by rb_tree_sample (int32[4]): status[0] = 1 if the batch now in the output buffers passed the
 * whole-batch validity test (memory.py:131), 0 otherwise; status[1] = draws used; status[2] = number of device-RNG
 * batches so far that were still invalid after max_attempts draws (cumulative; the caller zero-initialises it once).
 * A rejected batch has all its importance weights set to 0 (its loss gradient is exactly zero), and status[0] can be
 * handed as the `gate` of rb_clip_adam / rb_tree_update so neither the parameters nor the priorities are touched --
 * the device-side counterpart of the reference's redraw-until-valid loop (memory.py:128-132), without a host sync. */

typedef void* rb_stream_t; /* cudaStream_t */

/* kernel ids for the optional timing hooks (rb_profile_*) */
enum {
  RB_K_TREE_UPDATE = 0, RB_K_TREE_FIND, RB_K_TREE_SAMPLE, RB_K_GATHER, RB_K_ITER_STATES, RB_K_APPEND, RB_K_C51,
  RB_K_NOISY_RESAMPLE, RB_K_NOISY_COMPOSE, RB_K_SQNORM, RB_K_CLIP_ADAM, RB_K_HEAD_FC1, RB_K_HEAD_FC2, RB_K_HEAD_LOGITS,
  RB_K_HEAD_WGRAD2, RB_K_HEAD_DH, RB_K_HEAD_BWD1, RB_K_NOISE_FACTORS, RB_K_C51_DUELING, RB_K_BIAS_GRAD, RB_K_Q_VALUES,
  RB_K_HEAD_REDUCE1, RB_K_CONV_WGRAD, RB_K_CONV_FWD, RB_KERNEL_COUNT
};

int rb_abi_version(void);
const char* rb_last_error(void);

/* Diagnostics (no reference counterpart): when enabled, every kernel launch is bracketed by CUDA events
 * on its stream (do not enable during CUDA-graph capture).  rb_profile_collect synchronises on the
 * recorded events of one kernel id, returns their summed duration and count, and clears them. */
int rb_profile_enable(int on);
int rb_profile_collect(int kernel_id, double* total_ms, int* launches);

/* memory.py:157-159 ReplayMemory.update_priorities -> :44-48 SegmentTree.update
 * (-> :28-33 _propagate -> :23-25 _update_nodes).
 * leaf[tree_idx[k]] = raw_priority[k]^omega (duplicates: last k wins), parents recomputed
 * level by level as fl32(left+right) up to the root, running_max = max(running_max, max_k leaf).
 * omega_is_applied != 0 means raw_priority already holds exponentiated values (SegmentTree.update).
 * status[0] is set to 1 if any tree_idx lies outside the leaf range (nothing is written for it).
 * gate (optional device int32, may be NULL): when *gate == 0 the launch does nothing (rejected sample batch). */
int rb_tree_update(float* tree, int64_t tree_start, int64_t size, const int64_t* tree_idx,
                   const float* raw_priority, float omega, int omega_is_applied, int B, float* running_max,
                   int32_t* status, const int32_t* gate, rb_stream_t stream);

/* memory.py:79-82 SegmentTree.find (-> :64-76 _retrieve): float64 residual against float32 nodes,
 * strict '>' goes right, child indices clipped to the last element on the leaf level. */
int rb_tree_find(const float* tree, int64_t tree_start, int64_t size, const double* values, int B, float* probs,
                 int64_t* data_idx, int64_t* tree_idx, rb_stream_t stream);

/* memory.py:148-154 ReplayMemory.sample head + :124-132 _get_samples_from_segments:
 * p_total = tree[0]; seg = fl32(p_total/B); v_k = seg*u_k + k*seg (float64); find; whole-batch
 * validity test (memory.py:131) with redraw; importance weights (count*p/p_total)^-beta / max.
 *   u01 != NULL : parity mode.  u01 is float64[u01_attempts][B] of unit uniforms (what
 *                 RandomState.uniform consumes); attempt a uses row a; at most u01_attempts tries.
 *   u01 == NULL : device Philox4x32-10 keyed by `seed`, counter *rng_counter (advanced by the
 *                 number of draws); at most max_attempts tries.
 * beta_dev (optional, may be NULL) overrides `beta` with a device scalar (graph replay). */
int rb_tree_sample(const float* tree, int64_t tree_start, int64_t size, const int64_t* ring_state, int n,
                   int history, const double* u01, int u01_attempts, uint64_t seed, uint64_t* rng_counter, int B,
                   float beta, const float* beta_dev, int max_attempts, float* probs, int64_t* data_idx,
                   int64_t* tree_idx, float* weights, int32_t* status, rb_stream_t stream);

/* memory.py:111-121 _get_transitions + :134-145 (tail of _get_samples_from_segments) + :85-86 get:
 * window of history+n records around each data_idx (indices mod size), episode-boundary blanking,
 * states = u8/255 [B,history,84,84], next_states (window shifted by n), actions int64[B],
 * returns = sum_k gamma_pow[k]*reward[B], nonterminals float32[B] (of the last window record). */
int rb_gather(const uint8_t* frames, const int32_t* timestep, const int32_t* action, const float* reward,
              const uint8_t* nonterminal, int64_t size, const int64_t* data_idx, int B, int history, int n,
              const float* gamma_pow, float* states, float* next_states, int64_t* actions, float* returns,
              float* nonterminals, rb_stream_t stream);

/* memory.py:166-178 ReplayMemory.__next__, batched: states for current_idx = first .. first+count-1,
 * backward-only blanking, negative indices wrap.  out is float32[count][history][84*84]. */
int rb_iter_states(const uint8_t* frames, const int32_t* timestep, int64_t size, int64_t first, int count,
                   int history, float* out, rb_stream_t stream);

/* memory.py:105-108 ReplayMemory.append -> :56-61 SegmentTree.append (-> :51-54, :36-41):
 * quantise the newest frame (f32*255, truncating cast), store the record at ring_state.head with
 * timestep = ring_state.t_episode, set its leaf to *running_max and walk to the root, advance the
 * head, set full on wrap, t_episode = terminal ? 0 : t_episode+1.
 * state_last_frame: float32[84*84] device pointer (state[-1]). */
int rb_append(float* tree, int64_t tree_start, int64_t size, uint8_t* frames, int32_t* timestep, int32_t* action,
              float* reward, uint8_t* nonterminal, int64_t* ring_state, float* running_max,
              const float* state_last_frame, int32_t action_value, float reward_value, int terminal,
              rb_stream_t stream);

/* k consecutive rb_append calls in ONE launch (actor side batching, SURVEY.md 8(f).2): HOST arrays of length k --
 * last_frames[j] points at the j-th newest frame (float32[84*84], DEVICE memory or PINNED HOST memory, read in place),
 * actions / rewards / terminals its fields.  Result is identical to k rb_append calls in order.  1 <= k <= RB_APPEND_BATCH.
 * (ReplayMemory(defer_appends=True) uses it.) */
int rb_append_batch(float* tree, int64_t tree_start, int64_t size, uint8_t* frames, int32_t* timestep, int32_t* action,
                    float* reward, uint8_t* nonterminal, int64_t* ring_state, float* running_max,
                    const float* const* last_frames, const int32_t* actions, const float* rewards, const int32_t* terminals,
                    int k, rb_stream_t stream);

/* agent.py:66-96 Agent.learn minus the three network bodies, given PRE-softmax logits [B,A,Z]
 * (model.py:75 `q`; the softmax / log_softmax of model.py:76-79 are folded in):
 * double-DQN argmax with the online net, target distribution, Tz clamp, l/u projection with the
 * reference's fix-ups and accumulation order, loss_i = -sum m*logp (the TD priority of
 * agent.py:100), and d(mean_i w_i*loss_i)/dq_online_s.  m_out / astar_out may be NULL. */
int rb_c51_loss_grad(const float* q_online_s, const float* q_online_ns, const float* q_target_ns,
                     const int64_t* actions, const float* returns, const float* nonterminals,
                     const float* weights, const float* support, float vmin, float vmax, float delta_z,
                     float gamma_n, int B, int A, int Z, float* loss, float* grad_q_online_s, float* m_out,
                     int64_t* astar_out, rb_stream_t stream);

/* model.py:82-85 DQN.reset_noise -> :36-40 NoisyLinear.reset_noise -> :32-34 _scale_noise, all
 * layers of one net in one launch.  HOST arrays (length n_layers): weight_eps[l] -> float32[out][in],
 * bias_eps[l] -> float32[out], in_features, out_features.
 *   x_in / x_out != NULL : parity mode, raw standard normals, concatenated over layers in layer
 *                          order (eps_in of layer 0, of layer 1, ... / eps_out likewise).
 *   NULL                 : device Philox + Box-Muller keyed by seed and *rng_counter (+1 per call). */
int rb_noisy_resample(float* const* weight_eps, float* const* bias_eps, const int* in_features,
                      const int* out_features, int n_layers, const float* x_in, const float* x_out, uint64_t seed,
                      uint64_t* rng_counter, rb_stream_t stream);

/* Materialise weight_epsilon / bias_epsilon (model.py:39-40) from ALREADY SCALED factor vectors
 * f(eps_in) / f(eps_out) (concatenated over layers like x_in / x_out above): eps_w = f_out (outer) f_in. */
int rb_noisy_outer(float* const* weight_eps, float* const* bias_eps, const int* in_features, const int* out_features,
                   int n_layers, const float* f_in, const float* f_out, rb_stream_t stream);

/* model.py:36-38 for every NoisyLinear of a net, WITHOUT the outer product: f_in[n_in] / f_out[n_out] receive
 * f(eps_in) / f(eps_out) of all layers back to back (layer order).  Same Philox indexing as
 * rb_noisy_resample: rb_noise_factors + rb_noisy_outer == rb_noisy_resample for equal seed and counter.
 * x_in / x_out: optional injected raw normals (parity).  *rng_counter += 1 in Philox mode. */
int rb_noise_factors(float* f_in, int n_in, float* f_out, int n_out, const float* x_in, const float* x_out, uint64_t seed,
                     uint64_t* rng_counter, rb_stream_t stream);

/* ---- fused factorised-noise dueling head (small batches) -----------------------------------------------
 * model.py:69-75 minus the conv body:  h_s = relu(x W1_s^T + b1_s), z_s = h_s W2_s^T + b2_s for the value (s=0) and
 * advantage (s=1) streams, W = mu + sigma * (eps_out (outer) eps_in) composed on the fly from the factor vectors
 * (model.py:39-44) -- weight_epsilon never has to exist in memory.  All pointers are device pointers; the eight
 * eps_* pointers are either all given (training mode) or all NULL (eval mode, model.py:45-46).
 * Requirements: see rb_head_supported. */
typedef struct rb_head_params {
  const float* w1_mu[2];    const float* w1_sigma[2];   /* [hidden][conv_features]        fc_h_v, fc_h_a */
  const float* b1_mu[2];    const float* b1_sigma[2];   /* [hidden] */
  const float* w2_mu[2];    const float* w2_sigma[2];   /* [atoms][hidden], [actions*atoms][hidden]   fc_z_v, fc_z_a */
  const float* b2_mu[2];    const float* b2_sigma[2];
  const float* eps_in1[2];  const float* eps_out1[2];   /* f(eps): [conv_features], [hidden] */
  const float* eps_in2[2];  const float* eps_out2[2];   /* [hidden], [atoms] / [actions*atoms] */
  int conv_features, hidden, atoms, actions;
} rb_head_params;

typedef struct rb_head_grads {   /* gradients are OVERWRITTEN (not accumulated) */
  float* w1_mu[2]; float* w1_sigma[2]; float* b1_mu[2]; float* b1_sigma[2];
  float* w2_mu[2]; float* w2_sigma[2]; float* b2_mu[2]; float* b2_sigma[2];
} rb_head_grads;

/* split-K factors used by the head kernels: scratch part1 is float32[s1][M][2*hidden], part2 float32[s2][M][atoms*(1+actions)];
 * tickets is int32[rb_head_ticket_count()], zero-initialised ONCE by the caller (the kernels leave it zeroed).
 * s1 is the larger of the two layer-1 implementations' factors (tensor-core kernel, csrc/rb_head_tc.cu; FFMA kernel). */
int rb_head_splits(int conv_features, int hidden, int* s1, int* s2);
int rb_head_ticket_count(void);
/* RB_OK if rb_head_forward takes a head of this shape at `rows` rows and, with with_backward != 0, rb_head_backward takes it
 * at a batch of `rows`; RB_ERR_RANGE for exactly the shapes those two refuse (conv_features % 32, hidden % 64,
 * atoms <= RB_MAX_ATOMS, the forward's split-K tile count, B <= 32, the dh kernel's shared memory ~ actions * atoms <= 1065,
 * hidden <= 1024).  Launches nothing; callers route the other shapes to the library path. */
int rb_head_supported(int conv_features, int hidden, int atoms, int actions, int rows, int with_backward);
/* probes / tests only: bit 0 skips the layer-1 launch of rb_head_forward, bit 1 the layer-2 launch, bit 2 forces the FFMA
 * layer-1 kernel instead of the tensor-core one (0 = normal) */
int rb_head_debug(int flags);

/* Forward over M = m_lo + m_hi rows (x_lo: [m_lo][conv_features], x_hi: [m_hi][conv_features] or NULL).
 * Outputs: h[M][2*hidden] (post-ReLU hidden activations, value stream in columns [0,hidden), advantage stream in
 * [hidden,2*hidden)) and z[M][atoms*(1+actions)] = (z_value | z_advantage), biases included.
 * Layer 1 runs on the tensor cores (TMA + tcgen05.mma, error-compensated TF32 = fp32-equivalent results; csrc/rb_head_tc.cu)
 * followed by a fixed-order split-K reduction kernel; shapes that kernel does not cover (m_hi > 0 with m_lo % 8 != 0) and
 * RB_HEAD_TC=0 in the environment use the FFMA kernel whose last-arriving CTA reduces the partials.  Deterministic. */
int rb_head_forward(const rb_head_params* p, const float* x_lo, int m_lo, const float* x_hi, int m_hi, float* part1, float* part2,
                    int32_t* tickets, float* h, float* z, rb_stream_t stream);

/* q[M][actions][atoms] = zv + za - mean_a(za) (model.py:75) from z. */
int rb_head_logits(const float* z, int M, int actions, int atoms, float* q, rb_stream_t stream);

/* Backward for B <= 32 rows: given dz[B][atoms*(1+actions)] (value block first), x[B][conv_features] and h[B][2*hidden]
 * writes all 16 parameter gradients through `g` and dx[B][conv_features].  dh_scratch: float32[(B + 32) * 2*hidden]
 * (dh [B][2*hidden], then its transpose [2*hidden][32] for the layer-1 kernel).
 * relu_mask_x != 0 additionally zeroes dx where x <= 0, i.e. folds in the backward of the ReLU that produced the conv
 * features (model.py:59), so dx is the gradient w.r.t. the last conv layer's pre-activation.
 * `parts` selects which of the three launches to enqueue (so a caller can put the independent layer-2 weight
 * gradient on another stream): RB_HEAD_BWD_WGRAD2 (layer-2 parameter gradients), RB_HEAD_BWD_DH (dh_scratch),
 * RB_HEAD_BWD_LAYER1 (layer-1 parameter gradients + dx; needs dh_scratch); RB_HEAD_BWD_ALL = all, in that order. */
#define RB_HEAD_BWD_WGRAD2 1
#define RB_HEAD_BWD_DH 2
#define RB_HEAD_BWD_LAYER1 4
#define RB_HEAD_BWD_ALL 7
int rb_head_backward(const rb_head_params* p, const rb_head_grads* g, const float* x, const float* h, const float* dz, int B,
                     float* dh_scratch, float* dx, int relu_mask_x, int parts, rb_stream_t stream);

/* agent.py:53-55 Agent.act / :110-112 evaluate_q after the network body, for M states at once: from the head output
 * z[M][atoms*(1+actions)] computes q[m][a] = sum_z support_z * softmax_z(zv + za[a] - mean_a za) (model.py:75-79) and its
 * arg-max / max over actions.  q (float32[M][actions]), best_action (int64[M]), best_q (float32[M]) are each optional. */
int rb_q_values(const float* z, int M, int actions, int atoms, const float* support, float* q, int64_t* best_action,
                float* best_q, rb_stream_t stream);

/* Bias gradient of a conv layer (the sum over batch and pixels torch computes in convolution_backward):
 * out[c] = sum_{b,p} grad_out[b][c][p], grad_out float32[B][C][HW] contiguous. */
int rb_bias_grad(const float* grad_out, int B, int C, int HW, float* out, rb_stream_t stream);

/* Weight gradient of a conv layer whose data gradient is not needed (the network's first layer; the weight half of
 * torch's convolution_backward there): out[oc][ic][ky][kx] = sum_{b,y,x} grad_out[b][oc][y][x] * input[b][ic][y*stride+ky][x*stride+kx]
 * for a square K x K kernel without padding (K in {3, 4, 5, 8}; IC * K * ceil(OC/4) <= 256).  grad_out float32
 * [B][OC][OH][OW], input float32 [B][IC][IH][IW] (OH = (IH-K)/stride + 1), out float32 [OC][IC][K][K] (overwritten),
 * bias_out (optional, may be NULL) float32 [OC] = sum_{b,y,x} grad_out (the layer's bias gradient, from the same pass),
 * partials: scratch of rb_conv_wgrad_scratch_elems(...) floats.  Two launches, fixed summation order (deterministic). */
int rb_conv_wgrad_scratch_elems(int B, int IC, int IH, int OC, int K, int stride);
int rb_conv_wgrad(const float* grad_out, const float* input, int B, int IC, int IH, int IW, int OC, int K, int stride,
                  float* partials, float* out, float* bias_out, rb_stream_t stream);

/* model.py:55-63, one conv layer of the network body and the ReLU after it:
 * out[b][oc][oy][ox] = max(0, bias[oc] + sum_{ic,ky,kx} weight[oc][ic][ky][kx] * input[b][ic][oy*stride+ky][ox*stride+kx])
 * for a square K x K kernel without padding, dilation or groups.  input float32 [B][IC][IH][IW], weight float32
 * [OC][IC][K][K], bias float32 [OC], out float32 [B][OC][OH][OW] (OH = (IH-K)/stride + 1), all contiguous.
 * Runs on the tensor cores as an error-compensated TF32 product (fp32-equivalent results whatever torch's allow_tf32 says),
 * one launch, fixed summation order (deterministic).  (K, stride) in {(8,4), (4,2), (3,1), (5,5)} and OC % 32 == 0 are
 * instantiated; other shapes return RB_ERR_RANGE without launching anything. */
int rb_conv_forward(const float* input, const float* weight, const float* bias, int B, int IC, int IH, int IW, int OC, int K,
                    int stride, float* out, rb_stream_t stream);

/* rb_c51_loss_grad fed by the fused heads: z_online has 2B rows (s then s'), z_target B rows (s');
 * returns loss[B] and dz[B][atoms*(1+actions)] = d mean(w*loss) / d (z_value | z_advantage) of the online(s) rows
 * (the dueling combination model.py:75 and its backward are folded in). */
int rb_c51_dueling_loss_grad(const float* z_online, const float* z_target, int actions_n, int atoms, const int64_t* actions,
                             const float* returns, const float* nonterminals, const float* weights, const float* support,
                             float vmin, float vmax, float delta_z, float gamma_n, int B, float* loss, float* dz, float* m_out,
                             int64_t* astar_out, rb_stream_t stream);

/* model.py:43-44 NoisyLinear.forward weight composition W = mu + sigma*eps (elementwise),
 * used for both weights ([out*in]) and biases ([out]). */
int rb_noisy_compose(const float* mu, const float* sigma, const float* eps, int64_t count, float* out,
                     rb_stream_t stream);

/* agent.py:97-98 clip_grad_norm_(params, max_norm) + Adam.step() on FLAT float32 buffers of P
 * elements (all online-net parameters laid out back to back).  `step_count` is a device int64 holding
 * the number of steps already taken; the kernel increments it.  grad_scale multiplies the gradient
 * before everything else (1/world_size after a SUM all-reduce; 1.0 on one GPU).
 * partial_sums: scratch float64[rb_clip_adam_scratch_elems()], ZERO-INITIALISED once by the caller (its last element is a
 * self-resetting completion ticket).  norm_out (optional) receives the
 * pre-clip global L2 norm.  gate (optional device int32, may be NULL): when *gate == 0 neither the parameters, the
 * moments nor step_count change (rejected sample batch, see rb_tree_sample). */
int rb_clip_adam_scratch_elems(void);
int rb_clip_adam(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t P, float grad_scale,
                 float max_norm, float lr, float beta1, float beta2, float eps, int64_t* step_count,
                 double* partial_sums, float* norm_out, const int32_t* gate, rb_stream_t stream);

/* Multi-GPU replacement of "all-reduce the flat gradient, then rb_clip_adam on every rank" (agent.py:97-98 under data
 * parallelism; no reference counterpart): reduce-scatter by peer loads + clip + Adam on the owned 1/world parts (moments
 * sharded) + all-gather by peer stores, ordered by epoch flags in peer-visible memory.  HOST arrays of length `world`:
 * peer_grad[q] / peer_param[q] = rank q's flat gradient / parameter buffer, peer_flags[q] = rank q's uint64[4*world] flag
 * block, peer_norms[q] = rank q's double[world] block (both zero-initialised once), all mapped on this device.
 * epoch: device uint64 (zero-initialised, advanced once per step by rb_peer_adam_gather); scratch: rb_peer_scratch_bytes()
 * zeroed bytes.  Every rank must make the same calls each step.
 *
 * The flat buffer is exchanged as one or two SEGMENTS [seg_begin, seg_begin + seg_len) (seg_len % (4*world) == 0); rank r
 * owns part r (seg_len / world elements) of each.  rb_peer_reduce reduces one segment (it may be enqueued on another
 * stream as soon as that segment's gradients are final -- the learner sends the noisy-head segment while the conv backward
 * still runs); gred_part receives this rank's reduced part, multiplied by grad_scale (1/world for averaging).
 * rb_peer_adam_gather (after every segment's rb_peer_reduce, stream-ordered) publishes the partial norms, clips, runs Adam
 * on the owned parts -- gred / exp_avg / exp_avg_sq hold the parts of segment 0, then segment 1, back to back --, stores the
 * new parameters into every rank's buffer and returns when all ranks' parts have landed here.  multicast_param (optional,
 * may be NULL): the NVLS multicast mapping of the parameter buffers (one address that the NVSwitch replicates to every
 * rank); when given, the all-gather is a single multimem.st per 16 bytes instead of `world` peer stores.
 * rb_peer_clip_adam = rb_peer_reduce over [0, P) + rb_peer_adam_gather with that single segment.
 * Validated on 4 x B200 against NCCL all-reduce + rb_clip_adam (tools/peer_adam_check.py). */
int rb_peer_scratch_bytes(void);
int rb_peer_reduce(const float* const* peer_grad, uint64_t* const* peer_flags, int world, int rank, int seg, int64_t seg_begin,
                   int64_t seg_len, float grad_scale, float* gred_part, const uint64_t* epoch, void* scratch,
                   rb_stream_t stream);
int rb_peer_adam_gather(float* const* peer_param, uint64_t* const* peer_flags, double* const* peer_norms, int world, int rank,
                        int n_seg, const int64_t* seg_begin, const int64_t* seg_len, const float* gred, float* exp_avg,
                        float* exp_avg_sq, float max_norm, float lr, float beta1, float beta2, float eps, int64_t* step_count,
                        uint64_t* epoch, void* scratch, float* norm_out, float* multicast_param, rb_stream_t stream);
int rb_peer_clip_adam(const float* const* peer_grad, float* const* peer_param, uint64_t* const* peer_flags,
                      double* const* peer_norms, int world, int rank, int64_t P, float* gred, float* exp_avg,
                      float* exp_avg_sq, float grad_scale, float max_norm, float lr, float beta1, float beta2, float eps,
                      int64_t* step_count, uint64_t* epoch, void* scratch, float* norm_out, rb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* RAINBOW_B200_H */
