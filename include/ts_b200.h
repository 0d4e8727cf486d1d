/*
 * ts_b200.h -- C ABI of the B200-native policy-update hot path for Tianshou-style RL.
 *
 * The reference (thu-ml/tianshou 2.0.1) has NO FFI: its hot path is Python + numba @njit +
 * stock torch ops.  This header declares the entry points a maintainer binds (ctypes / cffi,
 * see INTEGRATION.md) in place of those numba kernels and torch loops.  Every function
 *   - takes plain device pointers, sizes and a cudaStream_t (passed as void*),
 *   - is asynchronous on that stream (no host sync, no allocation, no hidden global state),
 *   - returns 0 on success, non-zero on error; ts_last_error() gives the thread-local message.
 * Pointers are DEVICE pointers unless a parameter is documented as "host".  "u8" flags are
 * numpy/torch bool storage (one byte, 0/1).
 *
 * Each declaration cites the reference code it replaces (path:line under /root/reference).
 */
#ifndef TS_B200_H_
#define TS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TS_B200_ABI_VERSION 1

typedef void* ts_stream_t; /* cudaStream_t */

/* dtype tags for the few polymorphic entry points */
enum { TS_F32 = 0, TS_F64 = 1 };

int ts_version(void);
const char* ts_last_error(void);
/* number of kernel launches issued through this library by the calling process (for bench.py's
 * "gpu_launches" claim); ts_reset_launch_count() zeroes it. */
int64_t ts_launch_count(void);
void ts_reset_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * (1) GAE: segmented reverse scan.
 * Replaces numba `_gae` (tianshou/algorithm/algorithm_base.py:1085-1140) together with the
 * value-mask / end-flag / return-scaling arithmetic around it in
 * `Algorithm.compute_episodic_return` (:704-719) and
 * `ActorCriticOnPolicyAlgorithm._add_returns_and_advantages` (modelfree/a2c.py:131-152):
 *
 *   s      = rms_state ? sqrt(rms_state.var + rms_eps) : 1         (return_scaling un-normalise)
 *   vs     = v_s[i] * s ;  vn = v_s_next[i] * s * (terminated ? !terminated[i] : 1)
 *   delta  = rew[i] + vn*gamma - vs
 *   end    = (truncated?truncated[i]:0) | (terminated_ends?terminated[i]:0) | (extra_end?extra_end[i]:0)
 *   adv[i] = delta + (1-end)*gamma*lam * adv[i+1]        (adv[n] = 0; f64 accumulate)
 *   ret[i] = (adv[i] + vs) / s
 * and, if rms_state != NULL, merges mean/var/count of the UN-scaled returns (adv+vs) into
 * rms_state with Chan's formula exactly as `RunningMeanStd.update`
 * (tianshou/utils/statistics.py:99-114) -- after every block has read the old var.
 *
 * v_s / v_s_next: n values of v_dtype (TS_F32|TS_F64).  rew: n f64 (the buffer stores float64,
 * data/buffer/manager.py:183).  terminated / truncated / extra_end: n u8, each nullable.
 * terminated_ends: if non-zero `terminated` also ends a segment (the normal case); the value
 * mask always uses it when non-NULL.  adv_out / ret_out: n values of out_dtype.
 * rms_state: device double[3] = {mean, var, count} (nullable).
 * batch_moments_out: see ts_rms_merge below (nullable).
 * workspace: device scratch of ts_gae_workspace_bytes(n) bytes (contents ignored).
 * ------------------------------------------------------------------------------------------ */
size_t ts_gae_workspace_bytes(int64_t n);
int ts_gae(const void* v_s, const void* v_s_next, int v_dtype, const double* rew,
           const uint8_t* terminated, const uint8_t* truncated, const uint8_t* extra_end,
           int terminated_ends, int64_t n, double gamma, double lam, double* rms_state,
           double rms_eps, double* batch_moments_out, void* adv_out, void* ret_out, int out_dtype,
           void* workspace, ts_stream_t stream);
/* Multi-GPU return scaling: when batch_moments_out (device double[3] = {count, mean, M2} of this
 * call's un-scaled returns) is non-NULL, ts_gae writes it and leaves rms_state untouched; the
 * caller all-gathers the triples and folds them in rank order with ts_rms_merge so that every
 * replica holds the same RunningMeanStd (SURVEY 8e). */
int ts_rms_merge(double* rms_state, const double* moments /* parts x 3 */, int32_t parts,
                 ts_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (2) n-step return: windowed gather-reduce.
 * Replaces numba `_nstep_return` (algorithm_base.py:1160-1222) and the whole-buffer
 * `end_flag_B = done.copy(); end_flag_B[unfinished] = True` preparation (:799-800).
 *   rew: B f64 (whole buffer), end_flag: B u8, target_q: I*A f32 (already value-masked),
 *   stacked_idx: n_step rows of I int64 (row k = next^k(indices)), out: I*A of out_dtype.
 * Arithmetic is f64 in the reference's operation order (no FMA contraction) => bit-exact f64.
 * ------------------------------------------------------------------------------------------ */
int ts_nstep_return(const double* rew, const uint8_t* end_flag, const float* target_q,
                    const int64_t* stacked_idx, int64_t I, int64_t A, int32_t n_step,
                    double gamma, void* out, int out_dtype, ts_stream_t stream);

/* end_flag[i] = done[i] | (i is the last written slot of a non-empty sub-buffer); B = offset[E].
 * Replaces algorithm_base.py:799-800 + manager.py:85-91 without the host copy. */
int ts_buffer_end_flags(const uint8_t* done, const int64_t* offset, const int64_t* last_index,
                        const int64_t* lengths, int64_t E, uint8_t* end_flag_out,
                        ts_stream_t stream);

/* target_q[i, :] *= !terminated[idx[i]]  (Algorithm.value_mask, algorithm_base.py:633-651,798) */
int ts_value_mask_rows(float* target_q, const uint8_t* terminated, const int64_t* idx, int64_t I,
                       int64_t A, ts_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (3) Replay-buffer index kernels (bit-exact int64).
 * Sub-buffer e owns slots [offset[e], offset[e+1]); lengths[e] = current size; last_index[e] =
 * absolute last-written slot.  A plain ReplayBuffer is the E=1 case.
 * Replace numba `_next_index` / `_prev_index` (tianshou/data/buffer/manager.py:339-363,
 * :311-336) and ReplayBuffer.next/prev (buffer_base.py:319-334).
 * ------------------------------------------------------------------------------------------ */
int ts_next_index(const int64_t* index, int64_t n, const int64_t* offset, int64_t E,
                  const uint8_t* done, const int64_t* last_index, const int64_t* lengths,
                  int64_t* out, ts_stream_t stream);
int ts_prev_index(const int64_t* index, int64_t n, const int64_t* offset, int64_t E,
                  const uint8_t* done, const int64_t* last_index, const int64_t* lengths,
                  int64_t* out, ts_stream_t stream);
/* out[k*n + i] = next^k(index[i]) for k = 0..n_step-1 (algorithm_base.py:775-779). */
int ts_stack_next_indices(const int64_t* index, int64_t n, int32_t n_step, const int64_t* offset,
                          int64_t E, const uint8_t* done, const int64_t* last_index,
                          const int64_t* lengths, int64_t* out, ts_stream_t stream);
/* ReplayBufferManager.unfinished_index (manager.py:85-91; buffer_base.py:314-317): ordered list
 * of the slots before each sub-buffer's insertion index whose `done` is false.  insertion_idx: device
 * int64[E] relative to the sub-buffer start (nullable: last_index is used, which is the same slot for buffers
 * filled by add() alone).  out: capacity E; count_out: device int64[1]. */
int ts_unfinished_index(const int64_t* offset, int64_t E, const uint8_t* done,
                        const int64_t* last_index, const int64_t* lengths, const int64_t* insertion_idx,
                        int64_t* out, int64_t* count_out, ts_stream_t stream);
/* sample_indices(0): all valid slots, sub-buffer-major, chronological inside each sub-buffer
 * (manager.py:217-234, buffer_base.py:519-525).  insertion_idx: device int64[E], every sub-buffer's
 * `_insertion_idx` relative to its own start (nullable: derived as last_index + 1, which is only right for
 * buffers filled by add() alone -- from_data() / dropnull() move it independently).  seg_start: device
 * int64[E+1] scratch that receives the exclusive prefix sum of lengths; out capacity >= sum(lengths);
 * total_out int64[1]. */
int ts_sample_all_indices(const int64_t* offset, int64_t E, const int64_t* last_index,
                          const int64_t* lengths, const int64_t* insertion_idx, int64_t* seg_start,
                          int64_t* out, int64_t out_capacity, int64_t* total_out, ts_stream_t stream);
/* mark[p] = 1 if idx[p] is in `members` (np.isin, algorithm_base.py:715).  table: device u8
 * scratch of table_size >= max slot + 1, left zeroed on return. */
int ts_mark_members(const int64_t* idx, int64_t n, const int64_t* members,
                    const int64_t* member_count /* device int64[1] */, int64_t member_capacity,
                    uint8_t* table, int64_t table_size, uint8_t* mark_out, ts_stream_t stream);
/* dst[p, :] = src[idx[p], :] for rows of row_bytes (multiple of 4) -- ReplayBuffer.__getitem__
 * (buffer_base.py:605-649) / Batch.__getitem__ (data/batch.py:714-738) for array leaves. */
int ts_gather_rows(const void* src, int64_t row_bytes, const int64_t* idx, int64_t n, void* dst,
                   ts_stream_t stream);

/* dst[idx[p]] = src[p] for p < n, rows of row_bytes bytes: the device side of the asynchronous buffer mirror --
 * ReplayBuffer.add (buffer_base.py:420-501, manager.py:131-198) writes one row per env at scattered slots; the
 * rows arrive contiguously from pinned staging.  idx entries must be distinct. */
int ts_scatter_rows(const void* src, int64_t row_bytes, const int64_t* idx, int64_t n, void* dst,
                    ts_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (4) Sum tree for prioritized replay (f64 tree, bit-exact indices).
 * tree: double[2*bound], root at 1, leaves at [bound, bound+size) (data/utils/segtree.py:19-26).
 * Replace numba `_setitem` (:95-101), `_reduce` (:104-116), `_get_prefix_sum_idx` (:119-134).
 * ------------------------------------------------------------------------------------------ */
/* tree[bound+index[k]] = value[k] (duplicates: last wins), then parents re-summed bottom-up. */
int ts_segtree_setitem(double* tree, int64_t bound, const int64_t* index, const void* value,
                       int value_dtype, int64_t n, ts_stream_t stream);
/* out[0] = sum(leaves[start:end]) using the reference's bottom-up walk (same addition order). */
int ts_segtree_reduce(const double* tree, int64_t bound, int64_t start, int64_t end, double* out,
                      ts_stream_t stream);
/* out[k] = min i such that value[k] <= sum(leaves[0..i]) (ties go left).  value: n f64. */
int ts_segtree_prefix_sum_idx(const double* tree, int64_t bound, const double* value, int64_t n,
                              int64_t* out, ts_stream_t stream);
/* value[k] = u[k] * tree[1] then descent -- fuses `np.random.rand(bs) * weight.reduce()`
 * (data/buffer/prio.py:65-66); u stays a host-drawn numpy stream uploaded by the caller. */
int ts_segtree_sample(const double* tree, int64_t bound, const double* u, int64_t n, int64_t* out,
                      ts_stream_t stream);
/* PrioritizedReplayBuffer.update_weight (prio.py:81-90): w = |td|+eps; tree[idx] = w^alpha;
 * prio_minmax (device double[2] = {max_prio, min_prio}) updated with max/min of w. */
int ts_prio_update_weight(double* tree, int64_t bound, const int64_t* index, const void* td,
                          int td_dtype, int64_t n, double alpha, double eps, double* prio_minmax,
                          ts_stream_t stream);
/* PrioritizedReplayBuffer.get_weight (+ batch-max normalisation, prio.py:69-79,104-106):
 * out[k] = (tree[bound+idx[k]] / min_prio)^(-beta), divided by the batch max if weight_norm. */
int ts_prio_get_weight(const double* tree, int64_t bound, const int64_t* index, int64_t n,
                       const double* prio_minmax, double beta, int weight_norm, double* out,
                       ts_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (5) Actor-critic MLP (two tanh hidden layers of width `hidden`, separate actor and critic
 * trunks, Gaussian policy head with state-independent log-sigma) -- the network of
 * examples/mujoco/mujoco_ppo.py:90-120 built from tianshou/utils/net/common.py:172-179,343-369
 * and continuous.py:144-169,220-238.
 * All parameters live in ONE flat f32 buffer in torch layout ([out][in] row-major weights);
 * offsets are in floats.  The same offsets index the flat gradient / Adam-moment buffers.
 *
 * Variants selected by `flags` (the reference's discrete PPO test net, test/discrete/test_ppo_discrete.py:90-100:
 * ONE Net(obs -> 64 -> 64, ReLU) shared by DiscreteActor(softmax_output=True) and DiscreteCritic,
 * utils/net/discrete.py:29-123, policy distribution torch.distributions.Categorical(probs)):
 *   TS_AC_RELU         hidden activation max(x, 0) instead of tanh (Net's default, common.py MLP);
 *   TS_AC_CATEGORICAL  head = act_dim logits -> softmax -> Categorical; a_logstd is unused (-1); the
 *                      action array holds ONE index per row, stored as f32 (ppo.py:156 casts it so).
 * A SHARED trunk is expressed by aliased offsets (c_w1 == a_w1, c_b1 == a_b1, c_w2 == a_w2, c_b2 == a_b2): the
 * shared parameters are counted once in n_params and both losses' gradients add into the same slots.
 * Variants with flags != 0 or a shared trunk run the fp32 SIMT kernels.
 * ------------------------------------------------------------------------------------------ */
#define TS_AC_RELU 1
#define TS_AC_CATEGORICAL 2
typedef struct ts_actor_critic_desc {
    int32_t obs_dim;  /* <= 64 */
    int32_t act_dim;  /* <= 16 */
    int32_t hidden;   /* 64 */
    int32_t flags;           /* TS_AC_* bits; 0 = tanh trunks + diagonal-Gaussian head */
    int64_t a_w1, a_b1, a_w2, a_b2, a_w3, a_b3, a_logstd; /* actor: W1[h][obs] .. W3[act][h], logstd[act] */
    int64_t c_w1, c_b1, c_w2, c_b2, c_w3, c_b3;           /* critic: .. W3[1][h], b3[1] */
    int64_t n_params;
} ts_actor_critic_desc;

/* v_out[r] = critic(obs[r, :]) for r < n.  Up to two (obs, out) pairs in one launch (v_s and
 * v_s_ of a2c.py:123-126); pass obs1 = NULL for a single pass.  obs rows are obs_dim f32, dense. */
int ts_critic_forward(const float* params, const ts_actor_critic_desc* desc /* host */,
                      const float* obs0, float* v_out0, const float* obs1, float* v_out1,
                      int64_t n, ts_stream_t stream);
/* logp_out[r] = Independent(Normal(mu(obs[r]), exp(logstd)), 1).log_prob(act[r])
 * (ppo.py:157-161 with reinforce.py:167-192).  mu_out (n*act_dim, nullable) receives mu.
 * TS_AC_CATEGORICAL: logp_out[r] = Categorical(probs = softmax(logits(obs[r]))).log_prob(act[r]) with act one f32
 * index per row; mu_out receives the probabilities (the actor's output). */
int ts_actor_logp(const float* params, const ts_actor_critic_desc* desc /* host */,
                  const float* obs, const float* act, int64_t n, float* logp_out, float* mu_out,
                  ts_stream_t stream);

typedef struct ts_ppo_hparams {
    /* all hyper-parameters are doubles (Python floats in the reference); the kernels narrow to
     * f32 at the point where torch would (scalar operand of an f32 tensor op) */
    double eps_clip;
    double dual_clip;     /* <= 0: disabled */
    double vf_coef;
    double ent_coef;
    double max_grad_norm; /* <= 0: no clipping */
    double adv_eps;       /* 1e-8 in the reference (self._eps) */
    /* Adam (torch.optim.Adam semantics, algorithm/optim.py:89-110) */
    double lr, beta1, beta2, adam_eps, weight_decay;
    int32_t value_clip;
    int32_t advantage_normalization;
    int32_t loss_kind;    /* TS_LOSS_PPO (0): clipped surrogate, ppo.py:184-196; TS_LOSS_A2C (1): actor loss
                           * -mean(log_prob * adv) (a2c.py:262-266), eps_clip / dual_clip / logp_old / v_s unused */
} ts_ppo_hparams;
#define TS_LOSS_PPO 0
#define TS_LOSS_A2C 1

/* Per-optimiser-step device statistics: {loss, clip_loss, vf_loss, ent_loss, grad_norm, n_rows,
 * 0, 0} -- 8 floats per step (ppo.py:213-216 without the 4 host syncs). */
#define TS_PPO_STATS_STRIDE 8
/* grad buffer layout: n_params floats + TS_PPO_GRAD_EXTRA scalar slots {sum_clip, sum_vf,
 * sum_ent, n_rows} so that ONE allreduce carries gradients and loss sums (SURVEY 8e). */
#define TS_PPO_GRAD_EXTRA 4

/* One minibatch forward/backward (ppo.py:179-211 + loss.backward of algorithm_base.py:497):
 * rows are perm[lo..hi) of the rollout tensors.  Every CTA writes ITS OWN partial sum of
 * d(loss)/d(params) (already scaled by 1/global_rows) and of the four loss sums into row
 * blockIdx.x of `partials` ([ts_ppo_partial_rows()][n_params + TS_PPO_GRAD_EXTRA] floats) -- no
 * cross-CTA atomics, deterministic.  *n_partials_out (host) receives the number of rows written;
 * they are folded by ts_grad_reduce / ts_clip_adam_step.  `global_rows` is the minibatch size
 * over all ranks (the mean's denominator); adv_moments: device float[2] = {mean, std} when
 * advantage_normalization, else NULL.  perm may be NULL (identity). */
int32_t ts_ppo_partial_rows(void);

/* Bytes of the optional `weight_image` scratch of ts_ppo_update: a 128-byte control block (grid-barrier state of
 * the persistent kernel: must be ZERO when first used and is left zero by every launch; one scratch per model, never
 * shared by two updates in flight) followed by both networks' weights pre-split into the bf16x3 tensor-core operand
 * layout, so that a CTA stages a network with one bulk copy.  0 when the network
 * shape is not covered by the tensor-core kernels (pass NULL then). */
int64_t ts_ppo_weight_image_bytes(const ts_actor_critic_desc* desc);
int ts_ppo_grad(const float* params, const ts_actor_critic_desc* desc, const ts_ppo_hparams* hp,
                const float* obs, const float* act, const float* adv, const float* ret,
                const float* logp_old, const float* v_s, const int32_t* perm, int64_t lo,
                int64_t hi, int64_t global_rows, const float* adv_moments, float* partials,
                int32_t* n_partials_out /* host */, ts_stream_t stream);
/* grad[i] = sum_p partials[p][i] (fixed order) for i < n_params + TS_PPO_GRAD_EXTRA: the flat
 * gradient + loss sums a multi-GPU caller all-reduces before ts_clip_adam_step. */
int ts_grad_reduce(const float* partials, int32_t n_partials, const ts_actor_critic_desc* desc,
                   float* grad, ts_stream_t stream);
/* mean and unbiased std of adv[perm[lo..hi)] (ppo.py:184-186) -> out[0..1]; partial sums go to
 * sums (device double[2]) first so a multi-GPU caller can allreduce them; pass finalize=1 to
 * turn (sum, sumsq, count=global_rows) into {mean, std}. */
int ts_minibatch_adv_sums(const float* adv, const int32_t* perm, int64_t lo, int64_t hi,
                          double* sums, ts_stream_t stream);
int ts_adv_moments_finalize(const double* sums, int64_t global_rows, float* out,
                            ts_stream_t stream);
/* clip_grad_norm_ + Adam.step (algorithm_base.py:496-500; torch/optim/adam.py single-tensor
 * path) on the flat buffers, and one row of per-step statistics.  If partials != NULL the
 * gradient is first folded from the n_partials rows (single-GPU fast path: reduce + norm + clip
 * + Adam in ONE launch); otherwise `grad` must already hold the (all-reduced) gradient.
 * grad: n_params + TS_PPO_GRAD_EXTRA floats (scratch / input).  step_count: device int64[1],
 * incremented.  stats_row: device float[TS_PPO_STATS_STRIDE]. */
int ts_clip_adam_step(float* params, float* grad, const float* partials, int32_t n_partials,
                      float* exp_avg, float* exp_avg_sq, int64_t* step_count,
                      const ts_actor_critic_desc* desc, const ts_ppo_hparams* hp, float* stats_row,
                      ts_stream_t stream);

/* The whole single-GPU `PPO._update_with_batch` loop (ppo.py:164-224) on one stream:
 * for r in repeat: [recompute v_s/returns/adv (a2c.py:115-153)] ; for each minibatch of
 * perm[r] (Batch.split bounds, batch.py:1199-1215): grad + clip + Adam.  No host sync.
 * perm: repeat*N int32 (row r = the permutation of repeat r).  bounds: host int64[2*n_mb].
 * rollout tensors (all N rows, device): obs, obs_next, act f32; rew f64; terminated,
 * truncated, extra_end u8; v_s, returns, adv, logp_old f32 (in/out: must be valid on entry,
 * rewritten when recompute_adv).  stats: repeat*n_mb rows.  rms_state as in ts_gae (nullable
 * when return_scaling is off).  v_next_tmp: N f32 scratch.  gae_ws: ts_gae_workspace_bytes(N).
 * grad: n_params + TS_PPO_GRAD_EXTRA floats scratch; partials: ts_ppo_partial_rows() rows of the
 * same width.  adv_tmp: 32 + 8 * n_minibatch bytes of zero-initialised scratch (double[2] sums, float[2] moments,
 * then one (mean, std) float pair per minibatch).  weight_image: ts_ppo_weight_image_bytes(desc) bytes of scratch
 * (nullable: the kernels then gather + split the weights themselves every step); rebuilt from `params` on entry.
 * row_feed: NULL, or a feed from ts_host_perm_feed_start whose dev_rows == perm: pass r then waits (on `stream`, not on the
 * host) until row r of the host permutation job has arrived in `perm`.
 */
int ts_ppo_update(float* params, float* grad, float* partials, float* exp_avg, float* exp_avg_sq,
                  int64_t* step_count, const ts_actor_critic_desc* desc, const ts_ppo_hparams* hp,
                  const float* obs, const float* obs_next, const float* act, const double* rew,
                  const uint8_t* terminated, const uint8_t* truncated, const uint8_t* extra_end,
                  float* v_s, float* returns, float* adv, const float* logp_old,
                  float* v_next_tmp, int64_t N, const int32_t* perm, int32_t repeat,
                  const int64_t* bounds /* host */, int32_t n_minibatch, int32_t recompute_adv,
                  double gamma, double lam, double* rms_state, double rms_eps, void* gae_ws,
                  void* adv_tmp, void* weight_image, float* stats, void* row_feed, ts_stream_t stream);

/* ---- multi-GPU fused update: gradient all-reduce INSIDE the epoch kernel over NVLink peer memory -------------
 * Replaces, for one process per GPU (data-parallel replicas, each rank owns its own rollout shard), the
 * reference's single-process optimiser step (ppo.py:215-218) x world ranks: the loss is the mean over the
 * union of the ranks' local minibatches, the summed gradient / global-norm clip / Adam step are bit-identical
 * on every rank.  No NCCL call on the data path: after the local fold every CTA pushes its slice of the
 * gradient as (fp32 value, sequence number) 8-byte packets straight into every peer's exchange buffer and
 * gathers the peers' packets from its own.
 *
 * Plumbing: ts_peer_alloc cudaMalloc's + zeroes a buffer and returns its CUDA IPC handle (TS_PEER_HANDLE_BYTES
 * opaque bytes the host exchanges, e.g. with torch.distributed.all_gather); ts_peer_open maps a peer's buffer
 * into this process; ts_peer_close / ts_peer_free undo them.  Buffer size: ts_ppo_peer_buffer_bytes(desc, world)
 * (world <= 8).  The buffers carry a sequence number across launches: allocate once, zero-initialised, and use
 * them for every update of the same replicas. */
#define TS_PEER_HANDLE_BYTES 64
int ts_peer_alloc(int64_t bytes, void** ptr_out, uint8_t* handle_out /* TS_PEER_HANDLE_BYTES */);
int ts_peer_open(const uint8_t* handle, void** ptr_out);
int ts_peer_close(void* ptr);
int ts_peer_free(void* ptr);
int64_t ts_ppo_peer_buffer_bytes(const ts_actor_critic_desc* desc, int32_t world);

/* Per-minibatch advantage moments of one pass across ranks (ppo.py:181-183 on the global minibatch):
 * ts_epoch_adv_sums writes (sum, sum of squares) in f64 per minibatch of THIS rank's shard; the host all-reduces
 * the 2 * n_minibatch doubles; ts_epoch_adv_finalize turns them into (mean, unbiased std) float pairs for
 * minibatches of world * (hi - lo) rows. */
int ts_epoch_adv_sums(const float* adv, const int32_t* perm, int64_t lo0, int64_t mb_size, int64_t end,
                      int32_t n_minibatch, double* sums, ts_stream_t stream);
int ts_epoch_adv_finalize(const double* sums, int64_t lo0, int64_t mb_size, int64_t end, int32_t n_minibatch,
                          int32_t world, float* out, ts_stream_t stream);

/* ONE pass over the minibatches [lo0 + m * mb_size, ...) (last one ends at `end`; Batch.split bounds,
 * batch.py:1199-1215) of this rank's shard, every optimiser step of the pass in one persistent launch, gradients
 * summed over the `world` ranks in-kernel.  Arguments as ts_ppo_update (perm: this pass's N int32 or NULL;
 * stats: n_minibatch rows, global losses).  adv_moments: n_minibatch (mean, std) pairs from
 * ts_epoch_adv_finalize, required iff hp->advantage_normalization.  peer_buffers: host array of `world` device
 * pointers (index = rank; own buffer from ts_peer_alloc, the others from ts_peer_open); world == 1: may be NULL.
 * Every rank must call with the same shapes and the same number of minibatches.  A peer that does not show
 * up within 20 s traps the kernel (CUDA error at the next synchronisation) instead of hanging the GPU. */
int ts_ppo_epoch_multi(float* params, float* grad, float* partials, float* exp_avg, float* exp_avg_sq,
                       int64_t* step_count, const ts_actor_critic_desc* desc, const ts_ppo_hparams* hp,
                       const float* obs, const float* act, const float* adv, const float* returns,
                       const float* logp_old, const float* v_s, const int32_t* perm, int64_t lo0,
                       int64_t mb_size, int64_t end, int32_t n_minibatch, const float* adv_moments,
                       void* weight_image, float* stats, int32_t rank, int32_t world,
                       void* const* peer_buffers /* host */, ts_stream_t stream);

/* HOST function (no device work): out[0..n) = np.random.permutation(n) for numpy's legacy MT19937 RandomState whose
 * state is (key[624], *pos) -- the draw Batch.split makes once per pass (batch.py:1209).  Bit-identical to numpy
 * (MT19937 + random_interval masked rejection + backward Fisher-Yates of RandomState.shuffle); key / *pos are
 * advanced exactly as numpy would, so writing them back with np.random.set_state keeps the global stream in step.
 * Writes int32 directly (e.g. into the pinned upload buffer). */
int ts_host_mt19937_permutation(uint32_t* key /* in/out */, int32_t* pos /* in/out */, int64_t n, int32_t* out);

/* HOST, asynchronous: all `repeat` permutations of one update() (rows of out[repeat][n], int32, typically pinned),
 * identical to `repeat` consecutive np.random.permutation(n) draws from the state (key, pos).  A producer thread walks the
 * MT19937 stream, n_workers threads apply the swaps of different passes concurrently; ts_host_perm_job_wait(job, r)
 * blocks until row r is complete (rows complete in order of r up to worker interleaving); ts_host_perm_job_finish joins
 * the threads, returns the advanced generator state (write it back with np.random.set_state) and frees the job.
 * `out` must stay valid until finish.  Valid because nothing else consumes numpy's global stream inside
 * Algorithm.update() (batch.py:1209 is its only draw). */
int ts_host_perm_job_start(const uint32_t* key, int32_t pos, int64_t n, int32_t repeat, int32_t* out, int32_t n_workers,
                           void** job_out);
int ts_host_perm_job_wait(void* job, int32_t r);
int ts_host_perm_job_finish(void* job, uint32_t* key_out, int32_t* pos_out);

/* Asynchronous feed of a job's rows to the device -- the hand-over of `Batch.split`'s per-pass index array
 * (tianshou/data/batch.py:1209-1215: `indices = np.random.permutation(length)`, then one slice per minibatch) to the update
 * kernels; replaces the per-pass `perm.to(device)` of a host-driven loop: for
 * r in [0, repeat) a host function on an internal copy stream blocks that stream until row r is complete, then
 * host_rows[r] (pinned, the job's `out`) is copied to dev_rows[r] and an event is recorded.  ts_host_perm_feed_wait_row
 * makes `stream` wait for row r (ts_ppo_update does it before pass r when given the feed), so one asynchronous call enqueues
 * every pass of an update.  ts_host_perm_feed_finish: after the consumer's work has completed and BEFORE
 * ts_host_perm_job_finish (the host functions use the job). */
int ts_host_perm_feed_start(void* job, const int32_t* host_rows, int32_t* dev_rows, int64_t n, int32_t repeat, void** feed_out);
int ts_host_perm_feed_wait_row(void* feed, int32_t r, ts_stream_t stream);
int ts_host_perm_feed_finish(void* feed);

/* Device-side minibatch order (opt-in alternative to np.random.permutation, batch.py:1209):
 * out[r*n + i] = pi_r(i), pi_r a keyed bijection of [0,n) (cycle-walking Feistel/Philox). */
int ts_make_permutation(uint64_t seed, int32_t first_epoch, int32_t n_epochs, int64_t n,
                        int32_t* out, ts_stream_t stream);
/* int64 -> int32 narrowing of a host-drawn permutation already uploaded to the device. */
int ts_narrow_i64_i32(const int64_t* src, int64_t n, int32_t* dst, ts_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * (9) Layered networks of the off-policy algorithms (SURVEY.md 8(f) ranks 2-3): every nn.Linear / nn.Conv2d
 * forward and autograd backward inside SAC._update_with_batch (modelfree/sac.py:304-336),
 * _minimize_critic_squared_loss (modelfree/ddpg.py:267-285), DQN._update_with_batch (modelfree/dqn.py:382-404)
 * and DQNet (env/atari/atari_network.py:60-122) is ONE call of ts_net_gemm (tcgen05, fp32-faithful bf16x3):
 *
 *     C[M,N] (+)= act'(act_grad_src) * act( A[M,K] * B[N,K]^T + bias[N] )
 *
 * A / B are fp32 arrays; x_mn_major = 0: element (mn, k) at p[mn * ld + k] (k contiguous), 1: at p[k * ld + mn].
 *   forward      Y  = act(X W^T + b)   : A = X  (lda = in),  B = W  [out][in]            (0, 0)
 *   input grad   dX = (dY W) * mask    : A = dY (lda = out), B = W  as [k = out][n = in] (0, 1)
 *   weight grad  dW = dY^T X           : A = dY as [k = row][m = out] (1), B = X as [k = row][n = in] (1)
 * act_grad_src (nullable): OUTPUT y of the layer whose activation derivative multiplies the result --
 * act_grad_kind TS_ACT_RELU: * (y[m * ld_mask + n] > 0), TS_ACT_TANH: * (1 - y^2)  (back-propagation through the
 * activation of the layer that produced this GEMM's output operand).  workspace (nullable): ts_net_gemm_workspace_floats(M, N, K) floats enable split-K
 * for long reductions with few output tiles (weight gradients); partial sums are added in a fixed order. */
enum { TS_ACT_NONE = 0, TS_ACT_RELU = 1, TS_ACT_TANH = 2 };
int ts_net_gemm(const float* a, int64_t lda, int32_t a_mn_major, const float* b, int64_t ldb, int32_t b_mn_major,
                float* c, int64_t ldc, int32_t M, int32_t N, int32_t K, const float* bias, int32_t act,
                const float* act_grad_src, int64_t ld_mask, int32_t act_grad_kind, int32_t accumulate, float* workspace,
                int64_t workspace_floats, ts_stream_t stream);
int64_t ts_net_gemm_workspace_floats(int32_t M, int32_t N, int32_t K);
/* out[n] (+)= sum_m x[m * ld + n]  (bias gradients) */
int ts_net_colsum(const float* x, int64_t ld, int32_t M, int32_t N, float* out, int32_t accumulate, ts_stream_t stream);

/* PPO / A2C loss rows between the forward and backward GEMMs of a layered actor-critic (ppo.py:179-216, a2c.py:262-270):
 * head [B][A] = mu (Gaussian, sigma = exp(logstd[A])) or logits (categorical: Categorical(probs = softmax(logits)),
 * utils/net/discrete.py:69-92), value [B].  logp_out [B] always; with dhead != NULL also dhead [B][A], dvalue [B],
 * dlogstd_rows [B][A] (Gaussian, nullable), loss_rows [B][3] = (surrogate objective, value loss, entropy).
 * act: [B][A] (Gaussian) or [B] float-coded indices (categorical). */
int ts_ppo_rows(const float* head, const float* value, const float* logstd, const float* act, const float* adv,
                const float* ret, const float* logp_old, const float* v_s, int64_t B, int32_t A, int32_t categorical,
                const ts_ppo_hparams* hp, int64_t global_rows, const float* adv_moments, float* logp_out, float* dhead,
                float* dvalue, float* dlogstd_rows, float* loss_rows, ts_stream_t stream);
/* stats row (loss, actor loss, vf loss, entropy, -, rows) from loss_rows */
int ts_ppo_rows_stats(const float* loss_rows, int64_t B, const ts_ppo_hparams* hp, float* stats_row, ts_stream_t stream);

/* Frame stacking on the device (ReplayBuffer.get, data/buffer/buffer_base.py:557-603): out[i][s] for s = 0..S-1 is
 * the slot of the s-th oldest frame of the stacked observation of index[i] (out[i][S-1] = index[i], each earlier
 * one = prev() of the next, manager.py:311-336). */
int ts_stack_prev_indices(const int64_t* index, int64_t n, int32_t stack_num, const int64_t* offset, int64_t E,
                          const uint8_t* done, const int64_t* last_index, const int64_t* lengths, int64_t* out,
                          ts_stream_t stream);
/* im2col rows for nn.Conv2d(k, stride s, no padding) in torch's weight order (column = c*k*k + kh*k + kw):
 * col[(b, ho, wo)][:].  _u8: source = single uint8 frames [slot][H][W] (save_only_last_obs buffers), channel c of
 * sample b is frame stack_idx[b*C + c], values = fl32(v / denom) with the division in f64 (ScaledObsInputActionReprNet
 * divides the uint8 array by 255.0 in numpy, env/atari/atari_network.py:26-55; denom = 1 for raw values).
 * _f32: source = fp32 NHWC activations [B][H][W][C]. */
int ts_im2col_u8(const uint8_t* frames, const int64_t* stack_idx, int32_t B, int32_t C, int32_t H, int32_t W, int32_t k,
                 int32_t s, double denom, float* col, ts_stream_t stream);
int ts_im2col_f32(const float* x_nhwc, int32_t B, int32_t C, int32_t H, int32_t W, int32_t k, int32_t s, float* col,
                  ts_stream_t stream);
/* inverse of ts_im2col_f32 for gradients (gather form, deterministic); relu_src (nullable, NHWC like dx): zero
 * where relu_src <= 0 */
int ts_col2im_f32(const float* dcol, int32_t B, int32_t C, int32_t H, int32_t W, int32_t k, int32_t s,
                  const float* relu_src, float* dx_nhwc, ts_stream_t stream);
/* nn.Flatten of NCHW from NHWC activations and its backward */
int ts_nhwc_to_nchw_flat(const float* x, int32_t B, int32_t HW, int32_t C, float* y, ts_stream_t stream);
int ts_nchw_flat_to_nhwc(const float* dy, int32_t B, int32_t HW, int32_t C, const float* relu_src, float* dx, ts_stream_t stream);
/* out = concat([a, b], dim=1)  (critic input obs ++ act, utils/net/continuous.py:160-166) */
int ts_concat2(const float* a, int32_t wa, const float* b, int32_t wb, int64_t rows, float* out, ts_stream_t stream);

/* SACPolicy.forward (modelfree/sac.py:108-131) on the actor head rows head[b] = (mu[0..A) | raw log-sigma[0..A)), row
 * stride ld: sigma = exp(clamp(raw, sig_min, sig_max)), x = mu + sigma*noise, act = tanh(x), log_prob = Normal log-prob
 * summed over actions - sum log(1 - act^2 + eps) (:25-39). */
int ts_squashed_gaussian(const float* head, int64_t ld, const float* noise, int64_t B, int32_t A, float sig_min,
                         float sig_max, float eps, float* act, float* logp, float* sigma_out, ts_stream_t stream);
/* backward of mean(alpha*logp - min(q1,q2)) through the head: dact = d loss / d act from the critics (already / B);
 * dhead has the layout of head */
int ts_squashed_gaussian_bwd(const float* head, int64_t ld, const float* noise, const float* act, const float* sigma,
                             const float* dact, int64_t B, int32_t A, float sig_min, float sig_max, float eps,
                             float alpha_over_b, float* dhead, ts_stream_t stream);
/* td = q - target; loss rows td^2*w; dq = 2 td w / B   (modelfree/ddpg.py:279-284) */
int ts_critic_mse(const float* q, const float* target, const float* weight, int64_t B, float* td, float* dq, float* loss_rows,
                  ts_stream_t stream);
/* DQN loss (modelfree/dqn.py:384-399): td = returns - q[b][act[b]]; weighted MSE or Huber(delta > 0) */
int ts_dqn_loss(const float* q, const int64_t* act, const float* returns, const float* weight, int64_t B, int32_t A,
                float huber_delta, float* td, float* dq, float* loss_rows, ts_stream_t stream);
/* DQN._target_q (dqn.py:365-380): double -> q_target[b][argmax_a q_online[b][a]], else max_a q_target[b][a] */
int ts_dqn_target(const float* q_online, const float* q_target, int64_t B, int32_t A, int32_t is_double, float* out,
                  ts_stream_t stream);
/* min(q1, q2) - alpha * logp   (td3.py:94-102, sac.py:298-302).  logp == NULL means no entropy term: out = min(q1, q2),
 * TD3's target value (td3.py:94-102); alpha is then ignored. */
int ts_sac_target(const float* q1, const float* q2, const float* logp, float alpha, int64_t B, float* out, ts_stream_t stream);
/* ContinuousActorDeterministic.forward (utils/net/continuous.py:70-85) on the last Linear's output z[B][A] (row stride ld):
 * act = max_action * tanh(z).  With noise != NULL (a [B][A] standard-normal draw) TD3's target-policy smoothing
 * (td3.py:190-202): n = noise * policy_noise, clamped to [-noise_clip, noise_clip] if noise_clip > 0, act += n; the smoothed
 * action is not clamped to the action bounds, as in the reference.  act is dense [B][A]. */
int ts_det_actor_head(const float* z, int64_t ld, int64_t B, int32_t A, float max_action, const float* noise, float policy_noise,
                      float noise_clip, float* act, ts_stream_t stream);
/* backward of the head: dz = dact * max_action * (1 - tanh(z)^2), dz in the layout of z (utils/net/continuous.py:84) */
int ts_det_actor_head_bwd(const float* z, int64_t ld, const float* dact, int64_t B, int32_t A, float max_action, float* dz,
                          ts_stream_t stream);
/* DDPG / TD3 actor loss -critic(obs, actor(obs)).mean() (ddpg.py:406, td3.py:216): loss_rows = -q, dq = -1 / B */
int ts_det_actor_q_grad(const float* q, int64_t B, float* dq, float* loss_rows, ts_stream_t stream);
/* rows of alpha*logp - min(q1,q2) and d(-min)/dq / B with torch.minimum's tie rule (sac.py:315-321) */
int ts_sac_actor_q_grad(const float* q1, const float* q2, const float* logp, float alpha, int64_t B, float* dq1, float* dq2,
                        float* loss_rows, ts_stream_t stream);
int ts_mean(const float* x, int64_t n, float* out, ts_stream_t stream);
/* clip_grad_norm_ (optional) + torch.optim.Adam step on a flat parameter vector (algorithm_base.py:496-500, optim.py:89-110);
 * `step` = the 1-based step number of this call */
int ts_adam_step(float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, int64_t step, double lr,
                 double beta1, double beta2, double eps, double weight_decay, double max_grad_norm, double* norm_scratch,
                 ts_stream_t stream);
/* the same step with the step counter in DEVICE memory (*step_dev = steps taken so far; incremented by the call): no host-side
 * state in the launch, so a captured CUDA graph containing it can be replayed update after update */
int ts_adam_step_dev(float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, int64_t* step_dev, double lr,
                     double beta1, double beta2, double eps, double weight_decay, double max_grad_norm, double* norm_scratch,
                     ts_stream_t stream);
/* target = tau * source + (1 - tau) * target   (utils/lagged_network.py:8-18) */
int ts_polyak_update(float* target, const float* source, int64_t n, double tau, ts_stream_t stream);

#ifdef TS_B200_DIAGNOSTICS
/* Diagnostics build only (libts_b200_diag.so, `python -m tianshou_b200.csrc.build --diag`): not part of the product library. */
/* Hardware self-test of the tcgen05 / TMEM building blocks (csrc/umma.cuh), one CTA:
 * D[M,N] = a[M,K] * b[N,K]^T with dtype 0 = 3xTF32 (kind::tf32) or 1 = 3-way bf16 split (kind::f16),
 * M in {64,128}; a_mn / b_mn place the operand MN-major instead of K-major in shared memory; swap
 * exchanges LBO/SBO (diagnostic).  d receives the RAW accumulator: 128 TMEM lanes x N columns. */
int ts_umma_selftest(const float* a, const float* b, float* d, int32_t M, int32_t N, int32_t K,
                     int32_t dtype, int32_t a_mn, int32_t b_mn, int32_t swap, ts_stream_t stream);

/* Diagnostics: enable / read the phase timeline (32 x %globaltimer ns) that CTA 0 of the tensor-core
 * PPO step kernel records (csrc/mlp_tc.cu). */
int ts_tc_timeline(int32_t enable, uint64_t* out32 /* host, nullable */);
#endif /* TS_B200_DIAGNOSTICS */


#ifdef __cplusplus
}
#endif
#endif /* TS_B200_H_ */
