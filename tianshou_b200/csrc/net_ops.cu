// Non-GEMM pieces of the off-policy update bodies (SAC / DDPG-family critics, DQN with the NatureCNN):
// frame-stack + im2col gathers, col2im, layout permutes, loss rows with their analytic backward, Adam, Polyak.
// All HBM / latency bound elementwise or gather work: coalesced along the fastest output dimension, grid sized
// in multiples of the SM count, no atomics (every output element has one owner -> deterministic).
//
// Reference code replaced: ReplayBuffer.get frame stacking (data/buffer/buffer_base.py:557-603), DQNet conv stack
// (env/atari/atari_network.py:77-84), SACPolicy.forward tanh-squashed Gaussian (modelfree/sac.py:108-131),
// SAC actor / critic losses (sac.py:304-322, ddpg.py:279-285), the deterministic actor head of DDPG / TD3 with TD3's
// target-policy smoothing (utils/net/continuous.py:70-85, td3.py:190-202) and their actor loss (ddpg.py:406, td3.py:216), DQN loss (dqn.py:384-401), torch.optim.Adam
// single-tensor step (optim.py:89-110), polyak_parameter_update (utils/lagged_network.py:8-18).
#include <math.h>

#include "common.cuh"

namespace {

inline unsigned grid_for(int64_t n, int threads = 256) {
    int64_t b = (n + threads - 1) / threads;
    const int64_t cap = (int64_t)tsb::num_sms() * 16;
    if (b > cap) b = cap;
    if (b < 1) b = 1;
    return (unsigned)b;
}

// ---- frame stacking -------------------------------------------------------------------------------------------
// out[i][s] = prev^(S-1-s)(idx[i]): the S frames of the stacked observation, oldest first (buffer_base.py:585-600:
// stack = [..., prev(prev(i)), prev(i), i]).  Single-buffer / manager predecessor rule as in index.cu
// (manager.py:311-336): within the sub-buffer that owns i, s = (i - start - 1) mod L, e = done[s + start] |
// (s + start == last), result (s + e) mod L + start.
__global__ void stack_prev_kernel(const int64_t* __restrict__ idx, int64_t n, int S, const int64_t* __restrict__ offset, int64_t E,
                                  const uint8_t* __restrict__ done, const int64_t* __restrict__ last_index,
                                  const int64_t* __restrict__ lengths, int64_t* __restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t total = offset[E];
    int64_t cur = tsb::pymod(idx[i], total);
    const int64_t e = tsb::find_subbuffer(offset, E, cur);
    const int64_t start = offset[e];
    const int64_t L = lengths[e] > 1 ? lengths[e] : 1;
    const int64_t last = last_index[e];
    out[i * S + (S - 1)] = cur;
    for (int s = S - 2; s >= 0; --s) {
        const int64_t p = tsb::pymod(cur - start - 1, L);
        const int64_t end = (done[p + start] | (p + start == last)) ? 1 : 0;
        cur = tsb::pymod(p + end, L) + start;
        out[i * S + s] = cur;
    }
}

// ---- im2col ----------------------------------------------------------------------------------------------------
// col[(b, ho, wo)][c * k * k + kh * k + kw] = scale * x(b, c, ho * s + kh, wo * s + kw)      (torch weight order)
// U8 source: single uint8 frames [slot][H][W]; channel c of sample b is frame stack_idx[b * C + c].
__global__ void im2col_u8_kernel(const uint8_t* __restrict__ frames, const int64_t* __restrict__ stack_idx, int B, int C, int H, int W,
                                 int k, int s, int Ho, int Wo, double denom, float* __restrict__ col) {
    // value table: fl32(v / denom) with the division in f64, exactly what `obs / 255.0` (numpy, f64) followed by the cast to
    // float32 in DQNet.forward produces (atari_network.py:48-55,120)
    __shared__ float lut[256];
    for (int v = threadIdx.x; v < 256; v += blockDim.x) lut[v] = (float)((double)v / denom);
    __syncthreads();
    const int Kc = C * k * k;
    const int64_t total = (int64_t)B * Ho * Wo * Kc;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int kk = (int)(t % Kc);
        const int64_t row = t / Kc;
        const int wo = (int)(row % Wo), ho = (int)((row / Wo) % Ho), b = (int)(row / ((int64_t)Wo * Ho));
        const int c = kk / (k * k), kh = (kk / k) % k, kw = kk % k;
        const int64_t f = stack_idx[(int64_t)b * C + c];
        col[t] = lut[frames[(f * H + (ho * s + kh)) * W + (wo * s + kw)]];
    }
}
// fp32 NHWC source [B][H][W][C]
__global__ void im2col_f32_kernel(const float* __restrict__ x, int B, int C, int H, int W, int k, int s, int Ho, int Wo,
                                  float* __restrict__ col) {
    const int Kc = C * k * k;
    const int64_t total = (int64_t)B * Ho * Wo * Kc;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int kk = (int)(t % Kc);
        const int64_t row = t / Kc;
        const int wo = (int)(row % Wo), ho = (int)((row / Wo) % Ho), b = (int)(row / ((int64_t)Wo * Ho));
        const int c = kk / (k * k), kh = (kk / k) % k, kw = kk % k;
        col[t] = __ldg(x + (((int64_t)b * H + (ho * s + kh)) * W + (wo * s + kw)) * C + c);
    }
}
// dx[b][h][w][c] = (x[b][h][w][c] > 0 ? 1 : 0 if mask) * sum over the windows that cover (h, w) of dcol  -- gather form of
// col2im: one owner per input element, fixed summation order (kh, kw ascending)
__global__ void col2im_f32_kernel(const float* __restrict__ dcol, int B, int C, int H, int W, int k, int s, int Ho, int Wo,
                                  const float* __restrict__ relu_src, float* __restrict__ dx) {
    const int Kc = C * k * k;
    const int64_t total = (int64_t)B * H * W * C;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(t % C);
        const int64_t px = t / C;
        const int w = (int)(px % W), h = (int)((px / W) % H), b = (int)(px / ((int64_t)W * H));
        float acc = 0.0f;
        if (relu_src == nullptr || __ldg(relu_src + t) > 0.0f) {
            for (int kh = 0; kh < k; ++kh) {
                const int hh = h - kh;
                if (hh < 0 || hh % s != 0) continue;
                const int ho = hh / s;
                if (ho >= Ho) continue;
                for (int kw = 0; kw < k; ++kw) {
                    const int ww = w - kw;
                    if (ww < 0 || ww % s != 0) continue;
                    const int wo = ww / s;
                    if (wo >= Wo) continue;
                    acc += __ldg(dcol + (((int64_t)b * Ho + ho) * Wo + wo) * Kc + (c * k + kh) * k + kw);
                }
            }
        }
        dx[t] = acc;
    }
}
// nn.Flatten of an NCHW tensor from the NHWC activations: y[b][c * HW + p] = x[b][p][c]; backward = inverse (+ ReLU mask)
__global__ void nhwc_to_nchw_flat_kernel(const float* __restrict__ x, int B, int HW, int C, float* __restrict__ y) {
    const int64_t total = (int64_t)B * HW * C;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int p = (int)(t % HW), c = (int)((t / HW) % C);
        const int64_t b = t / ((int64_t)HW * C);
        y[t] = __ldg(x + (b * HW + p) * C + c);
    }
}
__global__ void nchw_flat_to_nhwc_kernel(const float* __restrict__ dy, int B, int HW, int C, const float* __restrict__ relu_src,
                                         float* __restrict__ dx) {
    const int64_t total = (int64_t)B * HW * C;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(t % C), p = (int)((t / C) % HW);
        const int64_t b = t / ((int64_t)HW * C);
        const float g = __ldg(dy + (b * C + c) * HW + p);
        dx[t] = (relu_src == nullptr || __ldg(relu_src + t) > 0.0f) ? g : 0.0f;
    }
}
// concat([a, b], dim=1) into a dense row-major matrix (critic input obs ++ act, utils/net/continuous.py:160-166)
__global__ void concat2_kernel(const float* __restrict__ a, int wa, const float* __restrict__ b, int wb, int64_t rows, float* __restrict__ out) {
    const int w = wa + wb;
    const int64_t total = rows * w;
    for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(t % w);
        const int64_t r = t / w;
        out[t] = c < wa ? __ldg(a + r * wa + c) : __ldg(b + r * wb + (c - wa));
    }
}

// ---- tanh-squashed Gaussian head (SACPolicy.forward, sac.py:108-131 + correct_log_prob_gaussian_tanh :25-39) -----
// head[b] = (mu[0..A), raw log-sigma[0..A)) ; sigma = exp(clamp(raw, -20, 2)) (continuous.py:231-235); x = mu + sigma * noise
// (Normal.rsample); act = tanh(x); log_prob = sum_a [ -(x - mu)^2 / (2 sigma^2) - log sigma - log sqrt(2 pi) ]
//                                             - sum_a log(1 - act^2 + eps)
__global__ void squashed_gaussian_kernel(const float* __restrict__ head, int64_t ld, const float* __restrict__ noise,
                                         int64_t B, int A, float sig_min, float sig_max, float eps, float* __restrict__ act,
                                         float* __restrict__ logp, float* __restrict__ sigma_out) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    float lp = 0.0f, corr = 0.0f;
    for (int a = 0; a < A; ++a) {
        const float m = head[b * ld + a];
        const float ls = fminf(fmaxf(head[b * ld + A + a], sig_min), sig_max);
        const float sg = expf(ls);
        const float x = fmaf(sg, noise[b * A + a], m);      // loc + eps * scale
        const float d = x - m;
        lp += -(d * d) / (2.0f * (sg * sg)) - logf(sg) - 0.9189385332046727f;
        const float t = tanhf(x);
        corr += logf(1.0f - t * t + eps);
        act[b * A + a] = t;
        if (sigma_out) sigma_out[b * A + a] = sg;
    }
    logp[b] = lp - corr;
}
// Backward of  L = mean_b( alpha * logp_b - min(q1_b, q2_b) )  w.r.t. (mu, raw log-sigma), given dq_da = d(-min(q1,q2))/d act
// already summed into `dact` by the critics' input-gradient GEMMs (scaled by 1/B) and alpha/B for the log-prob part.
// d logp / d x = 2 t (1 - t^2) / (1 - t^2 + eps)   [the Normal part cancels: x - mu = sigma * noise is constant in mu and its
// sigma-derivative cancels against the explicit one]; d logp / d sigma = -1 / sigma + noise * d logp / d x;
// d act / d x = 1 - t^2 ; d x / d mu = 1 ; d x / d sigma = noise ; d sigma / d raw = sigma inside the clamp range (inclusive).
__global__ void squashed_gaussian_bwd_kernel(const float* __restrict__ head, int64_t ld, const float* __restrict__ noise,
                                             const float* __restrict__ act, const float* __restrict__ sigma, const float* __restrict__ dact,
                                             int64_t B, int A, float sig_min, float sig_max, float eps, float alpha_over_b,
                                             float* __restrict__ dhead) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B * A) return;
    const int64_t b = t / A;
    const int a = (int)(t - b * A);
    const float tt = act[t], one_m = 1.0f - tt * tt;
    const float dlp_dx = 2.0f * tt * one_m / (one_m + eps);
    const float gx = alpha_over_b * dlp_dx + dact[t] * one_m;          // dL/dx
    const float sg = sigma[t], nz = noise[t];
    const float gsig = gx * nz - alpha_over_b / sg;
    const float r = head[b * ld + A + a];
    dhead[b * ld + a] = gx;
    dhead[b * ld + A + a] = (r >= sig_min && r <= sig_max) ? gsig * sg : 0.0f;
}

// ---- per-row losses ----------------------------------------------------------------------------------------------
// critic: td = q - target ; loss = mean(td^2 * w) ; dq = 2 td w / B          (ddpg.py:279-284)
__global__ void critic_mse_kernel(const float* __restrict__ q, const float* __restrict__ target, const float* __restrict__ weight, int64_t B,
                                  float* __restrict__ td_out, float* __restrict__ dq, float* __restrict__ loss_rows) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float td = q[b] - target[b];
    const float w = weight ? weight[b] : 1.0f;
    td_out[b] = td;
    dq[b] = 2.0f * td * w / (float)B;
    loss_rows[b] = td * td * w;
}
// DQN: q_sel = q[b][act[b]] ; td = returns - q_sel ; MSE (weighted) or Huber(delta) ; dq only at the taken action (dqn.py:384-399)
__global__ void dqn_loss_kernel(const float* __restrict__ q, const int64_t* __restrict__ act, const float* __restrict__ returns,
                                const float* __restrict__ weight, int64_t B, int A, float huber_delta, float* __restrict__ td_out,
                                float* __restrict__ dq, float* __restrict__ loss_rows) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const int a_sel = (int)act[b];
    const float qs = q[b * A + a_sel];
    const float td = returns[b] - qs;
    float lrow, g;       // g = d loss_row / d q_sel (before the 1 / B of the mean)
    if (huber_delta > 0.0f) {       // F.huber_loss(y = q, t = returns, delta), reduction mean, unweighted (dqn.py:388-394)
        const float d = qs - returns[b], ad = fabsf(d);
        if (ad < huber_delta) { lrow = 0.5f * d * d; g = d; }
        else { lrow = huber_delta * (ad - 0.5f * huber_delta); g = d > 0.0f ? huber_delta : -huber_delta; }
    } else {
        const float w = weight ? weight[b] : 1.0f;
        lrow = td * td * w;
        g = -2.0f * td * w;
    }
    td_out[b] = td;
    loss_rows[b] = lrow;
    for (int a = 0; a < A; ++a) dq[b * A + a] = a == a_sel ? g / (float)B : 0.0f;
}
// out[b] = argmax_a q[b][a] (first maximum, torch.max(dim=1)) ; val[b] = q2[b][out[b]] (double DQN) or max_a q2[b][a]
__global__ void dqn_target_kernel(const float* __restrict__ q_online, const float* __restrict__ q_target, int64_t B, int A, int is_double,
                                  float* __restrict__ out) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float* src = is_double ? q_online : q_target;
    int best = 0;
    float bv = src[b * A];
    for (int a = 1; a < A; ++a) { const float v = src[b * A + a]; if (v > bv) { bv = v; best = a; } }
    out[b] = q_target[b * A + best];
}
// SAC target: min(q1, q2) - alpha * logp   (td3.py:94-102, sac.py:298-302); logp == nullptr: min(q1, q2) alone (TD3)
__global__ void sac_target_kernel(const float* __restrict__ q1, const float* __restrict__ q2, const float* __restrict__ logp, float alpha,
                                  int64_t B, float* __restrict__ out) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    out[b] = logp ? fminf(q1[b], q2[b]) - alpha * logp[b] : fminf(q1[b], q2[b]);
}

// ---- deterministic actor head (ContinuousActorDeterministic.forward, utils/net/continuous.py:70-85) ----------------------
// act = max_action * tanh(z); with `noise` (TD3 target-policy smoothing, td3.py:190-202): n = noise * policy_noise, clamped to
// [-noise_clip, noise_clip] when noise_clip > 0, act += n.  The smoothed action is not clamped to the action bounds (nor is it
// in the reference).  One thread per element: B * A elements, row stride ld of z.
__global__ void det_actor_head_kernel(const float* __restrict__ z, int64_t ld, int64_t B, int A, float max_action,
                                      const float* __restrict__ noise, float policy_noise, float noise_clip, float* __restrict__ act) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B * A) return;
    const int64_t b = t / A;
    const int a = (int)(t - b * A);
    float y = max_action * tanhf(z[b * ld + a]);
    if (noise) {
        float n = noise[t] * policy_noise;
        if (noise_clip > 0.0f) n = fminf(fmaxf(n, -noise_clip), noise_clip);
        y += n;
    }
    act[t] = y;
}
// dz = dact * max_action * (1 - tanh(z)^2): the gradient at the last Linear's output (layout of z)
__global__ void det_actor_head_bwd_kernel(const float* __restrict__ z, int64_t ld, const float* __restrict__ dact, int64_t B, int A,
                                          float max_action, float* __restrict__ dz) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= B * A) return;
    const int64_t b = t / A;
    const int a = (int)(t - b * A);
    const float th = tanhf(z[b * ld + a]);
    dz[b * ld + a] = dact[t] * max_action * (1.0f - th * th);
}
// DDPG / TD3 actor loss -Q(s, actor(s)).mean() (ddpg.py:406, td3.py:216): loss rows -q, dq = -1 / B
__global__ void det_actor_q_grad_kernel(const float* __restrict__ q, int64_t B, float* __restrict__ dq, float* __restrict__ loss_rows) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    dq[b] = -1.0f / (float)B;
    loss_rows[b] = -q[b];
}
// d(-min(q1, q2))/d(q1, q2) / B with torch.minimum's tie rule (equal -> half each); also the actor-loss rows
__global__ void sac_actor_q_grad_kernel(const float* __restrict__ q1, const float* __restrict__ q2, const float* __restrict__ logp, float alpha,
                                        int64_t B, float* __restrict__ dq1, float* __restrict__ dq2, float* __restrict__ loss_rows) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const float a = q1[b], c = q2[b], g = -1.0f / (float)B;
    dq1[b] = a < c ? g : (a == c ? 0.5f * g : 0.0f);
    dq2[b] = c < a ? g : (a == c ? 0.5f * g : 0.0f);
    loss_rows[b] = alpha * logp[b] - fminf(a, c);
}
// mean of n values in a fixed order: one block, pairwise tree over 1024 lanes (the values are per-row loss terms)
__global__ void mean_kernel(const float* __restrict__ x, int64_t n, float* __restrict__ out) {
    __shared__ float s[1024];
    float acc = 0.0f;
    for (int64_t i = threadIdx.x; i < n; i += 1024) acc += x[i];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int off = 512; off > 0; off >>= 1) {
        if ((int)threadIdx.x < off) s[threadIdx.x] += s[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) *out = s[0] / (float)n;
}

// ---- optimiser ----------------------------------------------------------------------------------------------------
__global__ void sumsq_kernel(const float* __restrict__ g, int64_t n, double* __restrict__ partial) {
    __shared__ double s[256];
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) acc += (double)g[i] * (double)g[i];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) {
        if ((int)threadIdx.x < off) s[threadIdx.x] += s[threadIdx.x + off];
        __syncthreads();
    }
    if (threadIdx.x == 0) partial[blockIdx.x] = s[0];
}
// torch.optim.Adam single-tensor step (lerp / addcmul / addcdiv order), optional clip_grad_norm_ from `partial` block sums
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int64_t n,
                            float step_size, float bc2_sqrt, float beta1, float beta2, float eps, float wd, float max_norm,
                            const double* __restrict__ partial, int n_partial) {
    float coef = 1.0f;
    if (max_norm > 0.0f && partial) {
        double t = 0.0;
        for (int i = 0; i < n_partial; ++i) t += partial[i];
        coef = fminf(max_norm / ((float)sqrt(t) + 1e-6f), 1.0f);
    }
    const float w1 = 1.0f - beta1, w2 = 1.0f - beta2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float gi = g[i] * coef;
        float pv = p[i];
        if (wd != 0.0f) gi = fmaf(wd, pv, gi);
        float mm = m[i], vv = v[i];
        mm = mm + w1 * (gi - mm);
        vv = vv * beta2 + w2 * gi * gi;
        const float denom = sqrtf(vv) / bc2_sqrt + eps;
        pv = pv - step_size * (mm / denom);
        m[i] = mm; v[i] = vv; p[i] = pv;
    }
}
// Same step with the 1-based step number read from DEVICE memory (*step_dev + 1): the launch carries no host-side state, so a
// CUDA graph that contains it stays valid from one replay to the next.  step_inc_kernel advances the counter afterwards.
__global__ void adam_dev_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, int64_t n,
                                const int64_t* __restrict__ step_dev, double lr, double beta1d, double beta2d, float eps, float wd,
                                float max_norm, const double* __restrict__ partial, int n_partial) {
    __shared__ float s_step_size, s_bc2_sqrt, s_coef;
    if (threadIdx.x == 0) {
        const double step = (double)(*step_dev + 1);
        s_step_size = (float)(lr / (1.0 - pow(beta1d, step)));
        s_bc2_sqrt = (float)sqrt(1.0 - pow(beta2d, step));
        float coef = 1.0f;
        if (max_norm > 0.0f && partial) {
            double t = 0.0;
            for (int i = 0; i < n_partial; ++i) t += partial[i];
            coef = fminf(max_norm / ((float)sqrt(t) + 1e-6f), 1.0f);
        }
        s_coef = coef;
    }
    __syncthreads();
    const float step_size = s_step_size, bc2_sqrt = s_bc2_sqrt, coef = s_coef;
    const float beta1 = (float)beta1d, beta2 = (float)beta2d;
    const float w1 = 1.0f - beta1, w2 = 1.0f - beta2;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float gi = g[i] * coef;
        float pv = p[i];
        if (wd != 0.0f) gi = fmaf(wd, pv, gi);
        float mm = m[i], vv = v[i];
        mm = mm + w1 * (gi - mm);
        vv = vv * beta2 + w2 * gi * gi;
        const float denom = sqrtf(vv) / bc2_sqrt + eps;
        pv = pv - step_size * (mm / denom);
        m[i] = mm; v[i] = vv; p[i] = pv;
    }
}
__global__ void step_inc_kernel(int64_t* step_dev) { *step_dev += 1; }
// tgt = tau * src + (1 - tau) * tgt, each product rounded to fp32 before the add (torch evaluates two muls and an add)
__global__ void polyak_kernel(float* __restrict__ tgt, const float* __restrict__ src, int64_t n, float tau, float one_minus_tau) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        tgt[i] = __fadd_rn(__fmul_rn(tau, src[i]), __fmul_rn(one_minus_tau, tgt[i]));
}

}  // namespace

#define TS_LAUNCH_1D(kernel, n, ...)                                                            \
    do {                                                                                         \
        if ((n) > 0) kernel<<<grid_for((n)), 256, 0, tsb::as_stream(stream)>>>(__VA_ARGS__);     \
        return tsb::check_launch(#kernel);                                                       \
    } while (0)

extern "C" int ts_stack_prev_indices(const int64_t* index, int64_t n, int32_t stack_num, const int64_t* offset, int64_t E,
                                     const uint8_t* done, const int64_t* last_index, const int64_t* lengths, int64_t* out,
                                     ts_stream_t stream) {
    TS_REQUIRE(index && offset && done && last_index && lengths && out && stack_num >= 1 && E > 0, "ts_stack_prev_indices: bad argument");
    TS_LAUNCH_1D(stack_prev_kernel, n, index, n, stack_num, offset, E, done, last_index, lengths, out);
}
extern "C" int ts_im2col_u8(const uint8_t* frames, const int64_t* stack_idx, int32_t B, int32_t C, int32_t H, int32_t W, int32_t k,
                            int32_t s, double denom, float* col, ts_stream_t stream) {
    TS_REQUIRE(frames && stack_idx && col && k >= 1 && s >= 1 && H >= k && W >= k, "ts_im2col_u8: bad argument");
    const int Ho = (H - k) / s + 1, Wo = (W - k) / s + 1;
    TS_LAUNCH_1D(im2col_u8_kernel, (int64_t)B * Ho * Wo * C * k * k, frames, stack_idx, B, C, H, W, k, s, Ho, Wo, denom, col);
}
extern "C" int ts_im2col_f32(const float* x_nhwc, int32_t B, int32_t C, int32_t H, int32_t W, int32_t k, int32_t s, float* col,
                             ts_stream_t stream) {
    TS_REQUIRE(x_nhwc && col && k >= 1 && s >= 1 && H >= k && W >= k, "ts_im2col_f32: bad argument");
    const int Ho = (H - k) / s + 1, Wo = (W - k) / s + 1;
    TS_LAUNCH_1D(im2col_f32_kernel, (int64_t)B * Ho * Wo * C * k * k, x_nhwc, B, C, H, W, k, s, Ho, Wo, col);
}
extern "C" int ts_col2im_f32(const float* dcol, int32_t B, int32_t C, int32_t H, int32_t W, int32_t k, int32_t s,
                             const float* relu_src, float* dx_nhwc, ts_stream_t stream) {
    TS_REQUIRE(dcol && dx_nhwc && k >= 1 && s >= 1 && H >= k && W >= k, "ts_col2im_f32: bad argument");
    const int Ho = (H - k) / s + 1, Wo = (W - k) / s + 1;
    TS_LAUNCH_1D(col2im_f32_kernel, (int64_t)B * H * W * C, dcol, B, C, H, W, k, s, Ho, Wo, relu_src, dx_nhwc);
}
extern "C" int ts_nhwc_to_nchw_flat(const float* x, int32_t B, int32_t HW, int32_t C, float* y, ts_stream_t stream) {
    TS_REQUIRE(x && y, "ts_nhwc_to_nchw_flat: null pointer");
    TS_LAUNCH_1D(nhwc_to_nchw_flat_kernel, (int64_t)B * HW * C, x, B, HW, C, y);
}
extern "C" int ts_nchw_flat_to_nhwc(const float* dy, int32_t B, int32_t HW, int32_t C, const float* relu_src, float* dx,
                                    ts_stream_t stream) {
    TS_REQUIRE(dy && dx, "ts_nchw_flat_to_nhwc: null pointer");
    TS_LAUNCH_1D(nchw_flat_to_nhwc_kernel, (int64_t)B * HW * C, dy, B, HW, C, relu_src, dx);
}
extern "C" int ts_concat2(const float* a, int32_t wa, const float* b, int32_t wb, int64_t rows, float* out, ts_stream_t stream) {
    TS_REQUIRE(a && b && out, "ts_concat2: null pointer");
    TS_LAUNCH_1D(concat2_kernel, rows * (wa + wb), a, wa, b, wb, rows, out);
}
extern "C" int ts_squashed_gaussian(const float* head, int64_t ld, const float* noise, int64_t B, int32_t A, float sig_min,
                                    float sig_max, float eps, float* act, float* logp, float* sigma_out, ts_stream_t stream) {
    TS_REQUIRE(head && noise && act && logp && ld >= 2 * (int64_t)A, "ts_squashed_gaussian: bad argument");
    TS_LAUNCH_1D(squashed_gaussian_kernel, B, head, ld, noise, B, A, sig_min, sig_max, eps, act, logp, sigma_out);
}
extern "C" int ts_squashed_gaussian_bwd(const float* head, int64_t ld, const float* noise, const float* act, const float* sigma,
                                        const float* dact, int64_t B, int32_t A, float sig_min, float sig_max, float eps,
                                        float alpha_over_b, float* dhead, ts_stream_t stream) {
    TS_REQUIRE(head && noise && act && sigma && dact && dhead && ld >= 2 * (int64_t)A, "ts_squashed_gaussian_bwd: bad argument");
    TS_LAUNCH_1D(squashed_gaussian_bwd_kernel, B * A, head, ld, noise, act, sigma, dact, B, A, sig_min, sig_max, eps, alpha_over_b, dhead);
}
extern "C" int ts_critic_mse(const float* q, const float* target, const float* weight, int64_t B, float* td, float* dq, float* loss_rows,
                             ts_stream_t stream) {
    TS_REQUIRE(q && target && td && dq && loss_rows, "ts_critic_mse: null pointer");
    TS_LAUNCH_1D(critic_mse_kernel, B, q, target, weight, B, td, dq, loss_rows);
}
extern "C" int ts_dqn_loss(const float* q, const int64_t* act, const float* returns, const float* weight, int64_t B, int32_t A,
                           float huber_delta, float* td, float* dq, float* loss_rows, ts_stream_t stream) {
    TS_REQUIRE(q && act && returns && td && dq && loss_rows, "ts_dqn_loss: null pointer");
    TS_LAUNCH_1D(dqn_loss_kernel, B, q, act, returns, weight, B, A, huber_delta, td, dq, loss_rows);
}
extern "C" int ts_dqn_target(const float* q_online, const float* q_target, int64_t B, int32_t A, int32_t is_double, float* out,
                             ts_stream_t stream) {
    TS_REQUIRE(q_target && out && (!is_double || q_online), "ts_dqn_target: null pointer");
    TS_LAUNCH_1D(dqn_target_kernel, B, q_online, q_target, B, A, is_double, out);
}
extern "C" int ts_sac_target(const float* q1, const float* q2, const float* logp, float alpha, int64_t B, float* out, ts_stream_t stream) {
    TS_REQUIRE(q1 && q2 && out, "ts_sac_target: null pointer");
    TS_LAUNCH_1D(sac_target_kernel, B, q1, q2, logp, alpha, B, out);
}
extern "C" int ts_det_actor_head(const float* z, int64_t ld, int64_t B, int32_t A, float max_action, const float* noise,
                                 float policy_noise, float noise_clip, float* act, ts_stream_t stream) {
    TS_REQUIRE(z && act && A >= 1 && ld >= (int64_t)A, "ts_det_actor_head: bad argument");
    TS_LAUNCH_1D(det_actor_head_kernel, B * A, z, ld, B, A, max_action, noise, policy_noise, noise_clip, act);
}
extern "C" int ts_det_actor_head_bwd(const float* z, int64_t ld, const float* dact, int64_t B, int32_t A, float max_action, float* dz,
                                     ts_stream_t stream) {
    TS_REQUIRE(z && dact && dz && A >= 1 && ld >= (int64_t)A, "ts_det_actor_head_bwd: bad argument");
    TS_LAUNCH_1D(det_actor_head_bwd_kernel, B * A, z, ld, dact, B, A, max_action, dz);
}
extern "C" int ts_det_actor_q_grad(const float* q, int64_t B, float* dq, float* loss_rows, ts_stream_t stream) {
    TS_REQUIRE(q && dq && loss_rows, "ts_det_actor_q_grad: null pointer");
    TS_LAUNCH_1D(det_actor_q_grad_kernel, B, q, B, dq, loss_rows);
}
extern "C" int ts_sac_actor_q_grad(const float* q1, const float* q2, const float* logp, float alpha, int64_t B, float* dq1, float* dq2,
                                   float* loss_rows, ts_stream_t stream) {
    TS_REQUIRE(q1 && q2 && logp && dq1 && dq2 && loss_rows, "ts_sac_actor_q_grad: null pointer");
    TS_LAUNCH_1D(sac_actor_q_grad_kernel, B, q1, q2, logp, alpha, B, dq1, dq2, loss_rows);
}
extern "C" int ts_mean(const float* x, int64_t n, float* out, ts_stream_t stream) {
    TS_REQUIRE(x && out && n > 0, "ts_mean: bad argument");
    mean_kernel<<<1, 1024, 0, tsb::as_stream(stream)>>>(x, n, out);
    return tsb::check_launch("ts_mean");
}
extern "C" int ts_adam_step(float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, int64_t step, double lr,
                            double beta1, double beta2, double eps, double weight_decay, double max_grad_norm,
                            double* norm_scratch /* device double[>= 256], needed when max_grad_norm > 0 */, ts_stream_t stream) {
    TS_REQUIRE(params && grad && exp_avg && exp_avg_sq && step >= 1, "ts_adam_step: bad argument");
    if (n <= 0) return 0;
    cudaStream_t st = tsb::as_stream(stream);
    int n_partial = 0;
    if (max_grad_norm > 0.0) {
        TS_REQUIRE(norm_scratch, "ts_adam_step: clipping needs norm_scratch");
        n_partial = (int)tsb::imin((n + 255) / 256, 256);
        sumsq_kernel<<<n_partial, 256, 0, st>>>(grad, n, norm_scratch);
        if (tsb::check_launch("ts_adam_step/norm")) return 1;
    }
    const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
    adam_kernel<<<grid_for(n), 256, 0, st>>>(params, grad, exp_avg, exp_avg_sq, n, (float)(lr / bc1), (float)sqrt(bc2), (float)beta1,
                                             (float)beta2, (float)eps, (float)weight_decay, (float)max_grad_norm, norm_scratch, n_partial);
    return tsb::check_launch("ts_adam_step");
}
extern "C" int ts_adam_step_dev(float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, int64_t* step_dev, double lr,
                                double beta1, double beta2, double eps, double weight_decay, double max_grad_norm,
                                double* norm_scratch, ts_stream_t stream) {
    TS_REQUIRE(params && grad && exp_avg && exp_avg_sq && step_dev, "ts_adam_step_dev: bad argument");
    if (n <= 0) return 0;
    cudaStream_t st = tsb::as_stream(stream);
    int n_partial = 0;
    if (max_grad_norm > 0.0) {
        TS_REQUIRE(norm_scratch, "ts_adam_step_dev: clipping needs norm_scratch");
        n_partial = (int)tsb::imin((n + 255) / 256, 256);
        sumsq_kernel<<<n_partial, 256, 0, st>>>(grad, n, norm_scratch);
        if (tsb::check_launch("ts_adam_step_dev/norm")) return 1;
    }
    adam_dev_kernel<<<grid_for(n), 256, 0, st>>>(params, grad, exp_avg, exp_avg_sq, n, step_dev, lr, beta1, beta2, (float)eps,
                                                 (float)weight_decay, (float)max_grad_norm, norm_scratch, n_partial);
    if (tsb::check_launch("ts_adam_step_dev")) return 1;
    step_inc_kernel<<<1, 1, 0, st>>>(step_dev);
    return tsb::check_launch("ts_adam_step_dev/inc");
}
extern "C" int ts_polyak_update(float* target, const float* source, int64_t n, double tau, ts_stream_t stream) {
    TS_REQUIRE(target && source, "ts_polyak_update: null pointer");
    TS_LAUNCH_1D(polyak_kernel, n, target, source, n, (float)tau, (float)(1.0 - tau));
}
