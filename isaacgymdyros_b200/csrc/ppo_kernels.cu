// On-device PPO pieces around the env step (SURVEY 8f-1): the bodies of the rollout bookkeeping, GAE, the clipped
// surrogate / value loss gradient and the two Adam optimisers of the reference's rl_games fork, as sm_100a kernels.
// The two W-256-256-{13,1} MLPs stay library GEMMs (torch / cuBLAS); everything elementwise around them is here, so
// that one rollout step and one minibatch update are each a handful of launches inside a CUDA graph. W is the input width:
// the reference's 487 observation columns, or more with a height scan (DyrosPpoBuffers.obs_dim, DyrosPpoNet.inputs).
// Citations: A2C = learning/rl_games_custom/a2c_common_dyros.py, AG = learning/rl_games_custom/a2c_continuous_seperate.py,
// MD = learning/rl_games_custom/models_dyros.py, PPO = cfg/train/DyrosDynamicWalkPPO.yaml (reference tree). The loss
// formulas of rl_games 1.1.4 (common_losses.actor_loss / critic_loss, torch_ext.policy_kl; pinned by
// IsaacGymEnvs/setup.py:22, not vendored) are restated from their published definitions; oracle/ppo_oracle.py holds the
// plain-torch restatement the tests compare with.
#include <cuda_bf16.h>
#include <math.h>
#include <string.h>

#include "common.cuh"

namespace dyros {

constexpr int PPO_NA = 13, PPO_NOBS = 487;  // PPO_NOBS: the input width that obs_dim / inputs = 0 stand for
static inline int ppo_width(int w) { return w ? w : PPO_NOBS; }
static inline int ppo_padded_width(int w) { return (w + 7) & ~7; }  // K0: GEMM rows a multiple of 8 (DESIGN.md section 9)

// ---------------------------------------------------------------- rollout: act + record (A2C:629-647, MD:28-58)
// One warp per env. Samples a = mu + sigma * N(0,1) (Philox, counter = (env, global step)), its negative log
// likelihood (MD:60-63), and records obs / done / mu / value / action / neglogp at slot n = *step of the env-major
// rollout buffers, (N, H, .): a minibatch of the update is then a contiguous block of rows, as rl_games' dataset slices
// of the swap_and_flatten01 layout are (A2C:703, 32 envs x 128 steps for the reference's sizes).
__global__ void __launch_bounds__(256) k_ppo_act(DyrosPpoBuffers b, const float* __restrict__ mu, const float* __restrict__ value,
                                                 const float* __restrict__ logstd, const float* __restrict__ obs,
                                                 const long long* __restrict__ reset_buf, float* __restrict__ actions_env,
                                                 const float* __restrict__ inject_normal, int W) {
  const int lane = threadIdx.x & 31, e = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (e >= b.N) return;
  const int n = *b.step;
  const size_t row = (size_t)e * b.H + n;
  float a = 0.f, z = 0.f, m = 0.f, ls = 0.f;
  if (lane < PPO_NA) {
    m = mu[(size_t)e * PPO_NA + lane];
    ls = logstd[lane];
    if (inject_normal) z = inject_normal[((size_t)n * b.N + e) * PPO_NA + lane];
    else {
      const uint4 r = draw4(b.seed, *b.global_step, e, 7u /* policy site */, lane >> 1);
      const float2 nn = normal01_pair(r.x, r.y);
      z = (lane & 1) ? nn.y : nn.x;
    }
    a = m + expf(ls) * z;  // torch.distributions.Normal(mu, sigma).sample(), MD:46-47
  }
  // neglogp = 0.5 * sum(((a - mu) / sigma)^2) + 0.5 * log(2 pi) * 13 + sum(logstd), MD:60-63
  float t = 0.f;
  if (lane < PPO_NA) {
    const float d = (a - m) / expf(ls);
    t = 0.5f * d * d + ls;
  }
  t = warp_sum(t) + 0.5f * 1.8378770664093453f * (float)PPO_NA;
  if (lane < PPO_NA) {
    b.actions[row * PPO_NA + lane] = a;
    b.mus[row * PPO_NA + lane] = m;
    actions_env[(size_t)e * PPO_NA + lane] = a;  // the env clamps to [-1, 1] itself (VT:307; A2C:820-824 rescale = identity)
  }
  if (lane == 0) {
    b.neglogp[row] = t;
    b.values[row] = value[e];
    b.dones[row] = reset_buf[e] != 0 ? 1.f : 0.f;  // self.dones BEFORE the step (A2C:640)
  }
  const float* src = obs + (size_t)e * W;
  float* dst = b.obs + row * W;
  for (int i = lane; i < W; i += 32) dst[i] = src[i];
}

// after the env step: shaped reward with the time-out bootstrap (A2C:654-661), episode statistics (A2C:663-684)
__global__ void __launch_bounds__(256) k_ppo_reward(DyrosPpoBuffers b, const float* __restrict__ rew, const long long* __restrict__ timeout,
                                                    const long long* __restrict__ reset_buf) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = *b.step;
  if (e < b.N) {
    const size_t row = (size_t)e * b.H + n;
    float r = rew[e] * b.reward_scale;
    if (b.value_bootstrap && timeout[e] != 0) r += b.gamma * b.values[row];
    b.rewards[row] = r;
    const float cr = b.cur_reward[e] + rew[e], cl = b.cur_length[e] + 1.f;
    const bool done = reset_buf[e] != 0;
    if (done) {  // finished episodes feed the running means (game_rewards / game_lengths)
      atomicAdd(b.ep_stats + 0, cr);
      atomicAdd(b.ep_stats + 1, cl);
      atomicAdd(b.ep_stats + 2, 1.f);
    }
    b.cur_reward[e] = done ? 0.f : cr;
    b.cur_length[e] = done ? 0.f : cl;
  }
}
__global__ void k_ppo_advance(DyrosPpoBuffers b) {
  *b.step = (*b.step + 1) % b.H;
  *b.global_step = *b.global_step + 1;
}

// ---------------------------------------------------------------- GAE (A2C:485-500) + returns (A2C:692)
// One thread per env, walking its contiguous (H) rows backwards.
__global__ void __launch_bounds__(128) k_ppo_gae(DyrosPpoBuffers b, const float* __restrict__ last_values,
                                                 const long long* __restrict__ last_reset) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= b.N) return;
  const size_t r0 = (size_t)e * b.H;
  float lastgaelam = 0.f;
  float nextvalue = last_values[e];
  float nextnonterminal = 1.f - (last_reset[e] != 0 ? 1.f : 0.f);
  for (int t = b.H - 1; t >= 0; --t) {
    const float v = b.values[r0 + t];
    const float delta = b.rewards[r0 + t] + b.gamma * nextvalue * nextnonterminal - v;
    lastgaelam = delta + b.gamma * b.tau * nextnonterminal * lastgaelam;
    b.advantages[r0 + t] = lastgaelam;
    b.returns[r0 + t] = lastgaelam + v;
    nextvalue = v;
    nextnonterminal = 1.f - b.dones[r0 + t];
  }
}

// ---------------------------------------------------------------- loss gradient of one minibatch (AG:108-160)
// For rows [row0, row0 + mb): given the networks' outputs mu (mb,13) and value (mb), writes dLoss/dmu and dLoss/dvalue
// of  loss = mean(max(-A r, -A clip(r, 1-e, 1+e))) + 0.5 * critic_coef * mean((ret - v)^2)   (entropy and bound
// coefficients are 0 in PPO:80-92; sigma is a fixed, non-trainable parameter, network_builder_dyros.py:103) with
// r = exp(old_neglogp - neglogp(a | mu, sigma)), and accumulates the logged sums: actor loss, critic loss, KL
// (torch_ext.policy_kl), clip fraction. One warp per row.
__global__ void __launch_bounds__(256) k_ppo_loss_grad(DyrosPpoBuffers b, int row0, int mb, const float* __restrict__ mu,
                                                       const float* __restrict__ value, const float* __restrict__ logstd,
                                                       const float* __restrict__ adv_norm, float* __restrict__ dmu,
                                                       float* __restrict__ dvalue, float* __restrict__ stats) {
  __shared__ float acc[4][8];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int i = blockIdx.x * 8 + w;
  float s_a = 0.f, s_c = 0.f, s_kl = 0.f, s_cf = 0.f;
  if (i < mb) {
    const size_t row = (size_t)row0 + i;
    float m = 0.f, a = 0.f, ls = 0.f, om = 0.f, inv_s = 0.f;
    if (lane < PPO_NA) {
      m = mu[(size_t)i * PPO_NA + lane];
      a = b.actions[row * PPO_NA + lane];
      om = b.mus[row * PPO_NA + lane];
      ls = logstd[lane];
      inv_s = expf(-ls);
    }
    const float d = (a - m) * inv_s;
    float t = lane < PPO_NA ? 0.5f * d * d + ls : 0.f;
    const float neglogp = warp_sum(t) + 0.5f * 1.8378770664093453f * (float)PPO_NA;
    const float A = adv_norm[row];
    const float ratio = expf(b.neglogp[row] - neglogp);
    const float lo = 1.f - b.e_clip, hi = 1.f + b.e_clip;
    const float rc = fminf(fmaxf(ratio, lo), hi);
    const float l1 = -A * ratio, l2 = -A * rc;
    // d max(l1, l2) / d ratio: -A on the unclipped branch, -A * 1[lo < ratio < hi] on the clipped one
    const bool first = l1 >= l2;
    const float dl_dratio = first ? -A : ((ratio > lo && ratio < hi) ? -A : 0.f);
    // d ratio / d mu_k = ratio * (a_k - mu_k) / sigma_k^2
    const float inv_mb = 1.f / (float)mb;
    if (lane < PPO_NA) dmu[(size_t)i * PPO_NA + lane] = dl_dratio * ratio * d * inv_s * inv_mb;
    const float v = value[i], ret = b.returns[row];
    if (lane == 0) dvalue[i] = 0.5f * b.critic_coef * 2.f * (v - ret) * inv_mb;
    // KL(new || old) as torch_ext.policy_kl(p0 = new, p1 = old): sigma is shared, so c1 + c3 = log(1 + 1e-5) - 0.5
    float kl = 0.f;
    if (lane < PPO_NA) {
      const float s2 = expf(2.f * ls);
      kl = logf(1.f + 1e-5f) + (s2 + (om - m) * (om - m)) / (2.f * (s2 + 1e-5f)) - 0.5f;
    }
    s_kl = warp_sum(kl);
    s_a = fmaxf(l1, l2);
    s_c = (ret - v) * (ret - v);
    s_cf = fabsf(ratio - 1.f) > b.e_clip ? 1.f : 0.f;
  }
  if (lane == 0) {
    acc[0][w] = s_a; acc[1][w] = s_c; acc[2][w] = s_kl; acc[3][w] = s_cf;
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    float s = 0.f;
    for (int k = 0; k < 8; ++k) s += acc[threadIdx.x][k];
    atomicAdd(stats + threadIdx.x, s / (float)mb);
  }
}

// ---------------------------------------------------------------- the two Adam optimisers in one pass (AG:50-54, AG:164-187)
// Flat parameter / gradient / moment buffers: [0, n_actor) = actor (clip_grad_norm_(actor_param, grad_norm), AG:179),
// [n_actor, n) = critic (not clipped). grads are SUMS over ranks: grad_scale = 1 / world averages them (the reference's
// Horovod DistributedOptimizer averages, AG:161-163). lr and the step count live on the device (graph replays).
__global__ void __launch_bounds__(256) k_ppo_gradnorm(const float* __restrict__ g, int n_actor, float grad_scale, float* __restrict__ norm2) {
  float s = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_actor; i += gridDim.x * blockDim.x) {
    const float x = g[i] * grad_scale;
    s += x * x;
  }
  s = warp_sum(s);
  __shared__ float part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int k = 0; k < 8; ++k) t += part[k];
    atomicAdd(norm2, t);
  }
}
__global__ void __launch_bounds__(256) k_ppo_adam(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                  float* __restrict__ v, int n_actor, int n, float grad_scale, float max_norm,
                                                  float* __restrict__ norm2, const float* __restrict__ lr_dev, int* __restrict__ t_dev,
                                                  float beta1, float beta2, float eps) {
  const int t = *t_dev + 1;
  const float lr_actor = lr_dev[0], lr_critic = lr_dev[1];  // AG:53-54: the critic's rate is fixed, the actor's is scheduled
  const float norm = sqrtf(*norm2);
  const float clip = fminf(max_norm / (norm + 1e-6f), 1.f);  // torch.nn.utils.clip_grad_norm_
  const float bc1 = 1.f - powf(beta1, (float)t), bc2 = 1.f - powf(beta2, (float)t);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    float gi = g[i] * grad_scale;
    if (i < n_actor && max_norm > 0.f) gi *= clip;
    const float mi = beta1 * m[i] + (1.f - beta1) * gi;
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    p[i] -= (i < n_actor ? lr_actor : lr_critic) * (mi / bc1) / (sqrtf(vi / bc2) + eps);  // torch.optim.Adam, amsgrad off, weight_decay 0
  }
}
// ... and rl_games' LinearScheduler, which the reference steps once per MINIBATCH (schedule_type 'legacy', A2C:888-892;
// max_steps = max_epochs, A2C:135-137): lr = min_lr + (lr0 - min_lr) * max(0, max_steps - steps) / max_steps
__global__ void k_ppo_adam_finish(float* norm2, int* t_dev, float* lr_dev, float lr0, float lr_min, int max_steps) {
  *norm2 = 0.f;
  const int t = *t_dev + 1;
  *t_dev = t;
  if (max_steps > 0) {
    const int left = max_steps - t > 0 ? max_steps - t : 0;
    lr_dev[0] = lr_min + (lr0 - lr_min) * ((float)left / (float)max_steps);
  }
}


// ================================================================ packed bf16 path (DESIGN.md section 9, "update v2")
// The two MLPs as ONE batch-2 problem in GEMM layout (net 0 = actor, net 1 = critic): W0 [2][H][K0] (W inputs padded
// to K0, a multiple of 8: cuBLAS falls back to its slow align-1 kernels for an odd leading dimension), W1 [2][H][H],
// Wh [2][16][H] (13 / 1 rows used, the rest stay zero), bf16, biases fp32. The 8 GEMMs of a minibatch (3 forward, 5
// backward) are batched library calls; everything between them is here: 5 kernels instead of ~60 framework launches
// (casts, bias adds, ReLU masks, bf16 column sums for the bias gradients).
constexpr int PPO_HEAD = 16;
typedef __nv_bfloat16 bf16;
__device__ __forceinline__ float bf2f(bf16 x) { return __bfloat162float(x); }

// obs (N,W) fp32 -> bf16 rows of width K0 (columns W..K0-1 zero): the policy's input of this step and, when x_roll is
// given, the same row at slot *step of the env-major rollout store (row e*H + n). One warp per env; lane i of a pass
// reads the pair 2i, 2i+1, so a warp's loads cover 64 consecutive floats of the row.
__global__ void __launch_bounds__(256) k_ppo_cast_obs(const float* __restrict__ obs, int N, int W, int K0, bf16* __restrict__ x_step,
                                                      bf16* __restrict__ x_roll, const int* __restrict__ step, int H) {
  const int lane = threadIdx.x & 31, e = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (e >= N) return;
  const float* src = obs + (size_t)e * W;
  __nv_bfloat162* a = reinterpret_cast<__nv_bfloat162*>(x_step + (size_t)e * K0);
  __nv_bfloat162* r = x_roll ? reinterpret_cast<__nv_bfloat162*>(x_roll + ((size_t)e * H + *step) * K0) : nullptr;
  for (int i = lane; i < K0 / 2; i += 32) {
    const float lo = 2 * i < W ? src[2 * i] : 0.f, hi = 2 * i + 1 < W ? src[2 * i + 1] : 0.f;
    const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    a[i] = v;
    if (r) r[i] = v;
  }
}

// t[net][row][c] = relu(t + bias[net][c]) in place; 8 columns per thread
__global__ void __launch_bounds__(256) k_ppo_bias_relu(bf16* __restrict__ t, const float* __restrict__ bias, int rows, int hidden) {
  const size_t per_net = (size_t)rows * hidden, total8 = 2 * per_net / 8;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total8; i += (size_t)gridDim.x * blockDim.x) {
    const size_t el = i * 8;
    const int net = el >= per_net, c = (int)(el % hidden);
    uint4 raw = *reinterpret_cast<const uint4*>(t + el);
    bf16* v = reinterpret_cast<bf16*>(&raw);
    const float* bb = bias + net * hidden + c;
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = __float2bfloat16(fmaxf(bf2f(v[k]) + bb[k], 0.f));
    *reinterpret_cast<uint4*>(t + el) = raw;
  }
}

// g[net][row][c] = h > 0 ? g : 0 in place, and gbias[net][c] += sum over rows of the masked g (fp32).
// Block = 32 column groups of 8 x 8 row lanes over a tile of kRbRows rows of one net and 256 columns; a thread's
// kRbRows / 8 rows are loaded up front (independent 16-byte loads in flight), reduced over the row lanes in shared
// memory, one atomicAdd per column and block.
constexpr int kRbRows = 64;
__global__ void __launch_bounds__(256) k_ppo_relu_bwd(bf16* __restrict__ g, const bf16* __restrict__ h, float* __restrict__ gbias,
                                                      int rows, int hidden) {
  __shared__ float part[8][33 * 8];
  constexpr int kPer = kRbRows / 8;
  const int tiles = (rows + kRbRows - 1) / kRbRows, cblocks = (hidden + 255) / 256;
  const int net = blockIdx.x / (tiles * cblocks), rest = blockIdx.x % (tiles * cblocks);
  const int tile = rest / cblocks, c = (rest % cblocks) * 256 + (threadIdx.x & 31) * 8;
  const int cg = threadIdx.x & 31, rl = threadIdx.x >> 5;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  if (c < hidden) {
    uint4 gr[kPer], hr[kPer];
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
      const int r = tile * kRbRows + rl + 8 * q;
      if (r < rows) {
        const size_t el = ((size_t)net * rows + r) * hidden + c;
        gr[q] = *reinterpret_cast<const uint4*>(g + el);
        hr[q] = *reinterpret_cast<const uint4*>(h + el);
      }
    }
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
      const int r = tile * kRbRows + rl + 8 * q;
      if (r < rows) {
        bf16* gv = reinterpret_cast<bf16*>(&gr[q]);
        const bf16* hv = reinterpret_cast<const bf16*>(&hr[q]);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float x = bf2f(hv[k]) > 0.f ? bf2f(gv[k]) : 0.f;
          gv[k] = __float2bfloat16(x);
          acc[k] += x;
        }
        *reinterpret_cast<uint4*>(g + ((size_t)net * rows + r) * hidden + c) = gr[q];
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 8; ++k) part[rl][cg * 8 + k + cg / 4] = acc[k];  // (+cg/4: spreads the banks)
  __syncthreads();
  if (rl == 0 && c < hidden) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float s = 0.f;
#pragma unroll
      for (int q = 0; q < 8; ++q) s += part[q][cg * 8 + k + cg / 4];
      atomicAdd(gbias + net * hidden + c + k, s);
    }
  }
}

// k_ppo_act on the packed head output: out [2][N][16] bf16 (GEMM result without bias), bh [2][16]. Does not store obs
// (k_ppo_cast_obs keeps the bf16 rows).
__global__ void __launch_bounds__(256) k_ppo_act_packed(DyrosPpoBuffers b, const bf16* __restrict__ out, const float* __restrict__ bh,
                                                        const float* __restrict__ logstd, const long long* __restrict__ reset_buf,
                                                        float* __restrict__ actions_env, const float* __restrict__ inject_normal) {
  const int lane = threadIdx.x & 31, e = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (e >= b.N) return;
  const int n = *b.step;
  const size_t row = (size_t)e * b.H + n;
  float a = 0.f, z = 0.f, m = 0.f, ls = 0.f;
  if (lane < PPO_NA) {
    m = bf2f(out[(size_t)e * PPO_HEAD + lane]) + bh[lane];
    ls = logstd[lane];
    if (inject_normal) z = inject_normal[((size_t)n * b.N + e) * PPO_NA + lane];
    else {
      const uint4 r = draw4(b.seed, *b.global_step, e, 7u /* policy site */, lane >> 1);
      const float2 nn = normal01_pair(r.x, r.y);
      z = (lane & 1) ? nn.y : nn.x;
    }
    a = m + expf(ls) * z;
  }
  float t = 0.f;
  if (lane < PPO_NA) {
    const float d = (a - m) / expf(ls);
    t = 0.5f * d * d + ls;
  }
  t = warp_sum(t) + 0.5f * 1.8378770664093453f * (float)PPO_NA;
  if (lane < PPO_NA) {
    b.actions[row * PPO_NA + lane] = a;
    b.mus[row * PPO_NA + lane] = m;
    actions_env[(size_t)e * PPO_NA + lane] = a;
  }
  if (lane == 0) {
    b.neglogp[row] = t;
    b.values[row] = bf2f(out[((size_t)b.N + e) * PPO_HEAD]) + bh[PPO_HEAD];
    b.dones[row] = reset_buf[e] != 0 ? 1.f : 0.f;
  }
}

// k_ppo_loss_grad on the packed head output of a minibatch: writes d loss / d out [2][mb][16] in bf16 (zeros in the unused
// columns), accumulates the head's bias gradients gbh [2][16] (fp32), refreshes the stored old mu of the rows
// (dataset.update_mu_sigma, A2C:884) and the logged sums. One warp per row.
__global__ void __launch_bounds__(256) k_ppo_loss_grad_packed(DyrosPpoBuffers b, int row0, int mb, const bf16* __restrict__ out,
                                                              const float* __restrict__ bh, const float* __restrict__ logstd,
                                                              const float* __restrict__ adv_norm, bf16* __restrict__ dout,
                                                              float* __restrict__ gbh, float* __restrict__ stats) {
  __shared__ float acc[4][8];
  __shared__ float gb[8][PPO_NA + 1];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int i = blockIdx.x * 8 + w;
  float s_a = 0.f, s_c = 0.f, s_kl = 0.f, s_cf = 0.f, g_mu = 0.f, g_v = 0.f;
  if (i < mb) {
    const size_t row = (size_t)row0 + i;
    float m = 0.f, a = 0.f, ls = 0.f, om = 0.f, inv_s = 0.f;
    if (lane < PPO_NA) {
      m = bf2f(out[(size_t)i * PPO_HEAD + lane]) + bh[lane];
      a = b.actions[row * PPO_NA + lane];
      om = b.mus[row * PPO_NA + lane];
      ls = logstd[lane];
      inv_s = expf(-ls);
    }
    const float d = (a - m) * inv_s;
    float t = lane < PPO_NA ? 0.5f * d * d + ls : 0.f;
    const float neglogp = warp_sum(t) + 0.5f * 1.8378770664093453f * (float)PPO_NA;
    const float A = adv_norm[row];
    const float ratio = expf(b.neglogp[row] - neglogp);
    const float lo = 1.f - b.e_clip, hi = 1.f + b.e_clip;
    const float rc = fminf(fmaxf(ratio, lo), hi);
    const float l1 = -A * ratio, l2 = -A * rc;
    const bool first = l1 >= l2;
    const float dl_dratio = first ? -A : ((ratio > lo && ratio < hi) ? -A : 0.f);
    const float inv_mb = 1.f / (float)mb;
    if (lane < PPO_NA) g_mu = dl_dratio * ratio * d * inv_s * inv_mb;
    const float v = bf2f(out[((size_t)mb + i) * PPO_HEAD]) + bh[PPO_HEAD], ret = b.returns[row];
    g_v = 0.5f * b.critic_coef * 2.f * (v - ret) * inv_mb;
    if (lane < PPO_HEAD) {
      dout[(size_t)i * PPO_HEAD + lane] = __float2bfloat16(lane < PPO_NA ? g_mu : 0.f);
      dout[((size_t)mb + i) * PPO_HEAD + lane] = __float2bfloat16(lane == 0 ? g_v : 0.f);
    }
    float kl = 0.f;
    if (lane < PPO_NA) {
      const float s2 = expf(2.f * ls);
      kl = logf(1.f + 1e-5f) + (s2 + (om - m) * (om - m)) / (2.f * (s2 + 1e-5f)) - 0.5f;
      b.mus[row * PPO_NA + lane] = m;
    }
    s_kl = warp_sum(kl);
    s_a = fmaxf(l1, l2);
    s_c = (ret - v) * (ret - v);
    s_cf = fabsf(ratio - 1.f) > b.e_clip ? 1.f : 0.f;
  }
  if (lane == 0) {
    acc[0][w] = s_a; acc[1][w] = s_c; acc[2][w] = s_kl; acc[3][w] = s_cf;
    gb[w][PPO_NA] = g_v;
  }
  if (lane < PPO_NA) gb[w][lane] = g_mu;
  __syncthreads();
  if (threadIdx.x < 4) {
    float s = 0.f;
    for (int k = 0; k < 8; ++k) s += acc[threadIdx.x][k];
    atomicAdd(stats + threadIdx.x, s / (float)mb);
  }
  if (threadIdx.x >= 32 && threadIdx.x < 32 + PPO_NA + 1) {
    const int c = threadIdx.x - 32;
    float s = 0.f;
    for (int k = 0; k < 8; ++k) s += gb[k][c];
    atomicAdd(gbh + (c < PPO_NA ? c : PPO_HEAD), s);  // actor columns 0..12, critic column 0 of net 1
  }
}

// master layout of the flat fp32 buffers (ppo.py FlatActorCritic): per net [W0 (H x W), b0 (H), W1 (H x H), b1 (H),
// Wh (nout x H), bh (nout)], actor (nout 13, W = Wa) then critic (nout 1, W = Wc >= Wa: an asymmetric critic reads a
// wider row). Both W0 blocks share one leading dimension K0 = round_up(Wc, 8). The kernels below visit the master
// block's rows x cols only, so the columns Wa..K0-1 of the actor's packed W0 and Wc..K0-1 of the critic's are never
// written and stay zero: the actor is blind to the columns past its own.
struct PpoSeg {
  int master_off, rows, cols;  // the master block
  int dst_cols;                // leading dimension of the packed matrix (0: a bias vector)
  int which;                   // 0 w0, 1 b0, 2 w1, 3 b1, 4 wh, 5 bh
  int net;
};
struct PpoSegs {
  PpoSeg s[12];
};
static PpoSegs ppo_segments(int hidden, int Wa, int Wc) {
  PpoSegs S;
  int off = 0, k = 0;
  for (int net = 0; net < 2; ++net) {
    const int nout = net == 0 ? PPO_NA : 1, W = net == 0 ? Wa : Wc;
    S.s[k++] = PpoSeg{off, hidden, W, ppo_padded_width(Wc), 0, net}; off += hidden * W;
    S.s[k++] = PpoSeg{off, 1, hidden, 0, 1, net}; off += hidden;
    S.s[k++] = PpoSeg{off, hidden, hidden, hidden, 2, net}; off += hidden * hidden;
    S.s[k++] = PpoSeg{off, 1, hidden, 0, 3, net}; off += hidden;
    S.s[k++] = PpoSeg{off, nout, hidden, hidden, 4, net}; off += nout * hidden;
    S.s[k++] = PpoSeg{off, 1, nout, 0, 5, net}; off += nout;
  }
  return S;
}
__device__ __forceinline__ size_t ppo_packed_index(const PpoSeg& g, int hidden, int r, int c) {
  switch (g.which) {
    case 0: return ((size_t)g.net * hidden + r) * g.dst_cols + c;
    case 2: return ((size_t)g.net * hidden + r) * hidden + c;
    case 4: return ((size_t)g.net * PPO_HEAD + r) * hidden + c;
    case 5: return (size_t)g.net * PPO_HEAD + c;
    default: return (size_t)g.net * hidden + c;  // b0, b1
  }
}
// flat fp32 master parameters -> packed bf16 weights + fp32 biases. blockIdx.y = segment.
__global__ void __launch_bounds__(256) k_ppo_pack(PpoSegs S, DyrosPpoNet net, const float* __restrict__ flat) {
  const PpoSeg g = S.s[blockIdx.y];
  const int n = g.rows * g.cols;
  bf16* wdst = reinterpret_cast<bf16*>(g.which == 0 ? net.w0 : (g.which == 2 ? net.w1 : net.wh));
  float* bdst = g.which == 1 ? net.b0 : (g.which == 3 ? net.b1 : net.bh);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int r = i / g.cols, c = i % g.cols;
    const float x = flat[g.master_off + i];
    const size_t d = ppo_packed_index(g, net.hidden, r, c);
    if (g.dst_cols) wdst[d] = __float2bfloat16(x);
    else bdst[d] = x;
  }
}
// packed gradients (bf16 GEMM outputs, fp32 bias accumulators) -> flat fp32 master gradient; zeroes the accumulators
// norm2 (optional): += sum of squares of the actor's gradients (net 0), i.e. k_ppo_gradnorm folded in (single rank: no
// all-reduce sits between the two)
// epoch (optional): flat_grad points at TWO buffers of `stride` floats, the one of parity *epoch & 1 is written (the
// peer-memory exchange below)
__global__ void __launch_bounds__(256) k_ppo_unpack(PpoSegs S, DyrosPpoNet net, float* __restrict__ flat_grad, float* __restrict__ norm2,
                                                    const unsigned* __restrict__ epoch, size_t stride) {
  const PpoSeg g = S.s[blockIdx.y];
  if (epoch) flat_grad += (size_t)(*epoch & 1u) * stride;
  float sq = 0.f;
  const int n = g.rows * g.cols;
  const bf16* wsrc = reinterpret_cast<const bf16*>(g.which == 0 ? net.gw0 : (g.which == 2 ? net.gw1 : net.gwh));
  float* bsrc = g.which == 1 ? net.gb0 : (g.which == 3 ? net.gb1 : net.gbh);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int r = i / g.cols, c = i % g.cols;
    const size_t d = ppo_packed_index(g, net.hidden, r, c);
    float x;
    if (g.dst_cols) x = bf2f(wsrc[d]);
    else {
      x = bsrc[d];
      bsrc[d] = 0.f;
    }
    flat_grad[g.master_off + i] = x;
    sq += x * x;
  }
  if (norm2 && g.net == 0) {  // (uniform per block: blockIdx.y picks the segment)
    sq = warp_sum(sq);
    __shared__ float part[8];
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = sq;
    __syncthreads();
    if (threadIdx.x == 0) {
      float t = 0.f;
      for (int k = 0; k < 8; ++k) t += part[k];
      atomicAdd(norm2, t);
    }
  }
}
// k_ppo_adam per segment of the master layout, writing the packed bf16 / fp32 copy of every updated parameter as well
// (k_ppo_pack folded in)
__global__ void __launch_bounds__(256) k_ppo_adam_pack(PpoSegs S, DyrosPpoNet net, float* __restrict__ p, const float* __restrict__ gr,
                                                       float* __restrict__ m, float* __restrict__ v, float grad_scale, float max_norm,
                                                       const float* __restrict__ norm2, const float* __restrict__ lr_dev,
                                                       const int* __restrict__ t_dev, float beta1, float beta2, float eps) {
  const PpoSeg g = S.s[blockIdx.y];
  const int n = g.rows * g.cols;
  const int t = *t_dev + 1;
  const bool actor = g.net == 0;
  const float lr = lr_dev[actor ? 0 : 1];
  const float clip = actor && max_norm > 0.f ? fminf(max_norm / (sqrtf(*norm2) * grad_scale + 1e-6f), 1.f) : 1.f;
  const float bc1 = 1.f - powf(beta1, (float)t), bc2 = 1.f - powf(beta2, (float)t);
  bf16* wdst = reinterpret_cast<bf16*>(g.which == 0 ? net.w0 : (g.which == 2 ? net.w1 : net.wh));
  float* bdst = g.which == 1 ? net.b0 : (g.which == 3 ? net.b1 : net.bh);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int j = g.master_off + i;
    const float gi = gr[j] * grad_scale * clip;
    const float mi = beta1 * m[j] + (1.f - beta1) * gi;
    const float vi = beta2 * v[j] + (1.f - beta2) * gi * gi;
    m[j] = mi;
    v[j] = vi;
    const float x = p[j] - lr * (mi / bc1) / (sqrtf(vi / bc2) + eps);
    p[j] = x;
    const size_t d = ppo_packed_index(g, net.hidden, i / g.cols, i % g.cols);
    if (g.dst_cols) wdst[d] = __float2bfloat16(x);
    else bdst[d] = x;
  }
}

// ================================================================ gradient exchange over peer memory (NVLink / NVSwitch)
// What the reference does with Horovod's all-reduce between backward and optimizer.step (AG:161-173), as part of the
// optimiser's own kernels: every rank's flat gradient buffer is mapped into every other rank (CUDA IPC), a rank
// publishes "minibatch e written" in its peers' flag words (st.release.sys), waits for the same word from everybody
// (ld.acquire.sys) and then sums all ranks' buffers itself, reading the remote ones through NVLink, in rank order
// (so every rank forms bit-identical sums), folding in the squared norm for the actor's clip. Two buffers per rank,
// alternating with the minibatch counter: a rank can be at most one minibatch ahead of the slowest one, so the buffer
// it overwrites is never one a peer still reads (DESIGN.md section 9).
__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
  unsigned v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_cg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__global__ void __launch_bounds__(256) k_ppo_reduce_peers(DyrosPpoPeers P, float* __restrict__ out, int n, int n_actor,
                                                          float* __restrict__ norm2, unsigned* __restrict__ ticket) {
  const unsigned e = *P.epoch;  // minibatches finished so far; this one publishes e + 1
  const int par = (int)(e & 1u);
  if (blockIdx.x == 0 && (int)threadIdx.x < P.world) {
    __threadfence_system();
    st_release_sys(P.flags[threadIdx.x] + P.rank, e + 1u);
  }
  if ((int)threadIdx.x < P.world) {
    // (a rank that never arrives -- a crashed peer -- must not hang the device for ever: after 20 s the kernel traps and
    // the next CUDA call of the host reports it)
    unsigned long long t0 = 0, now = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (ld_acquire_sys(P.flags[P.rank] + threadIdx.x) < e + 1u) {
      __nanosleep(64);
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (now - t0 > 20000000000ull) __trap();
    }
  }
  __syncthreads();
  float sq = 0.f;
  const int n4 = n / 4;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
    float4 x[8];
#pragma unroll
    for (int r = 0; r < 8; ++r)  // all ranks' loads in flight before the first add (remote ones cross NVLink)
      if (r < P.world) x[r] = ld_cg4(P.grad[r][par] + 4 * i);
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < 8; ++r)
      if (r < P.world) {
        s.x += x[r].x; s.y += x[r].y; s.z += x[r].z; s.w += x[r].w;
      }
    reinterpret_cast<float4*>(out)[i] = s;
    const int j = 4 * i;
    if (j + 3 < n_actor) sq += s.x * s.x + s.y * s.y + s.z * s.z + s.w * s.w;
    else {
      if (j < n_actor) sq += s.x * s.x;
      if (j + 1 < n_actor) sq += s.y * s.y;
      if (j + 2 < n_actor) sq += s.z * s.z;
    }
  }
  if (blockIdx.x == 0 && (int)threadIdx.x < n - 4 * n4) {  // the tail (n is not a multiple of 4)
    const int j = 4 * n4 + threadIdx.x;
    float s = 0.f;
    for (int r = 0; r < P.world; ++r) s += __ldcg(P.grad[r][par] + j);
    out[j] = s;
    if (j < n_actor) sq += s * s;
  }
  sq = warp_sum(sq);
  __shared__ float part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = sq;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int k = 0; k < 8; ++k) t += part[k];
    if (norm2) atomicAdd(norm2, t);
    __threadfence();
    if (atomicAdd(ticket, 1u) == gridDim.x - 1) {  // the last block closes the minibatch
      *ticket = 0u;
      *P.epoch = e + 1u;
    }
  }
}

// ---- the same exchange in two phases (reduce-scatter, all-gather): at 8 ranks a rank reads 2 x 7/8 of a buffer over
// NVLink instead of 7 whole buffers. Slice r = floats [r * len, (r + 1) * len), len = stride / world rounded up to 4.
__device__ __forceinline__ void peers_wait(const unsigned* flags, int world, unsigned want) {
  if ((int)threadIdx.x < world) {
    unsigned long long t0 = 0, now = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (ld_acquire_sys(flags + threadIdx.x) < want) {
      __nanosleep(64);
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (now - t0 > 20000000000ull) __trap();
    }
  }
  __syncthreads();
}
__device__ __forceinline__ int peers_slice_len(const DyrosPpoPeers& P) { return ((P.stride + P.world - 1) / P.world + 3) & ~3; }
__global__ void __launch_bounds__(256) k_ppo_reduce_scatter_peers(DyrosPpoPeers P, float* __restrict__ out, int n, int n_actor) {
  const unsigned e = *P.epoch;
  const int par = (int)(e & 1u);
  if (blockIdx.x == 0 && (int)threadIdx.x < P.world) {
    __threadfence_system();
    st_release_sys(P.flags[threadIdx.x] + P.rank, e + 1u);
  }
  peers_wait(P.flags[P.rank], P.world, e + 1u);
  const int len = peers_slice_len(P), lo = P.rank * len, hi = min(P.stride, lo + len);
  float* mine = P.sum[P.rank][par];
  float sq = 0.f;
  for (int j = lo + 4 * (blockIdx.x * blockDim.x + threadIdx.x); j < hi; j += 4 * gridDim.x * blockDim.x) {
    float4 x[8];
#pragma unroll
    for (int r = 0; r < 8; ++r)
      if (r < P.world) x[r] = ld_cg4(P.grad[r][par] + j);
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int r = 0; r < 8; ++r)
      if (r < P.world) {
        s.x += x[r].x; s.y += x[r].y; s.z += x[r].z; s.w += x[r].w;
      }
    *reinterpret_cast<float4*>(mine + j) = s;
    const float v[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (j + c < n) {
        out[j + c] = v[c];
        if (j + c < n_actor) sq += v[c] * v[c];
      }
  }
  sq = warp_sum(sq);
  __shared__ float part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = sq;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int k = 0; k < 8; ++k) t += part[k];
    float* acc = reinterpret_cast<float*>(P.ticket + 2);
    atomicAdd(acc, t);
    __threadfence();
    if (atomicAdd(P.ticket, 1u) == gridDim.x - 1) {  // the last block publishes the slice and its partial norm
      *P.ticket = 0u;
      P.pnorm[P.rank][par] = *reinterpret_cast<volatile float*>(acc);
      *acc = 0.f;
      __threadfence_system();
      for (int q = 0; q < P.world; ++q) st_release_sys(P.flags2[q] + P.rank, e + 1u);
    }
  }
}
__global__ void __launch_bounds__(256) k_ppo_all_gather_peers(DyrosPpoPeers P, float* __restrict__ out, int n, float* __restrict__ norm2) {
  const unsigned e = *P.epoch;
  const int par = (int)(e & 1u);
  peers_wait(P.flags2[P.rank], P.world, e + 1u);
  const int len = peers_slice_len(P);
  // the other ranks' slices, one after the other: element index over (world - 1) * len / 4 float4s
  const int per4 = len / 4, total4 = (P.world - 1) * per4;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total4; i += gridDim.x * blockDim.x) {
    int q = i / per4;
    q += q >= P.rank;
    const int j = q * len + 4 * (i % per4);
    if (j >= P.stride) continue;
    const float4 s = ld_cg4(P.sum[q][par] + j);
    const float v[4] = {s.x, s.y, s.z, s.w};
#pragma unroll
    for (int c = 0; c < 4; ++c)
      if (j + c < n) out[j + c] = v[c];
  }
  if (threadIdx.x == 0) {
    if (blockIdx.x == 0 && norm2) {
      float t = 0.f;
      for (int q = 0; q < P.world; ++q) t += __ldcg(P.pnorm[q] + par);  // rank order: the same bits on every rank
      atomicAdd(norm2, t);
    }
    __threadfence();
    if (atomicAdd(P.ticket + 1, 1u) == gridDim.x - 1) {
      P.ticket[1] = 0u;
      *P.epoch = e + 1u;
    }
  }
}
}  // namespace dyros

using namespace dyros;
void dyros_set_error_ppo(const char* msg) { dyros::set_error("%s", msg); }
#define PPO_CHECK(cond, msg)   \
  do {                         \
    if (!(cond)) {             \
      dyros_set_error_ppo(msg); \
      return 1;                \
    }                          \
  } while (0)

namespace dyros {
static int configure_ppo_kernels() {  // (common.cuh: one carve-out for every kernel of the library)
  static bool done = false;
  if (done) return 0;
  DY_CUDA(prefer_max_smem_carveout(k_ppo_act)); DY_CUDA(prefer_max_smem_carveout(k_ppo_reward));
  DY_CUDA(prefer_max_smem_carveout(k_ppo_advance)); DY_CUDA(prefer_max_smem_carveout(k_ppo_gae));
  DY_CUDA(prefer_max_smem_carveout(k_ppo_loss_grad)); DY_CUDA(prefer_max_smem_carveout(k_ppo_gradnorm));
  DY_CUDA(prefer_max_smem_carveout(k_ppo_adam)); DY_CUDA(prefer_max_smem_carveout(k_ppo_adam_finish));
  DY_CUDA(prefer_max_smem_carveout(k_ppo_cast_obs)); DY_CUDA(prefer_max_smem_carveout(k_ppo_bias_relu));
  DY_CUDA(prefer_max_smem_carveout(k_ppo_relu_bwd)); DY_CUDA(prefer_max_smem_carveout(k_ppo_act_packed));
  DY_CUDA(prefer_max_smem_carveout(k_ppo_loss_grad_packed)); DY_CUDA(prefer_max_smem_carveout(k_ppo_pack));
  DY_CUDA(prefer_max_smem_carveout(k_ppo_unpack)); DY_CUDA(prefer_max_smem_carveout(k_ppo_adam_pack));
  DY_CUDA(prefer_max_smem_carveout(k_ppo_reduce_peers)); DY_CUDA(prefer_max_smem_carveout(k_ppo_reduce_scatter_peers));
  DY_CUDA(prefer_max_smem_carveout(k_ppo_all_gather_peers));
  done = true;
  return 0;
}
}  // namespace dyros

extern "C" {

int dyros_ppo_act(const DyrosPpoBuffers* b, const float* mu, const float* value, const float* logstd, const float* obs,
                  const int64_t* reset_buf, float* actions_env, const float* inject_normal, void* stream) {
  PPO_CHECK(b && mu && value && logstd && obs && reset_buf && actions_env, "dyros_ppo_act: null argument");
  PPO_CHECK(b->obs_dim >= 0, "dyros_ppo_act: DyrosPpoBuffers.obs_dim < 0 (0 means 487)");
  if (configure_ppo_kernels()) return 1;
  k_ppo_act<<<(b->N + 7) / 8, 256, 0, (cudaStream_t)stream>>>(*b, mu, value, logstd, obs, reinterpret_cast<const long long*>(reset_buf),
                                                              actions_env, inject_normal, ppo_width(b->obs_dim));
  DY_LAUNCH_CHECK();
  return 0;
}
int dyros_ppo_reward(const DyrosPpoBuffers* b, const float* rew, const int64_t* timeout, const int64_t* reset_buf, void* stream) {
  PPO_CHECK(b && rew && timeout && reset_buf, "dyros_ppo_reward: null argument");
  if (configure_ppo_kernels()) return 1;
  k_ppo_reward<<<(b->N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(*b, rew, reinterpret_cast<const long long*>(timeout),
                                                                    reinterpret_cast<const long long*>(reset_buf));
  k_ppo_advance<<<1, 1, 0, (cudaStream_t)stream>>>(*b);
  DY_LAUNCH_CHECK();
  return 0;
}
int dyros_ppo_gae(const DyrosPpoBuffers* b, const float* last_values, const int64_t* last_reset, void* stream) {
  PPO_CHECK(b && last_values && last_reset, "dyros_ppo_gae: null argument");
  if (configure_ppo_kernels()) return 1;
  k_ppo_gae<<<(b->N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(*b, last_values, reinterpret_cast<const long long*>(last_reset));
  DY_LAUNCH_CHECK();
  return 0;
}
int dyros_ppo_loss_grad(const DyrosPpoBuffers* b, int row0, int mb, const float* mu, const float* value, const float* logstd,
                        const float* adv_norm, float* dmu, float* dvalue, float* stats, void* stream) {
  PPO_CHECK(b && mu && value && logstd && adv_norm && dmu && dvalue && stats, "dyros_ppo_loss_grad: null argument");
  if (configure_ppo_kernels()) return 1;
  PPO_CHECK(row0 >= 0 && mb > 0 && (long long)row0 + mb <= (long long)b->N * b->H, "dyros_ppo_loss_grad: rows outside the rollout");
  k_ppo_loss_grad<<<(mb + 7) / 8, 256, 0, (cudaStream_t)stream>>>(*b, row0, mb, mu, value, logstd, adv_norm, dmu, dvalue, stats);
  DY_LAUNCH_CHECK();
  return 0;
}
int dyros_ppo_adam(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int n_actor, int n, float grad_scale,
                   float max_norm, float* norm2_scratch, float* lr_dev, int32_t* step_dev, float beta1, float beta2,
                   float eps, float lr0, float lr_min, int lr_max_steps, void* stream) {
  PPO_CHECK(params && grads && exp_avg && exp_avg_sq && norm2_scratch && lr_dev && step_dev, "dyros_ppo_adam: null argument");
  if (configure_ppo_kernels()) return 1;
  PPO_CHECK(n_actor >= 0 && n_actor <= n, "dyros_ppo_adam: n_actor outside [0, n]");
  cudaStream_t s = (cudaStream_t)stream;
  if (max_norm > 0.f && n_actor > 0) k_ppo_gradnorm<<<148, 256, 0, s>>>(grads, n_actor, grad_scale, norm2_scratch);
  k_ppo_adam<<<148 * 2, 256, 0, s>>>(params, grads, exp_avg, exp_avg_sq, n_actor, n, grad_scale, max_norm, norm2_scratch, lr_dev,
                                    step_dev, beta1, beta2, eps);
  k_ppo_adam_finish<<<1, 1, 0, s>>>(norm2_scratch, step_dev, lr_dev, lr0, lr_min, lr_max_steps);
  DY_LAUNCH_CHECK();
  return 0;
}


static bool ppo_net_ok(const DyrosPpoNet* n) {
  return n && n->hidden > 0 && n->hidden % 8 == 0 && n->w0 && n->b0 && n->w1 && n->b1 && n->wh && n->bh;
}
int dyros_ppo_cast_obs(const DyrosPpoBuffers* b, const float* obs, void* x_step, void* x_roll, void* stream) {
  PPO_CHECK(b && obs && x_step, "dyros_ppo_cast_obs: null argument");
  PPO_CHECK(b->obs_dim >= 0, "dyros_ppo_cast_obs: DyrosPpoBuffers.obs_dim < 0 (0 means 487)");
  if (configure_ppo_kernels()) return 1;
  const int W = ppo_width(b->obs_dim);
  k_ppo_cast_obs<<<(b->N + 7) / 8, 256, 0, (cudaStream_t)stream>>>(obs, b->N, W, ppo_padded_width(W), static_cast<bf16*>(x_step),
                                                                   static_cast<bf16*>(x_roll), b->step, b->H);
  DY_LAUNCH_CHECK();
  return 0;
}
int dyros_ppo_bias_relu(void* t, const float* bias, int rows, int hidden, void* stream) {
  PPO_CHECK(t && bias && rows > 0 && hidden > 0 && hidden % 8 == 0, "dyros_ppo_bias_relu: bad argument");
  if (configure_ppo_kernels()) return 1;
  const size_t total8 = (size_t)2 * rows * hidden / 8;
  k_ppo_bias_relu<<<(unsigned)std::min<size_t>((total8 + 255) / 256, 148 * 16), 256, 0, (cudaStream_t)stream>>>(static_cast<bf16*>(t), bias, rows, hidden);
  DY_LAUNCH_CHECK();
  return 0;
}
int dyros_ppo_relu_bwd(void* g, const void* h, float* gbias, int rows, int hidden, void* stream) {
  PPO_CHECK(g && h && gbias && rows > 0 && hidden > 0 && hidden % 8 == 0, "dyros_ppo_relu_bwd: bad argument");
  if (configure_ppo_kernels()) return 1;
  k_ppo_relu_bwd<<<2 * ((rows + kRbRows - 1) / kRbRows) * ((hidden + 255) / 256), 256, 0, (cudaStream_t)stream>>>(static_cast<bf16*>(g), static_cast<const bf16*>(h),
                                                                                        gbias, rows, hidden);
  DY_LAUNCH_CHECK();
  return 0;
}
int dyros_ppo_act_packed(const DyrosPpoBuffers* b, const void* out, const float* bh, const float* logstd, const int64_t* reset_buf,
                         float* actions_env, const float* inject_normal, void* stream) {
  PPO_CHECK(b && out && bh && logstd && reset_buf && actions_env, "dyros_ppo_act_packed: null argument");
  if (configure_ppo_kernels()) return 1;
  k_ppo_act_packed<<<(b->N + 7) / 8, 256, 0, (cudaStream_t)stream>>>(*b, static_cast<const bf16*>(out), bh, logstd,
                                                                     reinterpret_cast<const long long*>(reset_buf), actions_env, inject_normal);
  DY_LAUNCH_CHECK();
  return 0;
}
int dyros_ppo_loss_grad_packed(const DyrosPpoBuffers* b, int row0, int mb, const void* out, const float* bh, const float* logstd,
                               const float* adv_norm, void* dout, float* gbh, float* stats, void* stream) {
  PPO_CHECK(b && out && bh && logstd && adv_norm && dout && gbh && stats, "dyros_ppo_loss_grad_packed: null argument");
  PPO_CHECK(row0 >= 0 && mb > 0 && (long long)row0 + mb <= (long long)b->N * b->H, "dyros_ppo_loss_grad_packed: rows outside the rollout");
  if (configure_ppo_kernels()) return 1;
  k_ppo_loss_grad_packed<<<(mb + 7) / 8, 256, 0, (cudaStream_t)stream>>>(*b, row0, mb, static_cast<const bf16*>(out), bh, logstd, adv_norm,
                                                                         static_cast<bf16*>(dout), gbh, stats);
  DY_LAUNCH_CHECK();
  return 0;
}
// The critic's input width Wc of the *_ac entry points: 0 = the actor's (net->inputs); otherwise Wc >= the actor's.
// Writes dyros_last_error and returns -1 for a bad width.
static int ppo_critic_width(const DyrosPpoNet* net, int critic_inputs, const char* fn) {
  if (net->inputs < 0) {
    dyros::set_error("%s: DyrosPpoNet.inputs < 0 (0 means 487)", fn);
    return -1;
  }
  const int Wa = ppo_width(net->inputs);
  if (critic_inputs < 0 || (critic_inputs && critic_inputs < Wa)) {
    dyros::set_error("%s: critic_inputs %d must be 0 (the actor's width) or >= the actor's %d", fn, critic_inputs, Wa);
    return -1;
  }
  return critic_inputs ? critic_inputs : Wa;
}
int dyros_ppo_pack_params(const DyrosPpoNet* net, const float* flat, void* stream) {
  return dyros_ppo_pack_params_ac(net, 0, flat, stream);
}
int dyros_ppo_pack_params_ac(const DyrosPpoNet* net, int critic_inputs, const float* flat, void* stream) {
  PPO_CHECK(ppo_net_ok(net) && flat, "dyros_ppo_pack_params: bad argument");
  const int Wc = ppo_critic_width(net, critic_inputs, "dyros_ppo_pack_params");
  if (Wc < 0) return 1;
  if (configure_ppo_kernels()) return 1;
  k_ppo_pack<<<dim3(64, 12), 256, 0, (cudaStream_t)stream>>>(ppo_segments(net->hidden, ppo_width(net->inputs), Wc), *net, flat);
  DY_LAUNCH_CHECK();
  return 0;
}
int dyros_ppo_unpack_grads(const DyrosPpoNet* net, float* flat_grad, float* norm2_accum, void* stream) {
  return dyros_ppo_unpack_grads_ac(net, 0, flat_grad, norm2_accum, stream);
}
int dyros_ppo_unpack_grads_ac(const DyrosPpoNet* net, int critic_inputs, float* flat_grad, float* norm2_accum, void* stream) {
  PPO_CHECK(ppo_net_ok(net) && net->gw0 && net->gw1 && net->gwh && net->gb0 && net->gb1 && net->gbh && flat_grad,
            "dyros_ppo_unpack_grads: bad argument");
  const int Wc = ppo_critic_width(net, critic_inputs, "dyros_ppo_unpack_grads");
  if (Wc < 0) return 1;
  if (configure_ppo_kernels()) return 1;
  k_ppo_unpack<<<dim3(64, 12), 256, 0, (cudaStream_t)stream>>>(ppo_segments(net->hidden, ppo_width(net->inputs), Wc), *net, flat_grad,
                                                               norm2_accum, nullptr, 0);
  DY_LAUNCH_CHECK();
  return 0;
}

int dyros_ppo_adam_packed(const DyrosPpoNet* net, float* params, const float* grads, float* exp_avg, float* exp_avg_sq, float grad_scale,
                          float max_norm, int norm_done, float* norm2_scratch, float* lr_dev, int32_t* step_dev, float beta1, float beta2,
                          float eps, float lr0, float lr_min, int lr_max_steps, void* stream) {
  return dyros_ppo_adam_packed_ac(net, 0, params, grads, exp_avg, exp_avg_sq, grad_scale, max_norm, norm_done, norm2_scratch, lr_dev,
                                  step_dev, beta1, beta2, eps, lr0, lr_min, lr_max_steps, stream);
}
int dyros_ppo_adam_packed_ac(const DyrosPpoNet* net, int critic_inputs, float* params, const float* grads, float* exp_avg,
                             float* exp_avg_sq, float grad_scale, float max_norm, int norm_done, float* norm2_scratch, float* lr_dev,
                             int32_t* step_dev, float beta1, float beta2, float eps, float lr0, float lr_min, int lr_max_steps,
                             void* stream) {
  PPO_CHECK(ppo_net_ok(net) && params && grads && exp_avg && exp_avg_sq && norm2_scratch && lr_dev && step_dev, "dyros_ppo_adam_packed: bad argument");
  const int Wc = ppo_critic_width(net, critic_inputs, "dyros_ppo_adam_packed");
  if (Wc < 0) return 1;
  if (configure_ppo_kernels()) return 1;
  cudaStream_t s = (cudaStream_t)stream;
  const int H = net->hidden, W = ppo_width(net->inputs), n_actor = H * W + H + H * H + H + PPO_NA * H + PPO_NA;
  // norm2 holds the squared norm of the UNSCALED actor gradients (sum over ranks); the kernel scales it
  if (max_norm > 0.f && !norm_done) k_ppo_gradnorm<<<148, 256, 0, s>>>(grads, n_actor, 1.f, norm2_scratch);
  k_ppo_adam_pack<<<dim3(64, 12), 256, 0, s>>>(ppo_segments(H, W, Wc), *net, params, grads, exp_avg, exp_avg_sq, grad_scale, max_norm, norm2_scratch,
                                              lr_dev, step_dev, beta1, beta2, eps);
  k_ppo_adam_finish<<<1, 1, 0, s>>>(norm2_scratch, step_dev, lr_dev, lr0, lr_min, lr_max_steps);
  DY_LAUNCH_CHECK();
  return 0;
}

static bool ppo_peers_ok(const DyrosPpoPeers* p) {
  if (!p || p->world < 2 || p->world > 8 || p->rank < 0 || p->rank >= p->world || !p->epoch || !p->ticket || p->stride < 4 || p->stride % 4) return false;
  for (int r = 0; r < p->world; ++r)
    if (!p->grad[r][0] || !p->grad[r][1] || !p->flags[r]) return false;
  return true;
}
int dyros_ppo_unpack_grads_peers(const DyrosPpoNet* net, const DyrosPpoPeers* peers, void* stream) {
  return dyros_ppo_unpack_grads_peers_ac(net, 0, peers, stream);
}
int dyros_ppo_unpack_grads_peers_ac(const DyrosPpoNet* net, int critic_inputs, const DyrosPpoPeers* peers, void* stream) {
  PPO_CHECK(ppo_net_ok(net) && net->gw0 && net->gw1 && net->gwh && net->gb0 && net->gb1 && net->gbh && ppo_peers_ok(peers),
            "dyros_ppo_unpack_grads_peers: bad argument");
  PPO_CHECK(peers->grad[peers->rank][1] == peers->grad[peers->rank][0] + peers->stride, "dyros_ppo_unpack_grads_peers: the rank's two buffers must be `stride` apart");
  const int Wc = ppo_critic_width(net, critic_inputs, "dyros_ppo_unpack_grads_peers");
  if (Wc < 0) return 1;
  if (configure_ppo_kernels()) return 1;
  k_ppo_unpack<<<dim3(64, 12), 256, 0, (cudaStream_t)stream>>>(ppo_segments(net->hidden, ppo_width(net->inputs), Wc), *net, peers->grad[peers->rank][0], nullptr, peers->epoch,
                                                               (size_t)peers->stride);
  DY_LAUNCH_CHECK();
  return 0;
}
int dyros_ppo_reduce_peers(const DyrosPpoPeers* peers, float* flat_grad_sum, int n, int n_actor, float* norm2_accum, void* stream) {
  PPO_CHECK(ppo_peers_ok(peers) && flat_grad_sum && n > 0 && n <= peers->stride && n_actor >= 0 && n_actor <= n, "dyros_ppo_reduce_peers: bad argument");
  PPO_CHECK((reinterpret_cast<uintptr_t>(flat_grad_sum) & 15) == 0, "dyros_ppo_reduce_peers: the output must be 16-byte aligned");
  if (configure_ppo_kernels()) return 1;
  k_ppo_reduce_peers<<<148 * 2, 256, 0, (cudaStream_t)stream>>>(*peers, flat_grad_sum, n, n_actor, norm2_accum, peers->ticket);
  DY_LAUNCH_CHECK();
  return 0;
}
static bool ppo_peers2_ok(const DyrosPpoPeers* p) {
  if (!ppo_peers_ok(p)) return false;
  for (int r = 0; r < p->world; ++r)
    if (!p->sum[r][0] || !p->sum[r][1] || !p->flags2[r] || !p->pnorm[r]) return false;
  return true;
}
int dyros_ppo_reduce_scatter_peers(const DyrosPpoPeers* peers, float* flat_grad_sum, int n, int n_actor, void* stream) {
  PPO_CHECK(ppo_peers2_ok(peers) && flat_grad_sum && n > 0 && n <= peers->stride && n_actor >= 0 && n_actor <= n,
            "dyros_ppo_reduce_scatter_peers: bad argument");
  if (configure_ppo_kernels()) return 1;
  k_ppo_reduce_scatter_peers<<<48, 256, 0, (cudaStream_t)stream>>>(*peers, flat_grad_sum, n, n_actor);
  DY_LAUNCH_CHECK();
  return 0;
}
int dyros_ppo_all_gather_peers(const DyrosPpoPeers* peers, float* flat_grad_sum, int n, float* norm2_accum, void* stream) {
  PPO_CHECK(ppo_peers2_ok(peers) && flat_grad_sum && n > 0 && n <= peers->stride, "dyros_ppo_all_gather_peers: bad argument");
  if (configure_ppo_kernels()) return 1;
  k_ppo_all_gather_peers<<<148, 256, 0, (cudaStream_t)stream>>>(*peers, flat_grad_sum, n, norm2_accum);
  DY_LAUNCH_CHECK();
  return 0;
}

// Peer-shareable device memory (plain cudaMalloc + CUDA IPC): allocated and zeroed by its owner, opened by the other
// ranks of the node IN THE CONTEXT OF THE DEVICE THAT WILL DEREFERENCE IT (the current device), which is what makes
// cudaIpcMemLazyEnablePeerAccess enable the peer path (a mapping opened under the owner's device does not).
int dyros_peer_alloc(size_t bytes, void** ptr, unsigned char* handle64) {
  PPO_CHECK(bytes > 0 && ptr && handle64, "dyros_peer_alloc: bad argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t");
  DY_CUDA(cudaMalloc(ptr, bytes));
  DY_CUDA(cudaMemset(*ptr, 0, bytes));
  DY_CUDA(cudaDeviceSynchronize());
  cudaIpcMemHandle_t h;
  DY_CUDA(cudaIpcGetMemHandle(&h, *ptr));
  memcpy(handle64, &h, 64);
  return 0;
}
int dyros_peer_open(const unsigned char* handle64, void** ptr) {
  PPO_CHECK(handle64 && ptr, "dyros_peer_open: bad argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  DY_CUDA(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return 0;
}
int dyros_peer_close(void* ptr) {
  if (ptr) DY_CUDA(cudaIpcCloseMemHandle(ptr));
  return 0;
}
int dyros_peer_free(void* ptr) {
  if (ptr) DY_CUDA(cudaFree(ptr));
  return 0;
}

}  // extern "C"
