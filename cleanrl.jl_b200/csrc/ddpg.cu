// ddpg.cu — vectorised DDPG on Pendulum behind the crl_ddpg_* entry points of include/cleanrl_ddpg.h: N Pendulum envs
// stepping in lockstep with a deterministic actor plus Gaussian exploration noise, an HBM-resident ring replay buffer, and
// one learning step (sample without replacement -> critic TD regression against the target nets -> Adam; on every
// policy_frequency-th learning step the actor's -Q gradient through the just-updated critic -> Adam -> Polyak averaging of
// both targets) every train_freq iterations.
//
// The reference's ddpg.jl trains on MuJoCo HalfCheetah through PyCall and is not part of this checkout; the semantics are
// pinned by the header (CleanRL-Python's ddpg_continuous_action.py with 64-wide nets on Pendulum), not by ddpg.jl.
//
// Both nets are Dense(IN,64,relu) -> Dense(64,64,relu) -> Dense(64,1) (actor: IN = 3, then 2 tanh; critic: IN = 4 =
// [obs; action]). Every kernel evaluates them out of shared memory with mlp_forward: register tiles of 4 neurons x 4
// samples in the hidden layer, and every neuron is ONE fmaf chain over ascending k, so results do not depend on the tiling.
//
//   ddpg_act_kernel         32 envs per CTA of 256 threads. All threads evaluate the actor; warp 0 (one lane per env,
//                           state in registers) draws the warm-up or noise action from Philox stream 5, steps Pendulum,
//                           appends the transition at (ptr + step * N + env) % capacity and resets a finished env on the
//                           spot. The parameters only change at a learning step, so ONE launch runs every iteration up
//                           to the next learning step.
//   ddpg_critic_fwd_kernel  learning step, critic part 1: CTA c owns samples 16c..16c+15 of the batch: gather, target
//                           actor, target critic, TD target (Float64), critic forward, loss, backward deltas; what the
//                           weight gradients need is written sample-major to a global scratch (L2-resident).
//   ddpg_actor_fwd_kernel   actor part 1 on the same batch: actor forward, critic forward on [obs; mu(obs)], the
//                           gradient of -mean Q back through the critic to the action input, then through the actor.
//   ddpg_update_kernel<IN>  part 2 for either net: one thread per parameter sums its gradient over the batch in ascending
//                           sample order (deterministic, no float atomics) and applies Adam in place.
//   ddpg_polyak_kernel      theta' <- tau theta + (1 - tau) theta' for both targets, after the actor step only.
//
// TD3 (crl_td3_* of include/cleanrl_td3.h) runs on the same acting kernel, ring, batch sampling, actor step and Polyak
// kernel; only its critic step is its own:
//   td3_critic_fwd_kernel     grid (ceil(B/16), 2), blockIdx.y = k picks qf1 or qf2: gather, target actor, clipped
//                             smoothing noise (Philox stream 7), both target critics, y from their minimum (Float64),
//                             then critic k's forward, loss and backward into scratch k.
//   td3_critic_update_kernel  both critics' reductions and Adam steps in one launch (blockIdx.y picks the net); the body
//                             is ddpg_update_kernel's.
//   td3_polyak_kernel         qf2' after the actor step; ddpg_polyak_kernel does actor' and qf1'.
// SAC (crl_sac_* of include/cleanrl_sac.h) runs on the same ring, batch sampling and twin reduction, with an actor of two
// heads (mean, log_std: DNet<3, 2>) and a temperature learned on the device:
//   sac_act_kernel            ddpg_act_kernel's body with a = 2 tanh(mean + std z), z DDPG's stream-5 normal.
//   sac_critic_fwd_kernel     td3_critic_fwd_kernel's grid; a' and log_pi' from the current actor (Philox stream 8), y
//                             from the minimum of both target critics minus alpha log_pi'; then td3_critic_update_kernel.
//   sac_actor_fwd_kernel      one actor iteration: sample (stream 9), both critics, backward through the minimum, the
//                             squash and the log-prob into both heads; then sac_actor_update_kernel (two-head reduction).
//   sac_alpha_fwd_kernel      a fresh sample (stream 10) and per-CTA sums of log_pi; sac_alpha_update_kernel, one thread,
//                             steps log_alpha with Adam.
//   sac_polyak_kernel         qf1' and qf2' in one launch.
// The raw entry points run the same kernels on rows the caller passes in (sample b = row b), with the gradient written
// out instead of an Adam step, so that each can be compared with a reference on its own. Every decision that only
// depends on counters (learn on this iteration?, actor step?, Adam's beta powers) is taken on the host, so a run is a
// plain sequence of launches on one stream without any device-to-host read.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <string>

#include "../../include/cleanrl_ddpg.h"
#include "../../include/cleanrl_td3.h"
#include "../../include/cleanrl_sac.h"
#include "device_math.cuh"
#include "kernels.h"

namespace {

// ---- network geometry (the one place the widths live)
constexpr int DD_D = 3, DD_A = 1, DD_H = 64;   // observation [cos th, sin th, thdot], torque, hidden width
constexpr float DD_MAX_TORQUE = 2.0f;
// flat Flux.params order, each W (out,in) column-major. HO Dense(64,1) heads, each its W then its b (head h at W3 + h HS):
// one for DDPG's and TD3's nets, two (mean, log_std) for SAC's actor
template <int IN, int HO = 1> struct DNet {
  static constexpr int W1 = 0, B1 = W1 + DD_H * IN, W2 = B1 + DD_H, B2 = W2 + DD_H * DD_H, W3 = B2 + DD_H, B3 = W3 + DD_H,
                       HS = DD_H + 1, P = W3 + HO * HS, PP = (P + 3) & ~3;
};
using ANet = DNet<DD_D>;           // actor mu
using CNet = DNet<DD_D + DD_A>;    // critic Q
using SNet = DNet<DD_D, 2>;        // SAC actor: fc_mean, fc_logstd
static_assert(ANet::P == CRL_DDPG_ACTOR_PARAMS && CNet::P == CRL_DDPG_CRITIC_PARAMS, "parameter counts");
static_assert(SNet::P == CRL_SAC_ACTOR_PARAMS, "SAC actor parameter count");
static_assert(ANet::W2 % 4 == 0 && CNet::W2 % 4 == 0, "128-bit weight loads of the hidden layer");

constexpr uint32_t STREAM_DDPG_ACT = 5u, STREAM_DDPG_BATCH = 6u, STREAM_TD3_SMOOTH = 7u;
constexpr uint32_t STREAM_SAC_TARGET = 8u, STREAM_SAC_ACTOR = 9u, STREAM_SAC_ALPHA = 10u;
constexpr int ACT_E = 32;                 // envs per CTA in ddpg_act_kernel
constexpr int ACT_SP = ACT_E + 4;         // activation row stride (floats): rows stay 16-byte aligned
constexpr int ACT_T = 256;                // threads of ddpg_act_kernel
constexpr int ACT_MAX_STEPS = 1024;       // iterations per ddpg_act_kernel launch (bounds one launch's duration)
constexpr int LEARN_B = 256;              // max batch size
constexpr int LF_S = 16, LF_SP = LF_S + 4, LF_T = 256;   // learning forward kernels: samples per CTA, row stride, threads
constexpr int LF_MAX_BLOCKS = LEARN_B / LF_S;
constexpr int XS = 4;                     // row stride of the gathered inputs in the scratch (critic: 4, actor: 3 used)
constexpr int LU_T = 256;                 // ddpg_update_kernel threads

struct DdpgDev {               // device-resident scalars
  double critic_loss, actor_loss;
  double sum_return, sum_length;
  unsigned long long episodes;
};

// global -> shared copy of one parameter vector of P floats (128-bit loads; cudaMalloc'ed source, 16-byte aligned dst)
template <int P, int NT> __device__ __forceinline__ void load_params(const float* __restrict__ g, float* sp, int tid) {
  const float4* g4 = reinterpret_cast<const float4*>(g);
  float4* s4 = reinterpret_cast<float4*>(sp);
  constexpr int N4 = P / 4, PER = (N4 + NT - 1) / NT;
  float4 tmp[PER];   // every load is in flight before the first store
#pragma unroll
  for (int u = 0; u < PER; u++) if (tid + u * NT < N4) tmp[u] = g4[tid + u * NT];
#pragma unroll
  for (int u = 0; u < PER; u++) if (tid + u * NT < N4) s4[tid + u * NT] = tmp[u];
  if (tid < P % 4) sp[N4 * 4 + tid] = g[N4 * 4 + tid];
}

// Dense(IN,64,relu) -> Dense(64,64,relu) -> Dense(64,1) for a tile of NS samples by the NT threads of the CTA (every
// thread must call this: __syncthreads between the layers and at the end). p: parameters in shared memory (16-byte
// aligned); xs [IN][SP] the inputs, h1/h2 [64][SP] the activations, out [SP] the head's pre-activation. A thread owns 4
// consecutive samples of one first-layer neuron, then 4 neurons x 4 samples of the hidden layer (one 128-bit weight load
// + one 128-bit activation load per k for 16 FMAs), then one sample of one head. With HO heads, out is [HO][SP].
template <int IN, int NS, int SP, int NT, int HO = 1>
__device__ __forceinline__ void mlp_forward(const float* __restrict__ p, const float* xs, float* h1, float* h2, float* out, int tid) {
  using N = DNet<IN, HO>;
  constexpr int EQ = NS / 4;
  static_assert(NS % 4 == 0 && SP % 4 == 0 && SP >= NS && NS <= NT, "tile geometry");
  for (int w = tid; w < DD_H * EQ; w += NT) {
    const int eq = w % EQ, j = w / EQ;
    float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll
    for (int k = 0; k < IN; k++) {
      const float wt = p[N::W1 + j + DD_H * k];
      const float4 x = *reinterpret_cast<const float4*>(xs + k * SP + 4 * eq);
      acc.x = fmaf(wt, x.x, acc.x); acc.y = fmaf(wt, x.y, acc.y); acc.z = fmaf(wt, x.z, acc.z); acc.w = fmaf(wt, x.w, acc.w);
    }
    const float b = p[N::B1 + j];
    *reinterpret_cast<float4*>(h1 + j * SP + 4 * eq) =
        make_float4(fmaxf(acc.x + b, 0.0f), fmaxf(acc.y + b, 0.0f), fmaxf(acc.z + b, 0.0f), fmaxf(acc.w + b, 0.0f));
  }
  __syncthreads();
  for (int w = tid; w < (DD_H / 4) * EQ; w += NT) {
    const int eq = w % EQ, j = 4 * (w / EQ);
    float acc[4][4];   // 16 independent scalar chains
#pragma unroll
    for (int n = 0; n < 4; n++)
#pragma unroll
      for (int c = 0; c < 4; c++) acc[n][c] = 0.0f;
#pragma unroll 8
    for (int k = 0; k < DD_H; k++) {
      const float4 wv4 = *reinterpret_cast<const float4*>(p + N::W2 + j + DD_H * k);
      const float4 hv4 = *reinterpret_cast<const float4*>(h1 + k * SP + 4 * eq);
      const float wv[4] = {wv4.x, wv4.y, wv4.z, wv4.w}, hv[4] = {hv4.x, hv4.y, hv4.z, hv4.w};
#pragma unroll
      for (int n = 0; n < 4; n++)
#pragma unroll
        for (int c = 0; c < 4; c++) acc[n][c] = fmaf(wv[n], hv[c], acc[n][c]);
    }
#pragma unroll
    for (int n = 0; n < 4; n++) {
      const float b = p[N::B2 + j + n];
      *reinterpret_cast<float4*>(h2 + (j + n) * SP + 4 * eq) =
          make_float4(fmaxf(acc[n][0] + b, 0.0f), fmaxf(acc[n][1] + b, 0.0f), fmaxf(acc[n][2] + b, 0.0f), fmaxf(acc[n][3] + b, 0.0f));
    }
  }
  __syncthreads();
  if constexpr (HO == 1) {
    if (tid < NS) {
      float acc = 0.0f;
#pragma unroll 16
      for (int k = 0; k < DD_H; k++) acc = fmaf(p[N::W3 + k], h2[k * SP + tid], acc);
      out[tid] = acc + p[N::B3];
    }
  } else {
    static_assert(HO * NS <= NT, "one thread per head output");
    if (tid < HO * NS) {
      const int h = tid / NS, i = tid % NS;
      float acc = 0.0f;
#pragma unroll 16
      for (int k = 0; k < DD_H; k++) acc = fmaf(p[N::W3 + h * N::HS + k], h2[k * SP + i], acc);
      out[h * SP + i] = acc + p[N::B3 + h * N::HS];
    }
  }
  __syncthreads();
}

// mu = 2 tanh(head), the torque limit of Pendulum
__device__ __forceinline__ float actor_out(float u) { return DD_MAX_TORQUE * tanhf(u); }

// Backward of Dense(IN,64,relu) -> Dense(64,64,relu) -> Dense(64,1) for the CTA's NS samples given d(head) per sample
// in dout: exports x (rows 0..IN-1 of xs), h1, h2, dz2 and dz1 sample-major (neuron fastest) for samples b0 + i < B, and
// leaves dz1 in z1s when it is not null (the actor step needs the critic's dz1 for the gradient of the action input).
// With HO heads, dout is [HO][SP] and dT is exported [B][HO].
struct Scratch {
  float *xT, *h1T, *h2T, *z1T, *z2T, *dT;   // [B][XS], [B][64] x4, [B][HO]
};
template <int IN, int NS, int SP, int NT, int HO = 1>
__device__ __forceinline__ void mlp_backward(const float* __restrict__ p, const float* xs, const float* h1, const float* h2,
                                             const float* dout, float* z2s, float* z1s, const Scratch& s, int b0, int B,
                                             bool do_export, int tid) {
  using N = DNet<IN, HO>;
  for (int w = tid; w < DD_H * NS; w += NT) {
    const int k = w % DD_H, i = w / DD_H, b = b0 + i;
    const float hv = h2[k * SP + i];
    float z;   // relu'(0) = 0, as Flux
    if constexpr (HO == 1) z = hv > 0.0f ? p[N::W3 + k] * dout[i] : 0.0f;
    else z = hv > 0.0f ? fmaf(p[N::W3 + N::HS + k], dout[SP + i], p[N::W3 + k] * dout[i]) : 0.0f;
    z2s[k * SP + i] = z;
    if (do_export && b < B) { s.h1T[b * DD_H + k] = h1[k * SP + i]; s.h2T[b * DD_H + k] = hv; s.z2T[b * DD_H + k] = z; }
  }
  if (do_export && tid < NS && b0 + tid < B) {
    const int b = b0 + tid;
#pragma unroll
    for (int c = 0; c < IN; c++) s.xT[b * XS + c] = xs[c * SP + tid];
#pragma unroll
    for (int h = 0; h < HO; h++) s.dT[b * HO + h] = dout[h * SP + tid];
  }
  __syncthreads();
  for (int w = tid; w < DD_H * NS; w += NT) {
    const int k = w % DD_H, i = w / DD_H, b = b0 + i;
    float acc = 0.0f;
    const float* wc = p + N::W2 + DD_H * k;   // column k of W2: W2(j, k) for ascending j
#pragma unroll 16
    for (int j = 0; j < DD_H; j++) acc = fmaf(wc[j], z2s[j * SP + i], acc);
    const float z = h1[k * SP + i] > 0.0f ? acc : 0.0f;
    if (z1s) z1s[k * SP + i] = z;
    if (do_export && b < B) s.z1T[b * DD_H + k] = z;
  }
  __syncthreads();
}

struct ActArgs {
  const float* actor;
  float* env_state; int* env_t; double* ep_ret; int* ep_len; uint32_t* resets;
  float *b_obs, *b_next, *b_act, *b_rew; uint8_t* b_term;
  DdpgDev* dev;
  unsigned long long seed, it0;   // it0 = iteration number (1-based) of step 0 of this launch
  long long learning_starts;
  float sigma;                    // exploration_noise * max torque
  int n_steps;
  int N, C, ptr, max_steps;
};

// Warps 0-7 evaluate the actor for the CTA's 32 envs (skipped while every step of the launch is warm-up); warp 0 (one
// lane per env) then draws the action, records the transition and advances its env. HO = 1: DDPG's actor and
// clamp(mu + sigma z, -2, 2); HO = 2: SAC's actor and 2 tanh(mean + std z), z the same draw.
// (tid is read in the kernel, where __launch_bounds__ bounds it)
template <int HO>
__device__ __forceinline__ void act_body(const ActArgs& a, int tid) {
  using N = DNet<DD_D, HO>;
  extern __shared__ __align__(16) float smem[];
  constexpr int SP = ACT_SP;
  float* p = smem;                        // [N::PP]
  float* h1 = p + N::PP;                  // [64][SP]
  float* h2 = h1 + DD_H * SP;             // [64][SP]
  float* uo = h2 + DD_H * SP;             // [HO][SP]
  float* xs = uo + HO * SP;               // [3][SP] current observation of the CTA's envs
  const bool any_policy = (long long)(a.it0 + a.n_steps - 1) * a.N > a.learning_starts;
  if (any_policy) load_params<N::P, ACT_T>(a.actor, p, tid);
  const int n = blockIdx.x * ACT_E + tid;
  const bool owner = tid < ACT_E, valid = owner && n < a.N;
  const uint32_t gid = (uint32_t)n;       // Philox is keyed by the global env id
  float st[2] = {0.0f, 0.0f};
  int t = 0, len = 0;
  double ret = 0.0;
  uint32_t rc = 0;
  if (valid) {
    const float2 s2 = reinterpret_cast<const float2*>(a.env_state)[n];
    st[0] = s2.x; st[1] = s2.y;
    t = a.env_t[n]; ret = a.ep_ret[n]; len = a.ep_len[n]; rc = a.resets[n];
  }
  for (int s = 0; s < a.n_steps; s++) {
    const unsigned long long it = a.it0 + (unsigned long long)s;
    const bool warm = (long long)it * a.N <= a.learning_starts;   // uniform over the grid
    float obs[DD_D];
    env_obs<CRL_ENV_PENDULUM>(st, obs);
    if (owner) {
#pragma unroll
      for (int k = 0; k < DD_D; k++) xs[k * SP + tid] = obs[k];
    }
    if (!warm) {
      __syncthreads();
      mlp_forward<DD_D, ACT_E, SP, ACT_T, HO>(p, xs, h1, h2, uo, tid);   // mu(obs), or mean and the log_std head
    }
    if (valid) {
      uint32_t r[4];
      philox_draw(a.seed, gid, it, STREAM_DDPG_ACT, r);
      float act;
      if (warm) {
        act = __fmaf_rn(2.0f * DD_MAX_TORQUE, (float)(r[0] >> 8) * (1.0f / 16777216.0f), -DD_MAX_TORQUE);   // U[-2, 2)
      } else {
        // Box-Muller standard normal from 24-bit uniforms (u1 in (0, 1]), as rng_action_normals
        const float u1 = (float)((r[0] >> 8) + 1u) * (1.0f / 16777216.0f);
        const float u2 = (float)(r[1] >> 8) * (1.0f / 16777216.0f);
        const float z = sqrtf(-2.0f * logf(u1)) * cosf(6.283185307179586f * u2);
        if constexpr (HO == 1) {
          act = fmaf(a.sigma, z, actor_out(uo[tid]));
          act = fminf(fmaxf(act, -DD_MAX_TORQUE), DD_MAX_TORQUE);
        } else {
          const float log_std = -5.0f + 3.5f * (tanhf(uo[SP + tid]) + 1.0f);
          act = actor_out(fmaf(expf(log_std), z, uo[tid]));
        }
      }
      float rew;
      bool done;
      pendulum_step(st, t, act, a.max_steps, rew, done);
      float nobs[DD_D];
      env_obs<CRL_ENV_PENDULUM>(st, nobs);                         // next_obs before any reset
      const long long slot = ((long long)a.ptr + (long long)s * a.N + n) % a.C;
#pragma unroll
      for (int k = 0; k < DD_D; k++) { a.b_obs[slot * DD_D + k] = obs[k]; a.b_next[slot * DD_D + k] = nobs[k]; }
      a.b_act[slot] = act;
      a.b_rew[slot] = rew;
      a.b_term[slot] = done ? 1 : 0;
      ret += (double)rew;
      len += 1;
      if (done) {
        atomicAdd(&a.dev->episodes, 1ull);
        atomicAdd(&a.dev->sum_return, ret);
        atomicAdd(&a.dev->sum_length, (double)len);
        ret = 0.0;
        len = 0;
        float u4[4];
        rng_reset_uniforms(a.seed, gid, rc, u4);
        pendulum_reset(st, t, u4);
        rc += 1;
      }
    }
    if (!warm) __syncthreads();   // uo and xs are rewritten by the next step
  }
  if (valid) {
    a.ep_ret[n] = ret; a.ep_len[n] = len; a.env_t[n] = t; a.resets[n] = rc;
    reinterpret_cast<float2*>(a.env_state)[n] = make_float2(st[0], st[1]);
  }
}

__global__ void __launch_bounds__(ACT_T, 1) ddpg_act_kernel(ActArgs a) { act_body<1>(a, threadIdx.x); }
__global__ void __launch_bounds__(ACT_T, 1) sac_act_kernel(ActArgs a) { act_body<2>(a, threadIdx.x); }

// crl_ddpg_forward_raw: the acting kernel's actor forward pass (same mlp_forward instantiation, 32 samples per CTA) and
// the critic on [obs; act] with the same tiling; rows past n are zero and not written back
__global__ void __launch_bounds__(ACT_T, 1) ddpg_forward_raw_kernel(const float* actor, const float* critic, const float* obs,
                                                                    const float* act, float* mu_out, float* q_out, int64_t n) {
  extern __shared__ __align__(16) float smem[];
  constexpr int SP = ACT_SP;
  float* pa = smem;                       // [ANet::PP]
  float* pc = pa + ANet::PP;              // [CNet::PP]
  float* h1 = pc + CNet::PP;              // [64][SP]
  float* h2 = h1 + DD_H * SP;             // [64][SP]
  float* uo = h2 + DD_H * SP;             // [SP]
  float* xs = uo + SP;                    // [4][SP]
  const int tid = threadIdx.x;
  load_params<ANet::P, ACT_T>(actor, pa, tid);
  load_params<CNet::P, ACT_T>(critic, pc, tid);
  const int64_t i = (int64_t)blockIdx.x * ACT_E + tid;
  if (tid < ACT_E) {
#pragma unroll
    for (int k = 0; k < DD_D; k++) xs[k * SP + tid] = i < n ? obs[i * DD_D + k] : 0.0f;
    xs[DD_D * SP + tid] = i < n ? act[i] : 0.0f;
  }
  __syncthreads();
  mlp_forward<DD_D, ACT_E, SP, ACT_T>(pa, xs, h1, h2, uo, tid);
  if (tid < ACT_E && i < n) mu_out[i] = actor_out(uo[tid]);
  __syncthreads();
  mlp_forward<DD_D + DD_A, ACT_E, SP, ACT_T>(pc, xs, h1, h2, uo, tid);
  if (tid < ACT_E && i < n) q_out[i] = uo[tid];
}

struct LearnArgs {
  const float *actor, *critic, *actor_tgt, *critic_tgt;
  const float *b_obs, *b_next, *b_act, *b_rew; const uint8_t* b_term;
  unsigned long long seed, learn_step;
  double gamma;
  int B, size;
  int in_order;           // sample b is row b of the b_* arrays (raw entry points), not entry b of the keyed permutation
  Scratch s;
  double* loss_part;      // [LF_MAX_BLOCKS]
};

// sample(1:size, B, replace=false): the first B entries of a keyed permutation of [0, size), Philox stream 6 keyed by the
// learning-step index (the critic and the actor step of one learning step see the same batch)
__device__ __forceinline__ uint32_t batch_row(const LearnArgs& a, int b) {
  if (a.in_order) return (uint32_t)b;
  uint32_t keys[8];
  philox_draw(a.seed, 0u, a.learn_step, STREAM_DDPG_BATCH, keys);
  philox_draw(a.seed, 0x80000000u, a.learn_step, STREAM_DDPG_BATCH, keys + 4);
  return perm_index((uint32_t)b, (uint32_t)a.size, perm_half_bits((uint32_t)a.size), keys);
}

// the squared errors (or Q-values) of the CTA's 16 samples summed in Float64 by lanes 0-15 of warp 0, in a fixed order
__device__ __forceinline__ void block_part(double v, double* part) {
#pragma unroll
  for (int o = LF_S / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0x0000ffffu, v, o);
  if (threadIdx.x == 0) part[blockIdx.x] = v;
}

__global__ void __launch_bounds__(LF_T) ddpg_critic_fwd_kernel(LearnArgs a) {
  extern __shared__ __align__(16) float smem[];
  constexpr int SP = LF_SP;
  float* pat = smem;                      // target actor
  float* pct = pat + ANet::PP;            // target critic
  float* pc = pct + CNet::PP;             // critic
  float* h1 = pc + CNet::PP;              // [64][SP]
  float* h2 = h1 + DD_H * SP;             // [64][SP]
  float* z2 = h2 + DD_H * SP;             // [64][SP]
  float* xin = z2 + DD_H * SP;            // [4][SP] obs, action
  float* xn = xin + 4 * SP;               // [4][SP] next_obs, mu'(next_obs)
  float* out = xn + 4 * SP;               // [SP]
  float* dout = out + SP;                 // [SP]
  __shared__ float s_rew[LF_S];
  __shared__ int s_term[LF_S];
  const int tid = threadIdx.x, B = a.B, b0 = blockIdx.x * LF_S;
  // the gather (HBM latency) is issued first and completes under the parameter loads
  float o[DD_D] = {0.0f, 0.0f, 0.0f}, nx[DD_D] = {0.0f, 0.0f, 0.0f}, act = 0.0f, rew = 0.0f;
  int term = 0;
  if (tid < LF_S && b0 + tid < B) {
    const uint32_t idx = batch_row(a, b0 + tid);
#pragma unroll
    for (int k = 0; k < DD_D; k++) { o[k] = a.b_obs[idx * DD_D + k]; nx[k] = a.b_next[idx * DD_D + k]; }
    act = a.b_act[idx]; rew = a.b_rew[idx]; term = a.b_term[idx];
  }
  load_params<ANet::P, LF_T>(a.actor_tgt, pat, tid);
  load_params<CNet::P, LF_T>(a.critic_tgt, pct, tid);
  load_params<CNet::P, LF_T>(a.critic, pc, tid);
  if (tid < LF_S) {
#pragma unroll
    for (int k = 0; k < DD_D; k++) { xin[k * SP + tid] = o[k]; xn[k * SP + tid] = nx[k]; }
    xin[DD_D * SP + tid] = act;
    s_rew[tid] = rew; s_term[tid] = term;
  }
  __syncthreads();
  mlp_forward<DD_D, LF_S, SP, LF_T>(pat, xn, h1, h2, out, tid);             // target_actor(next_obs)
  if (tid < LF_S) xn[DD_D * SP + tid] = actor_out(out[tid]);
  __syncthreads();
  mlp_forward<DD_D + DD_A, LF_S, SP, LF_T>(pct, xn, h1, h2, out, tid);      // qf1_target(next_obs, mu'(next_obs))
  double y = 0.0;
  if (tid < LF_S) y = (double)s_rew[tid] + a.gamma * (1.0 - (double)s_term[tid]) * (double)out[tid];
  mlp_forward<DD_D + DD_A, LF_S, SP, LF_T>(pc, xin, h1, h2, out, tid);      // qf1(obs, action)
  if (tid < LF_S) {
    const bool in = b0 + tid < B;
    const double diff = (double)out[tid] - y;
    dout[tid] = in ? (float)(2.0 * diff / (double)B) : 0.0f;               // d mse / d q
    block_part(in ? diff * diff : 0.0, a.loss_part);
  }
  __syncthreads();
  mlp_backward<DD_D + DD_A, LF_S, SP, LF_T>(pc, xin, h1, h2, dout, z2, nullptr, a.s, b0, B, true, tid);
}

__global__ void __launch_bounds__(LF_T) ddpg_actor_fwd_kernel(LearnArgs a) {
  extern __shared__ __align__(16) float smem[];
  constexpr int SP = LF_SP;
  float* pa = smem;                       // actor
  float* pc = pa + ANet::PP;              // critic (as just updated)
  float* h1a = pc + CNet::PP;             // [64][SP]
  float* h2a = h1a + DD_H * SP;
  float* h1c = h2a + DD_H * SP;
  float* h2c = h1c + DD_H * SP;
  float* z2 = h2c + DD_H * SP;
  float* z1c = z2 + DD_H * SP;
  float* xin = z1c + DD_H * SP;           // [4][SP] obs, mu(obs)
  float* out = xin + 4 * SP;              // [SP]
  float* dout = out + SP;                 // [SP]
  const int tid = threadIdx.x, B = a.B, b0 = blockIdx.x * LF_S;
  float o[DD_D] = {0.0f, 0.0f, 0.0f};
  if (tid < LF_S && b0 + tid < B) {
    const uint32_t idx = batch_row(a, b0 + tid);
#pragma unroll
    for (int k = 0; k < DD_D; k++) o[k] = a.b_obs[idx * DD_D + k];
  }
  load_params<ANet::P, LF_T>(a.actor, pa, tid);
  load_params<CNet::P, LF_T>(a.critic, pc, tid);
  if (tid < LF_S) {
#pragma unroll
    for (int k = 0; k < DD_D; k++) xin[k * SP + tid] = o[k];
  }
  __syncthreads();
  mlp_forward<DD_D, LF_S, SP, LF_T>(pa, xin, h1a, h2a, out, tid);           // actor(obs)
  float u = 0.0f;
  if (tid < LF_S) { u = out[tid]; xin[DD_D * SP + tid] = actor_out(u); }
  __syncthreads();
  mlp_forward<DD_D + DD_A, LF_S, SP, LF_T>(pc, xin, h1c, h2c, out, tid);    // qf1(obs, actor(obs))
  if (tid < LF_S) {
    const bool in = b0 + tid < B;
    dout[tid] = in ? (float)(-1.0 / (double)B) : 0.0f;                     // d(-mean Q) / dQ
    block_part(in ? (double)out[tid] : 0.0, a.loss_part);
  }
  __syncthreads();
  // through the critic (its gradient is not kept) to the action input: dL/da = sum_j W1c(j, action) dz1c(j)
  mlp_backward<DD_D + DD_A, LF_S, SP, LF_T>(pc, xin, h1c, h2c, dout, z2, z1c, a.s, b0, B, false, tid);
  if (tid < LF_S) {
    float da = 0.0f;
#pragma unroll 16
    for (int j = 0; j < DD_H; j++) da = fmaf(pc[CNet::W1 + j + DD_H * DD_D], z1c[j * SP + tid], da);
    // d(2 tanh u)/du = 2 sech^2 u, from cosh: 1 - tanh^2 would cancel where the head saturates
    const float ch = coshf(u);
    dout[tid] = b0 + tid < B ? da * (DD_MAX_TORQUE / (ch * ch)) : 0.0f;
  }
  __syncthreads();
  mlp_backward<DD_D, LF_S, SP, LF_T>(pa, xin, h1a, h2a, dout, z2, nullptr, a.s, b0, B, true, tid);
}

struct UpdArgs {
  float *params, *m, *v;
  float* grads_out;        // non-null: write the gradient and leave params, m, v alone (raw entry points)
  Scratch s;
  const double* loss_part;
  int n_parts, B;
  double loss_sign;        // +1: critic (mean squared error), -1: actor (-mean Q)
  double* loss_out;
  double lr, bp1, bp2;     // beta1^t, beta2^t of Adam, kept on the host
};

// Parameter i of a DNet<IN, HO>: its gradient summed over the batch in ascending sample order (one fmaf chain), then
// Flux.Adam / torch.optim.Adam in the form of dqn_adam: Float64 scalars, Float32 state. Thread 0 also writes the loss.
template <int IN, int HO = 1>
__device__ __forceinline__ void update_param(const UpdArgs& a, int i) {
  using N = DNet<IN, HO>;
  if (i == 0) {
    double sum = 0.0;
    for (int c = 0; c < a.n_parts; c++) sum += a.loss_part[c];
    *a.loss_out = a.loss_sign * sum / (double)a.B;
  }
  if (i >= N::P) return;
  const int B = a.B;
  const float *u, *w = nullptr;   // gradient = sum_b u[b * us] * w[b * ws] (w == nullptr: sum_b u[b * us])
  int us, ws = 0;
  if (i < N::B1) { u = a.s.z1T + (i % DD_H); us = DD_H; w = a.s.xT + i / DD_H; ws = XS; }
  else if (i < N::W2) { u = a.s.z1T + (i - N::B1); us = DD_H; }
  else if (i < N::B2) { const int r = i - N::W2; u = a.s.z2T + r % DD_H; us = DD_H; w = a.s.h1T + r / DD_H; ws = DD_H; }
  else if (i < N::W3) { u = a.s.z2T + (i - N::B2); us = DD_H; }
  else if constexpr (HO == 1) {
    if (i < N::B3) { u = a.s.dT; us = 1; w = a.s.h2T + (i - N::W3); ws = DD_H; }
    else { u = a.s.dT; us = 1; }
  } else {
    const int h = (i - N::W3) / N::HS, j = (i - N::W3) % N::HS;   // head h: W (j < 64) or b
    u = a.s.dT + h; us = HO;
    if (j < DD_H) { w = a.s.h2T + j; ws = DD_H; }
  }
  float g = 0.0f;
  if (w) {
#pragma unroll 8
    for (int b = 0; b < B; b++) g = fmaf(__ldg(u + b * us), __ldg(w + b * ws), g);
  } else {
#pragma unroll 8
    for (int b = 0; b < B; b++) g += __ldg(u + b * us);
  }
  if (a.grads_out) { a.grads_out[i] = g; return; }
  const double b1 = 0.9, b2 = 0.999, eps = 1e-8;
  const float m0 = a.m[i], v0 = a.v[i], p0 = a.params[i];
  const double c1 = 1.0 - a.bp1, c2 = 1.0 - a.bp2;
  const float mt = (float)__dadd_rn(__dmul_rn(b1, (double)m0), __dmul_rn(1.0 - b1, (double)g));
  const float vt = (float)__dadd_rn(__dmul_rn(b2, (double)v0), __dmul_rn(__dmul_rn(1.0 - b2, (double)g), (double)g));
  const double den = __dadd_rn(sqrt(__ddiv_rn((double)vt, c2)), eps);
  const float step = (float)__dmul_rn(__ddiv_rn(__ddiv_rn((double)mt, c1), den), a.lr);
  a.m[i] = mt;
  a.v[i] = vt;
  a.params[i] = __fsub_rn(p0, step);
}

// one thread per parameter of one net
template <int IN>
__global__ void __launch_bounds__(LU_T) ddpg_update_kernel(UpdArgs a) {
  update_param<IN>(a, blockIdx.x * LU_T + threadIdx.x);
}

// theta' <- tau theta + (1 - tau) theta' for the actor (i < ANet::P) and the critic, in Float64 and rounded once
__global__ void __launch_bounds__(256) ddpg_polyak_kernel(const float* actor, float* actor_tgt, const float* critic, float* critic_tgt, double tau) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const float* p = i < ANet::P ? actor + i : critic + (i - ANet::P);
  float* t = i < ANet::P ? actor_tgt + i : critic_tgt + (i - ANet::P);
  if (i >= ANet::P + CNet::P) return;
  *t = (float)__dadd_rn(__dmul_rn(tau, (double)*p), __dmul_rn(1.0 - tau, (double)*t));
}

// ---- TD3: twin critics with target-policy smoothing on the DDPG kernels (include/cleanrl_td3.h)
struct Td3Args {
  LearnArgs l;                        // actor_tgt, critic = qf1, critic_tgt = qf1', the batch, and qf1's scratch and loss parts
  const float *critic2, *critic2_tgt; // qf2, qf2'
  Scratch s2;
  double* loss_part2;
  float policy_noise, noise_clip;
};

// Part 1 of the learning step of both critics, grid (ceil(B/16), 2): blockIdx.y = k picks qf(k+1). Every CTA gathers its
// 16 samples, runs the target actor, draws the clipped smoothing noise (Philox stream 7, word = position in the batch,
// counter = learning-step index), runs both target critics, forms y from their minimum with DDPG's expression, and then
// runs critic k's forward and backward into scratch k. The two y-halves of a sample run the same instructions on the same
// inputs, so both critics regress on bit-identical targets.
__global__ void __launch_bounds__(LF_T) td3_critic_fwd_kernel(Td3Args t) {
  extern __shared__ __align__(16) float smem[];
  constexpr int SP = LF_SP;
  const LearnArgs& a = t.l;
  const int k = blockIdx.y;
  float* pat = smem;                      // target actor
  float* pq1t = pat + ANet::PP;           // qf1'
  float* pq2t = pq1t + CNet::PP;          // qf2'
  float* pc = pq2t + CNet::PP;            // critic k
  float* h1 = pc + CNet::PP;              // [64][SP]
  float* h2 = h1 + DD_H * SP;             // [64][SP]
  float* z2 = h2 + DD_H * SP;             // [64][SP]
  float* xin = z2 + DD_H * SP;            // [4][SP] obs, action
  float* xn = xin + 4 * SP;               // [4][SP] next_obs, smoothed mu'(next_obs)
  float* out = xn + 4 * SP;               // [SP]
  float* dout = out + SP;                 // [SP]
  __shared__ float s_rew[LF_S];
  __shared__ int s_term[LF_S];
  const int tid = threadIdx.x, B = a.B, b0 = blockIdx.x * LF_S;
  float o[DD_D] = {0.0f, 0.0f, 0.0f}, nx[DD_D] = {0.0f, 0.0f, 0.0f}, act = 0.0f, rew = 0.0f;
  int term = 0;
  if (tid < LF_S && b0 + tid < B) {
    const uint32_t idx = batch_row(a, b0 + tid);
#pragma unroll
    for (int c = 0; c < DD_D; c++) { o[c] = a.b_obs[idx * DD_D + c]; nx[c] = a.b_next[idx * DD_D + c]; }
    act = a.b_act[idx]; rew = a.b_rew[idx]; term = a.b_term[idx];
  }
  load_params<ANet::P, LF_T>(a.actor_tgt, pat, tid);
  load_params<CNet::P, LF_T>(a.critic_tgt, pq1t, tid);
  load_params<CNet::P, LF_T>(t.critic2_tgt, pq2t, tid);
  load_params<CNet::P, LF_T>(k ? t.critic2 : a.critic, pc, tid);
  if (tid < LF_S) {
#pragma unroll
    for (int c = 0; c < DD_D; c++) { xin[c * SP + tid] = o[c]; xn[c * SP + tid] = nx[c]; }
    xin[DD_D * SP + tid] = act;
    s_rew[tid] = rew; s_term[tid] = term;
  }
  __syncthreads();
  mlp_forward<DD_D, LF_S, SP, LF_T>(pat, xn, h1, h2, out, tid);             // target_actor(next_obs)
  if (tid < LF_S) {
    // eps = clamp(policy_noise z, -noise_clip, noise_clip) * 2 with z Box-Muller as in ddpg_act_kernel; every operation
    // in Float32 in this order (no contraction), then a' = clamp(mu' + eps, -2, 2)
    uint32_t r[4];
    philox_draw(a.seed, (uint32_t)(b0 + tid), a.learn_step, STREAM_TD3_SMOOTH, r);
    const float u1 = (float)((r[0] >> 8) + 1u) * (1.0f / 16777216.0f);
    const float u2 = (float)(r[1] >> 8) * (1.0f / 16777216.0f);
    const float z = sqrtf(-2.0f * logf(u1)) * cosf(6.283185307179586f * u2);
    const float eps = __fmul_rn(fminf(fmaxf(__fmul_rn(t.policy_noise, z), -t.noise_clip), t.noise_clip), DD_MAX_TORQUE);
    xn[DD_D * SP + tid] = fminf(fmaxf(__fadd_rn(actor_out(out[tid]), eps), -DD_MAX_TORQUE), DD_MAX_TORQUE);
  }
  __syncthreads();
  mlp_forward<DD_D + DD_A, LF_S, SP, LF_T>(pq1t, xn, h1, h2, out, tid);     // qf1_target(next_obs, a')
  const float q1n = tid < LF_S ? out[tid] : 0.0f;
  mlp_forward<DD_D + DD_A, LF_S, SP, LF_T>(pq2t, xn, h1, h2, out, tid);     // qf2_target(next_obs, a')
  double y = 0.0;
  if (tid < LF_S) y = (double)s_rew[tid] + a.gamma * (1.0 - (double)s_term[tid]) * (double)fminf(q1n, out[tid]);
  mlp_forward<DD_D + DD_A, LF_S, SP, LF_T>(pc, xin, h1, h2, out, tid);      // qf_k(obs, action)
  if (tid < LF_S) {
    const bool in = b0 + tid < B;
    const double diff = (double)out[tid] - y;
    dout[tid] = in ? (float)(2.0 * diff / (double)B) : 0.0f;               // d mse / d q
    block_part(in ? diff * diff : 0.0, k ? t.loss_part2 : a.loss_part);
  }
  __syncthreads();
  mlp_backward<DD_D + DD_A, LF_S, SP, LF_T>(pc, xin, h1, h2, dout, z2, nullptr, k ? t.s2 : a.s, b0, B, true, tid);
}

// part 2 of both critics in one launch: blockIdx.y picks the net, its scratch, its loss parts and its Adam state
__global__ void __launch_bounds__(LU_T) td3_critic_update_kernel(UpdArgs q1, UpdArgs q2) {
  update_param<DD_D + DD_A>(blockIdx.y ? q2 : q1, blockIdx.x * LU_T + threadIdx.x);
}

// qf2' <- tau qf2 + (1 - tau) qf2', as ddpg_polyak_kernel does for the actor and qf1
__global__ void __launch_bounds__(256) td3_polyak_kernel(const float* critic2, float* critic2_tgt, double tau) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= CNet::P) return;
  critic2_tgt[i] = (float)__dadd_rn(__dmul_rn(tau, (double)critic2[i]), __dmul_rn(1.0 - tau, (double)critic2_tgt[i]));
}

// ---- SAC: squashed-Gaussian actor, twin critics and a learned temperature on the DDPG kernels (include/cleanrl_sac.h)
struct SacDev {                // device-resident SAC scalars (the losses of DdpgDev are qf1's and the actor's)
  double alpha, alpha_loss, qf2_loss;
  float log_alpha, la_m, la_v;   // the temperature's parameter and its Adam moments (Float32, as a torch parameter)
};

struct SacArgs {
  LearnArgs l;                        // actor = the SAC actor, critic = qf1, critic_tgt = qf1', the batch, scratch and loss parts
  const float *critic2, *critic2_tgt; // qf2, qf2'
  Scratch s2;                         // critic step: qf2's scratch
  double* loss_part2;                 // critic step: qf2's squared errors; actor step: log_pi sums (NULL: not kept)
  const double* alpha;                // the temperature as it stands before this launch
  unsigned long long draw;            // counter of the noise: learning-step index (stream 8) or actor iteration (9, 10)
};

// standard normal in Float64 by Box-Muller from the 24-bit uniforms of Philox(seed, word, counter, stream), the bit
// recipe of the acting noise
__device__ __forceinline__ double normal_f64(unsigned long long seed, uint32_t word, unsigned long long counter, uint32_t stream) {
  uint32_t r[4];
  philox_draw(seed, word, counter, stream, r);
  const double u1 = (double)((r[0] >> 8) + 1u) * (1.0 / 16777216.0), u2 = (double)(r[1] >> 8) * (1.0 / 16777216.0);
  return sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
}

// the reparameterised tanh-squashed sample of one row and what its gradient needs, in Float64 from the Float32 heads:
// log_std = -5 + 3.5 (tanh(l) + 1), x = mean + exp(log_std) z, a = 2 tanh x,
// log_pi = -z^2/2 - log_std - log(2 pi)/2 - log(2 (1 - tanh^2 x) + 1e-6); 1 - tanh^2 x is taken as 1/cosh^2 x, which
// does not cancel where x saturates
struct Squash {
  double z, std, t, s2, sq, dls, logpi;   // s2 = 1 - tanh^2 x, sq = 2 s2 + 1e-6, dls = d log_std / dl
  float a;
};
__device__ __forceinline__ Squash squash(float mean, float l, double z) {
  Squash q;
  q.z = z;
  const double cl = cosh((double)l);
  const double log_std = -5.0 + 3.5 * (tanh((double)l) + 1.0);
  q.dls = 3.5 / (cl * cl);
  q.std = exp(log_std);
  const double x = (double)mean + q.std * z;
  const double cx = cosh(x);
  q.t = tanh(x);
  q.s2 = 1.0 / (cx * cx);
  q.sq = 2.0 * q.s2 + 1e-6;
  q.logpi = -0.5 * z * z - log_std - 0.91893853320467274 - log(q.sq);
  q.a = (float)(2.0 * q.t);
  return q;
}

// Part 1 of both critics' learning step, grid (ceil(B/16), 2) as td3_critic_fwd_kernel: blockIdx.y = k picks qf(k+1).
// The actor's sample at s' (Philox stream 8, word = position in the batch, counter = learning-step index) gives a' and
// log_pi'; y = r + gamma (1 - d) (min(qf1'(s', a'), qf2'(s', a')) - alpha log_pi') in Float64, the same bits for k = 0, 1.
__global__ void __launch_bounds__(LF_T) sac_critic_fwd_kernel(SacArgs t) {
  extern __shared__ __align__(16) float smem[];
  constexpr int SP = LF_SP;
  const LearnArgs& a = t.l;
  const int k = blockIdx.y;
  float* pa = smem;                       // actor
  float* pq1t = pa + SNet::PP;            // qf1'
  float* pq2t = pq1t + CNet::PP;          // qf2'
  float* pc = pq2t + CNet::PP;            // critic k
  float* h1 = pc + CNet::PP;              // [64][SP]
  float* h2 = h1 + DD_H * SP;             // [64][SP]
  float* z2 = h2 + DD_H * SP;             // [64][SP]
  float* xin = z2 + DD_H * SP;            // [4][SP] obs, action
  float* xn = xin + 4 * SP;               // [4][SP] next_obs, a'
  float* out = xn + 4 * SP;               // [2][SP]
  float* dout = out + 2 * SP;             // [SP]
  __shared__ float s_rew[LF_S];
  __shared__ int s_term[LF_S];
  const int tid = threadIdx.x, B = a.B, b0 = blockIdx.x * LF_S;
  float o[DD_D] = {0.0f, 0.0f, 0.0f}, nx[DD_D] = {0.0f, 0.0f, 0.0f}, act = 0.0f, rew = 0.0f;
  int term = 0;
  if (tid < LF_S && b0 + tid < B) {
    const uint32_t idx = batch_row(a, b0 + tid);
#pragma unroll
    for (int c = 0; c < DD_D; c++) { o[c] = a.b_obs[idx * DD_D + c]; nx[c] = a.b_next[idx * DD_D + c]; }
    act = a.b_act[idx]; rew = a.b_rew[idx]; term = a.b_term[idx];
  }
  load_params<SNet::P, LF_T>(a.actor, pa, tid);
  load_params<CNet::P, LF_T>(a.critic_tgt, pq1t, tid);
  load_params<CNet::P, LF_T>(t.critic2_tgt, pq2t, tid);
  load_params<CNet::P, LF_T>(k ? t.critic2 : a.critic, pc, tid);
  if (tid < LF_S) {
#pragma unroll
    for (int c = 0; c < DD_D; c++) { xin[c * SP + tid] = o[c]; xn[c * SP + tid] = nx[c]; }
    xin[DD_D * SP + tid] = act;
    s_rew[tid] = rew; s_term[tid] = term;
  }
  __syncthreads();
  mlp_forward<DD_D, LF_S, SP, LF_T, 2>(pa, xn, h1, h2, out, tid);          // mean, log_std head at next_obs
  double logpi = 0.0;
  if (tid < LF_S) {
    const Squash q = squash(out[tid], out[SP + tid], normal_f64(a.seed, (uint32_t)(b0 + tid), t.draw, STREAM_SAC_TARGET));
    xn[DD_D * SP + tid] = q.a;
    logpi = q.logpi;
  }
  __syncthreads();
  mlp_forward<DD_D + DD_A, LF_S, SP, LF_T>(pq1t, xn, h1, h2, out, tid);     // qf1_target(next_obs, a')
  const float q1n = tid < LF_S ? out[tid] : 0.0f;
  mlp_forward<DD_D + DD_A, LF_S, SP, LF_T>(pq2t, xn, h1, h2, out, tid);     // qf2_target(next_obs, a')
  double y = 0.0;
  if (tid < LF_S)
    y = (double)s_rew[tid] + a.gamma * (1.0 - (double)s_term[tid]) * ((double)fminf(q1n, out[tid]) - *t.alpha * logpi);
  mlp_forward<DD_D + DD_A, LF_S, SP, LF_T>(pc, xin, h1, h2, out, tid);      // qf_k(obs, action)
  if (tid < LF_S) {
    const bool in = b0 + tid < B;
    const double diff = (double)out[tid] - y;
    dout[tid] = in ? (float)(2.0 * diff / (double)B) : 0.0f;               // d mse / d q
    block_part(in ? diff * diff : 0.0, k ? t.loss_part2 : a.loss_part);
  }
  __syncthreads();
  mlp_backward<DD_D + DD_A, LF_S, SP, LF_T>(pc, xin, h1, h2, dout, z2, nullptr, k ? t.s2 : a.s, b0, B, true, tid);
}

// Part 1 of one actor iteration: the actor's sample at s (Philox stream 9, counter = actor iteration), both critics on
// [s; a], loss mean(alpha log_pi - min(qf1, qf2)); backward through each critic to its action input, the minimum (the
// smaller critic's gradient, half of each on a tie, as torch.minimum), the squash and the log-prob into both heads, then
// through the actor into a.s (dT is [B][2]). loss_part2, when set, receives the per-CTA sums of log_pi.
__global__ void __launch_bounds__(LF_T) sac_actor_fwd_kernel(SacArgs t) {
  extern __shared__ __align__(16) float smem[];
  constexpr int SP = LF_SP;
  const LearnArgs& a = t.l;
  float* pa = smem;                       // actor
  float* pc1 = pa + SNet::PP;             // qf1 (as just updated)
  float* pc2 = pc1 + CNet::PP;            // qf2
  float* h1a = pc2 + CNet::PP;            // [64][SP]
  float* h2a = h1a + DD_H * SP;
  float* h1c = h2a + DD_H * SP;
  float* h2c = h1c + DD_H * SP;
  float* z2 = h2c + DD_H * SP;
  float* z1c = z2 + DD_H * SP;
  float* xin = z1c + DD_H * SP;           // [4][SP] obs, a
  float* out = xin + 4 * SP;              // [2][SP]
  float* dout = out + 2 * SP;             // [2][SP]
  const int tid = threadIdx.x, B = a.B, b0 = blockIdx.x * LF_S;
  float o[DD_D] = {0.0f, 0.0f, 0.0f};
  if (tid < LF_S && b0 + tid < B) {
    const uint32_t idx = batch_row(a, b0 + tid);
#pragma unroll
    for (int c = 0; c < DD_D; c++) o[c] = a.b_obs[idx * DD_D + c];
  }
  load_params<SNet::P, LF_T>(a.actor, pa, tid);
  load_params<CNet::P, LF_T>(a.critic, pc1, tid);
  load_params<CNet::P, LF_T>(t.critic2, pc2, tid);
  if (tid < LF_S) {
#pragma unroll
    for (int c = 0; c < DD_D; c++) xin[c * SP + tid] = o[c];
  }
  __syncthreads();
  mlp_forward<DD_D, LF_S, SP, LF_T, 2>(pa, xin, h1a, h2a, out, tid);       // mean, log_std head
  Squash q;
  if (tid < LF_S) {
    q = squash(out[tid], out[SP + tid], normal_f64(a.seed, (uint32_t)(b0 + tid), t.draw, STREAM_SAC_ACTOR));
    xin[DD_D * SP + tid] = q.a;
  }
  __syncthreads();
  float qv[2], g[2];   // Q_k(s, a) and dQ_k/da of the sample's thread
#pragma unroll
  for (int c = 0; c < 2; c++) {
    const float* pc = c ? pc2 : pc1;
    mlp_forward<DD_D + DD_A, LF_S, SP, LF_T>(pc, xin, h1c, h2c, out, tid);
    if (tid < LF_S) { qv[c] = out[tid]; dout[tid] = b0 + tid < B ? 1.0f : 0.0f; }
    __syncthreads();
    mlp_backward<DD_D + DD_A, LF_S, SP, LF_T>(pc, xin, h1c, h2c, dout, z2, z1c, a.s, b0, B, false, tid);
    if (tid < LF_S) {
      float da = 0.0f;
#pragma unroll 16
      for (int j = 0; j < DD_H; j++) da = fmaf(pc[CNet::W1 + j + DD_H * DD_D], z1c[j * SP + tid], da);
      g[c] = da;
    }
  }
  if (tid < LF_S) {
    const bool in = b0 + tid < B;
    const double alpha = *t.alpha;
    const float dq = qv[0] < qv[1] ? g[0] : qv[1] < qv[0] ? g[1] : 0.5f * g[0] + 0.5f * g[1];
    // d(alpha log_pi - min Q)/dx with da/dx = 2 (1 - tanh^2 x) and d log_pi/dx = 4 tanh x (1 - tanh^2 x) / sq
    const double gx = alpha * 4.0 * q.t * q.s2 / q.sq - (double)dq * 2.0 * q.s2;
    dout[tid] = in ? (float)(gx / (double)B) : 0.0f;                                     // d loss / d mean
    dout[SP + tid] = in ? (float)((gx * q.std * q.z - alpha) * q.dls / (double)B) : 0.0f; // d loss / d l
    block_part(in ? alpha * q.logpi - (double)fminf(qv[0], qv[1]) : 0.0, a.loss_part);
    if (t.loss_part2) block_part(in ? q.logpi : 0.0, t.loss_part2);
  }
  __syncthreads();
  mlp_backward<DD_D, LF_S, SP, LF_T, 2>(pa, xin, h1a, h2a, dout, z2, nullptr, a.s, b0, B, true, tid);
}

// part 2 of the actor iteration: the width-2 reduction with Adam; logpi_out (raw entry point) gets the batch's mean log_pi
__global__ void __launch_bounds__(LU_T) sac_actor_update_kernel(UpdArgs u, const double* logpi_part, double* logpi_out) {
  const int i = blockIdx.x * LU_T + threadIdx.x;
  update_param<DD_D, 2>(u, i);
  if (i == 0 && logpi_out) {
    double sum = 0.0;
    for (int c = 0; c < u.n_parts; c++) sum += logpi_part[c];
    *logpi_out = sum / (double)u.B;
  }
}

// the temperature's forward: a fresh sample from the actor just updated (Philox stream 10, counter = actor iteration)
// and per-CTA Float64 sums of log_pi into a.loss_part
__global__ void __launch_bounds__(LF_T) sac_alpha_fwd_kernel(SacArgs t) {
  extern __shared__ __align__(16) float smem[];
  constexpr int SP = LF_SP;
  const LearnArgs& a = t.l;
  float* pa = smem;                       // actor
  float* h1 = pa + SNet::PP;              // [64][SP]
  float* h2 = h1 + DD_H * SP;
  float* xin = h2 + DD_H * SP;            // [4][SP] obs
  float* out = xin + 4 * SP;              // [2][SP]
  const int tid = threadIdx.x, B = a.B, b0 = blockIdx.x * LF_S;
  float o[DD_D] = {0.0f, 0.0f, 0.0f};
  if (tid < LF_S && b0 + tid < B) {
    const uint32_t idx = batch_row(a, b0 + tid);
#pragma unroll
    for (int c = 0; c < DD_D; c++) o[c] = a.b_obs[idx * DD_D + c];
  }
  load_params<SNet::P, LF_T>(a.actor, pa, tid);
  if (tid < LF_S) {
#pragma unroll
    for (int c = 0; c < DD_D; c++) xin[c * SP + tid] = o[c];
  }
  __syncthreads();
  mlp_forward<DD_D, LF_S, SP, LF_T, 2>(pa, xin, h1, h2, out, tid);
  if (tid < LF_S) {
    const Squash q = squash(out[tid], out[SP + tid], normal_f64(a.seed, (uint32_t)(b0 + tid), t.draw, STREAM_SAC_ALPHA));
    block_part(b0 + tid < B ? q.logpi : 0.0, a.loss_part);
  }
}

// the temperature's step, one thread: alpha_loss = -exp(log_alpha) (mean log_pi + target_entropy), which is also its
// gradient with respect to log_alpha; Adam as update_param (Float32 gradient and state, Float64 scalars); then alpha
struct AlphaArgs {
  const double* part;
  int n_parts, B;
  SacDev* dev;
  double lr, bp1, bp2;   // the actor's beta powers: the temperature's step count is the actor's
};
constexpr double SAC_TARGET_ENTROPY = -1.0;   // -dim(action space)
__global__ void sac_alpha_update_kernel(AlphaArgs a) {
  double sum = 0.0;
  for (int c = 0; c < a.n_parts; c++) sum += a.part[c];
  SacDev* d = a.dev;
  const float la = d->log_alpha;
  const double loss = -exp((double)la) * (sum / (double)a.B + SAC_TARGET_ENTROPY);
  d->alpha_loss = loss;
  const float g = (float)loss;
  const double b1 = 0.9, b2 = 0.999, eps = 1e-8;
  const double c1 = 1.0 - a.bp1, c2 = 1.0 - a.bp2;
  const float mt = (float)__dadd_rn(__dmul_rn(b1, (double)d->la_m), __dmul_rn(1.0 - b1, (double)g));
  const float vt = (float)__dadd_rn(__dmul_rn(b2, (double)d->la_v), __dmul_rn(__dmul_rn(1.0 - b2, (double)g), (double)g));
  const double den = __dadd_rn(sqrt(__ddiv_rn((double)vt, c2)), eps);
  const float step = (float)__dmul_rn(__ddiv_rn(__ddiv_rn((double)mt, c1), den), a.lr);
  d->la_m = mt;
  d->la_v = vt;
  d->log_alpha = __fsub_rn(la, step);
  d->alpha = exp((double)d->log_alpha);
}

// qf1' and qf2' <- tau theta + (1 - tau) theta', in Float64 and rounded once
__global__ void __launch_bounds__(256) sac_polyak_kernel(const float* critic, float* critic_tgt, const float* critic2, float* critic2_tgt,
                                                         double tau) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * CNet::P) return;
  const float* p = i < CNet::P ? critic + i : critic2 + (i - CNet::P);
  float* t = i < CNet::P ? critic_tgt + i : critic2_tgt + (i - CNet::P);
  *t = (float)__dadd_rn(__dmul_rn(tau, (double)*p), __dmul_rn(1.0 - tau, (double)*t));
}

// crl_sac_forward_raw: the acting kernel's actor forward (mean, and log_std after its squash) and a critic on
// [obs; act], 32 samples per CTA; rows past n are zero and not written back
__global__ void __launch_bounds__(ACT_T, 1) sac_forward_raw_kernel(const float* actor, const float* critic, const float* obs,
                                                                   const float* act, float* mean_out, float* log_std_out,
                                                                   float* q_out, int64_t n) {
  extern __shared__ __align__(16) float smem[];
  constexpr int SP = ACT_SP;
  float* pa = smem;                       // [SNet::PP]
  float* pc = pa + SNet::PP;              // [CNet::PP]
  float* h1 = pc + CNet::PP;              // [64][SP]
  float* h2 = h1 + DD_H * SP;             // [64][SP]
  float* uo = h2 + DD_H * SP;             // [2][SP]
  float* xs = uo + 2 * SP;                // [4][SP]
  const int tid = threadIdx.x;
  load_params<SNet::P, ACT_T>(actor, pa, tid);
  load_params<CNet::P, ACT_T>(critic, pc, tid);
  const int64_t i = (int64_t)blockIdx.x * ACT_E + tid;
  if (tid < ACT_E) {
#pragma unroll
    for (int k = 0; k < DD_D; k++) xs[k * SP + tid] = i < n ? obs[i * DD_D + k] : 0.0f;
    xs[DD_D * SP + tid] = i < n ? act[i] : 0.0f;
  }
  __syncthreads();
  mlp_forward<DD_D, ACT_E, SP, ACT_T, 2>(pa, xs, h1, h2, uo, tid);
  if (tid < ACT_E && i < n) {
    mean_out[i] = uo[tid];
    log_std_out[i] = -5.0f + 3.5f * (tanhf(uo[SP + tid]) + 1.0f);
  }
  __syncthreads();
  mlp_forward<DD_D + DD_A, ACT_E, SP, ACT_T>(pc, xs, h1, h2, uo, tid);
  if (tid < ACT_E && i < n) q_out[i] = uo[tid];
}

__global__ void ddpg_reset_kernel(int N, unsigned long long seed, float* env_state, int* env_t, double* ep_ret, int* ep_len, uint32_t* resets) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float u4[4], st[2];
  int t;
  rng_reset_uniforms(seed, (uint32_t)n, 0, u4);
  pendulum_reset(st, t, u4);
  env_state[2 * n] = st[0]; env_state[2 * n + 1] = st[1];
  env_t[n] = t; ep_ret[n] = 0.0; ep_len[n] = 0; resets[n] = 1;
}

constexpr size_t ACT_SMEM = (ANet::PP + (2 * DD_H + 1 + DD_D) * ACT_SP) * sizeof(float);
constexpr size_t FWD_RAW_SMEM = (ANet::PP + CNet::PP + (2 * DD_H + 1 + 4) * ACT_SP) * sizeof(float);
constexpr size_t CF_SMEM = (ANet::PP + 2 * CNet::PP + (3 * DD_H + 8 + 2) * LF_SP) * sizeof(float);
constexpr size_t AF_SMEM = (ANet::PP + CNet::PP + (6 * DD_H + 4 + 2) * LF_SP) * sizeof(float);
constexpr size_t TCF_SMEM = (ANet::PP + 3 * CNet::PP + (3 * DD_H + 8 + 2) * LF_SP) * sizeof(float);
static_assert(ACT_SMEM <= 227 * 1024 && FWD_RAW_SMEM <= 227 * 1024 && CF_SMEM <= 227 * 1024 && AF_SMEM <= 227 * 1024, "ddpg shared memory");
static_assert(TCF_SMEM <= 227 * 1024, "td3 shared memory");
constexpr size_t SACT_SMEM = (SNet::PP + (2 * DD_H + 2 + DD_D) * ACT_SP) * sizeof(float);
constexpr size_t SFWD_RAW_SMEM = (SNet::PP + CNet::PP + (2 * DD_H + 2 + 4) * ACT_SP) * sizeof(float);
constexpr size_t SCF_SMEM = (SNet::PP + 3 * CNet::PP + (3 * DD_H + 8 + 3) * LF_SP) * sizeof(float);
constexpr size_t SAF_SMEM = (SNet::PP + 2 * CNet::PP + (6 * DD_H + 4 + 4) * LF_SP) * sizeof(float);
constexpr size_t SAL_SMEM = (SNet::PP + (2 * DD_H + 4 + 2) * LF_SP) * sizeof(float);
static_assert(SACT_SMEM <= 227 * 1024 && SFWD_RAW_SMEM <= 227 * 1024 && SCF_SMEM <= 227 * 1024 && SAF_SMEM <= 227 * 1024 &&
              SAL_SMEM <= 227 * 1024, "sac shared memory");
constexpr size_t SCRATCH_FLOATS = (size_t)LEARN_B * (XS + 4 * DD_H + 1);
constexpr size_t SAC_SCRATCH_FLOATS = SCRATCH_FLOATS + LEARN_B;   // dT of the two-headed actor is [B][2]

int dfail(int code, const std::string& msg) { return crl_internal_fail(code, msg.c_str()); }
#define DCK(call)                                                                                           \
  do {                                                                                                      \
    cudaError_t e__ = (call);                                                                               \
    if (e__ != cudaSuccess)                                                                                 \
      return dfail(CRL_ERR_CUDA, std::string(#call) + " failed: " + cudaGetErrorString(e__) + " (ddpg.cu)"); \
  } while (0)

template <typename T> cudaError_t dzalloc(T** p, size_t n) {
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), (n ? n : 1) * sizeof(T));
  if (e != cudaSuccess) return e;
  return cudaMemset(*p, 0, (n ? n : 1) * sizeof(T));
}

Scratch carve(float* base) {
  Scratch s;
  s.h1T = base; s.h2T = s.h1T + LEARN_B * DD_H; s.z1T = s.h2T + LEARN_B * DD_H; s.z2T = s.z1T + LEARN_B * DD_H;
  s.xT = s.z2T + LEARN_B * DD_H; s.dT = s.xT + LEARN_B * XS;
  return s;
}

cudaError_t set_smem_attrs() {
  cudaError_t e = cudaFuncSetAttribute(ddpg_act_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ACT_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(ddpg_forward_raw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FWD_RAW_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(ddpg_critic_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)CF_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(ddpg_actor_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)AF_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(td3_critic_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TCF_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(sac_act_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SACT_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(sac_forward_raw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SFWD_RAW_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(sac_critic_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SCF_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(sac_actor_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SAF_SMEM);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(sac_alpha_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SAL_SMEM);
  return e;
}

// the two kernels of one net's step: forward + deltas, then the reduction with Adam (grads_out == nullptr) or without
cudaError_t launch_net_step(bool critic, const LearnArgs& l, UpdArgs u, cudaStream_t s) {
  const int fwd_blocks = (l.B + LF_S - 1) / LF_S;
  if (critic) ddpg_critic_fwd_kernel<<<fwd_blocks, LF_T, CF_SMEM, s>>>(l);
  else ddpg_actor_fwd_kernel<<<fwd_blocks, LF_T, AF_SMEM, s>>>(l);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  u.s = l.s; u.loss_part = l.loss_part; u.n_parts = fwd_blocks; u.B = l.B; u.loss_sign = critic ? 1.0 : -1.0;
  if (critic) ddpg_update_kernel<DD_D + DD_A><<<(CNet::P + LU_T - 1) / LU_T, LU_T, 0, s>>>(u);
  else ddpg_update_kernel<DD_D><<<(ANet::P + LU_T - 1) / LU_T, LU_T, 0, s>>>(u);
  return cudaGetLastError();
}

// TD3's critic step: both critics' forward + deltas in one launch, then both reductions with Adam (or without) in one
cudaError_t launch_td3_critic_step(const Td3Args& t, UpdArgs u1, UpdArgs u2, cudaStream_t s) {
  const int fwd_blocks = (t.l.B + LF_S - 1) / LF_S;
  td3_critic_fwd_kernel<<<dim3(fwd_blocks, 2), LF_T, TCF_SMEM, s>>>(t);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  u1.s = t.l.s; u1.loss_part = t.l.loss_part;
  u2.s = t.s2; u2.loss_part = t.loss_part2;
  for (UpdArgs* u : {&u1, &u2}) { u->n_parts = fwd_blocks; u->B = t.l.B; u->loss_sign = 1.0; }
  td3_critic_update_kernel<<<dim3((CNet::P + LU_T - 1) / LU_T, 2), LU_T, 0, s>>>(u1, u2);
  return cudaGetLastError();
}

// SAC's critic step: sac_critic_fwd_kernel, then TD3's twin reduction with Adam (or without)
cudaError_t launch_sac_critic_step(const SacArgs& t, UpdArgs u1, UpdArgs u2, cudaStream_t s) {
  const int fwd_blocks = (t.l.B + LF_S - 1) / LF_S;
  sac_critic_fwd_kernel<<<dim3(fwd_blocks, 2), LF_T, SCF_SMEM, s>>>(t);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  u1.s = t.l.s; u1.loss_part = t.l.loss_part;
  u2.s = t.s2; u2.loss_part = t.loss_part2;
  for (UpdArgs* u : {&u1, &u2}) { u->n_parts = fwd_blocks; u->B = t.l.B; u->loss_sign = 1.0; }
  td3_critic_update_kernel<<<dim3((CNet::P + LU_T - 1) / LU_T, 2), LU_T, 0, s>>>(u1, u2);
  return cudaGetLastError();
}

// one SAC actor iteration: sac_actor_fwd_kernel, then the width-2 reduction with Adam (or without)
cudaError_t launch_sac_actor_step(const SacArgs& t, UpdArgs u, double* logpi_out, cudaStream_t s) {
  const int fwd_blocks = (t.l.B + LF_S - 1) / LF_S;
  sac_actor_fwd_kernel<<<fwd_blocks, LF_T, SAF_SMEM, s>>>(t);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  u.s = t.l.s; u.loss_part = t.l.loss_part; u.n_parts = fwd_blocks; u.B = t.l.B; u.loss_sign = 1.0;
  sac_actor_update_kernel<<<(SNet::P + LU_T - 1) / LU_T, LU_T, 0, s>>>(u, t.loss_part2, logpi_out);
  return cudaGetLastError();
}

}  // namespace

struct crl_ddpg_ctx {
  crl_ddpg_config cfg;
  cudaStream_t stream;
  float *actor, *critic, *actor_tgt, *critic_tgt, *am, *av, *cm, *cv;
  float* env_state; int* env_t; double* ep_ret; int* ep_len; uint32_t* resets;
  float *b_obs, *b_next, *b_act, *b_rew; uint8_t* b_term;
  DdpgDev* dev;
  float* scratch;
  double* loss_part;
  double abp1, abp2, cbp1, cbp2;   // beta1^t, beta2^t of the actor's and the critic's Adam
  int size, ptr;
  long long it, learn_steps, actor_steps, launches;
  bool params_set, reset_done;
};

static int ddpg_validate(const crl_ddpg_config* cfg) {
  if (cfg->struct_size != (int32_t)sizeof(crl_ddpg_config)) return dfail(CRL_ERR_INVALID, "crl_ddpg_config.struct_size mismatch");
  if (cfg->num_envs < 1 || cfg->buffer_size < cfg->num_envs) return dfail(CRL_ERR_INVALID, "need 1 <= num_envs <= buffer_size");
  if (cfg->batch_size < 1 || cfg->batch_size > LEARN_B) return dfail(CRL_ERR_INVALID, "batch_size must be in [1, 256]");
  if (cfg->train_freq < 1 || cfg->policy_frequency < 1 || cfg->max_episode_steps < 1)
    return dfail(CRL_ERR_INVALID, "train_freq, policy_frequency and max_episode_steps must be positive");
  if (!(cfg->tau > 0.0 && cfg->tau <= 1.0)) return dfail(CRL_ERR_INVALID, "tau must be in (0, 1]");
  if (cfg->learning_starts < 0) return dfail(CRL_ERR_INVALID, "learning_starts must be >= 0");
  if (!(cfg->exploration_noise >= 0.0) || !(cfg->lr > 0.0)) return dfail(CRL_ERR_INVALID, "need exploration_noise >= 0 and lr > 0");
  return CRL_OK;
}

static int ddpg_device_check(int device) {
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return dfail(CRL_ERR_CUDA, "no CUDA device: libcleanrl_cuda has no CPU fallback");
  if (device < 0 || device >= ndev) return dfail(CRL_ERR_INVALID, "device ordinal out of range");
  cudaDeviceProp prop;
  DCK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return dfail(CRL_ERR_CUDA, "libcleanrl_cuda is built for sm_100a only");
  return CRL_OK;
}

extern "C" CRL_API int crl_ddpg_create(const crl_ddpg_config* cfg, crl_ddpg_ctx** out) {
  if (!cfg || !out) return dfail(CRL_ERR_INVALID, "NULL argument");
  *out = nullptr;
  if (int rc = ddpg_validate(cfg)) return rc;
  if (int rc = ddpg_device_check(cfg->device)) return rc;
  DCK(cudaSetDevice(cfg->device));
  crl_ddpg_ctx* c = new crl_ddpg_ctx();
  memset(c, 0, sizeof(*c));
  // from here on a failure must release what was allocated so far (crl_ddpg_destroy skips null members)
#define DCKC(call)                                                                                            \
  do {                                                                                                        \
    cudaError_t e__ = (call);                                                                                 \
    if (e__ != cudaSuccess) {                                                                                 \
      crl_ddpg_destroy(c);                                                                                    \
      return dfail(CRL_ERR_CUDA, std::string(#call) + " failed: " + cudaGetErrorString(e__) + " (ddpg.cu)"); \
    }                                                                                                         \
  } while (0)
  c->cfg = *cfg;
  const size_t N = cfg->num_envs, C = cfg->buffer_size;
  DCKC(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  DCKC(dzalloc(&c->actor, ANet::PP)); DCKC(dzalloc(&c->actor_tgt, ANet::PP)); DCKC(dzalloc(&c->am, ANet::P)); DCKC(dzalloc(&c->av, ANet::P));
  DCKC(dzalloc(&c->critic, CNet::PP)); DCKC(dzalloc(&c->critic_tgt, CNet::PP)); DCKC(dzalloc(&c->cm, CNet::P)); DCKC(dzalloc(&c->cv, CNet::P));
  DCKC(dzalloc(&c->env_state, 2 * N)); DCKC(dzalloc(&c->env_t, N)); DCKC(dzalloc(&c->ep_ret, N)); DCKC(dzalloc(&c->ep_len, N));
  DCKC(dzalloc(&c->resets, N));
  DCKC(dzalloc(&c->b_obs, DD_D * C)); DCKC(dzalloc(&c->b_next, DD_D * C)); DCKC(dzalloc(&c->b_act, C)); DCKC(dzalloc(&c->b_rew, C));
  DCKC(dzalloc(&c->b_term, C)); DCKC(dzalloc(&c->dev, 1));
  DCKC(dzalloc(&c->scratch, SCRATCH_FLOATS)); DCKC(dzalloc(&c->loss_part, LF_MAX_BLOCKS));
  DCKC(set_smem_attrs());
#undef DCKC
  *out = c;
  return CRL_OK;
}

extern "C" CRL_API int crl_ddpg_destroy(crl_ddpg_ctx* c) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  cudaSetDevice(c->cfg.device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  void* ptrs[] = {c->actor, c->critic, c->actor_tgt, c->critic_tgt, c->am, c->av, c->cm, c->cv, c->env_state, c->env_t, c->ep_ret,
                  c->ep_len, c->resets, c->b_obs, c->b_next, c->b_act, c->b_rew, c->b_term, c->dev, c->scratch, c->loss_part};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
  return CRL_OK;
}

extern "C" CRL_API int crl_ddpg_set_params(crl_ddpg_ctx* c, const float* actor, int32_t n_actor, const float* critic, int32_t n_critic) {
  if (!c || !actor || !critic) return dfail(CRL_ERR_INVALID, "NULL argument");
  if (n_actor != ANet::P || n_critic != CNet::P) return dfail(CRL_ERR_INVALID, "DDPG parameter vectors must have 4481 (actor) and 4545 (critic) floats");
  DCK(cudaSetDevice(c->cfg.device));
  DCK(cudaMemcpyAsync(c->actor, actor, sizeof(float) * ANet::P, cudaMemcpyHostToDevice, c->stream));
  DCK(cudaMemcpyAsync(c->critic, critic, sizeof(float) * CNet::P, cudaMemcpyHostToDevice, c->stream));
  DCK(cudaMemcpyAsync(c->actor_tgt, c->actor, sizeof(float) * ANet::P, cudaMemcpyDeviceToDevice, c->stream));
  DCK(cudaMemcpyAsync(c->critic_tgt, c->critic, sizeof(float) * CNet::P, cudaMemcpyDeviceToDevice, c->stream));
  DCK(cudaMemsetAsync(c->am, 0, sizeof(float) * ANet::P, c->stream)); DCK(cudaMemsetAsync(c->av, 0, sizeof(float) * ANet::P, c->stream));
  DCK(cudaMemsetAsync(c->cm, 0, sizeof(float) * CNet::P, c->stream)); DCK(cudaMemsetAsync(c->cv, 0, sizeof(float) * CNet::P, c->stream));
  DdpgDev d;
  memset(&d, 0, sizeof(d));
  DCK(cudaMemcpyAsync(c->dev, &d, sizeof(d), cudaMemcpyHostToDevice, c->stream));
  DCK(cudaStreamSynchronize(c->stream));
  c->abp1 = c->cbp1 = 0.9; c->abp2 = c->cbp2 = 0.999;
  c->params_set = true;
  return CRL_OK;
}

extern "C" CRL_API int crl_ddpg_get_params(crl_ddpg_ctx* c, float* actor, float* critic, float* actor_target, float* critic_target) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  DCK(cudaSetDevice(c->cfg.device));
  if (actor) DCK(cudaMemcpyAsync(actor, c->actor, sizeof(float) * ANet::P, cudaMemcpyDeviceToHost, c->stream));
  if (critic) DCK(cudaMemcpyAsync(critic, c->critic, sizeof(float) * CNet::P, cudaMemcpyDeviceToHost, c->stream));
  if (actor_target) DCK(cudaMemcpyAsync(actor_target, c->actor_tgt, sizeof(float) * ANet::P, cudaMemcpyDeviceToHost, c->stream));
  if (critic_target) DCK(cudaMemcpyAsync(critic_target, c->critic_tgt, sizeof(float) * CNet::P, cudaMemcpyDeviceToHost, c->stream));
  DCK(cudaStreamSynchronize(c->stream));
  return CRL_OK;
}

extern "C" CRL_API int crl_ddpg_get_adam_state(crl_ddpg_ctx* c, float* actor_m, float* actor_v, float* critic_m, float* critic_v,
                                               double* beta_pow) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  DCK(cudaSetDevice(c->cfg.device));
  if (actor_m) DCK(cudaMemcpyAsync(actor_m, c->am, sizeof(float) * ANet::P, cudaMemcpyDeviceToHost, c->stream));
  if (actor_v) DCK(cudaMemcpyAsync(actor_v, c->av, sizeof(float) * ANet::P, cudaMemcpyDeviceToHost, c->stream));
  if (critic_m) DCK(cudaMemcpyAsync(critic_m, c->cm, sizeof(float) * CNet::P, cudaMemcpyDeviceToHost, c->stream));
  if (critic_v) DCK(cudaMemcpyAsync(critic_v, c->cv, sizeof(float) * CNet::P, cudaMemcpyDeviceToHost, c->stream));
  DCK(cudaStreamSynchronize(c->stream));
  if (beta_pow) { beta_pow[0] = c->abp1; beta_pow[1] = c->abp2; beta_pow[2] = c->cbp1; beta_pow[3] = c->cbp2; }
  return CRL_OK;
}

extern "C" CRL_API int crl_ddpg_reset(crl_ddpg_ctx* c) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  DCK(cudaSetDevice(c->cfg.device));
  const int N = c->cfg.num_envs;
  ddpg_reset_kernel<<<(N + 127) / 128, 128, 0, c->stream>>>(N, c->cfg.seed, c->env_state, c->env_t, c->ep_ret, c->ep_len, c->resets);
  DCK(cudaGetLastError());
  c->size = 0; c->ptr = 0; c->it = 0; c->learn_steps = 0; c->actor_steps = 0;   /* launches is a lifetime counter */
  c->reset_done = true;
  return CRL_OK;
}

// One acting launch for every iteration from k up to (and including) the next learning step: the parameters are constant
// in between. Bounded by `iterations`, by ACT_MAX_STEPS and by the ring capacity (steps of one launch must not share a
// slot). Advances k and the iteration, ring and launch counters; `learn` is set when the last iteration learns.
// `actor` and `kernel` are DDPG's (ddpg_act_kernel, ACT_SMEM) or SAC's (sac_act_kernel, SACT_SMEM).
static int act_launch(crl_ddpg_ctx* c, const float* actor, void (*kernel)(ActArgs), size_t smem, int64_t iterations, int64_t& k,
                      bool& learn) {
  const crl_ddpg_config& g = c->cfg;
  const int N = g.num_envs, C = g.buffer_size;
  ActArgs a;
  a.actor = actor; a.env_state = c->env_state; a.env_t = c->env_t; a.ep_ret = c->ep_ret; a.ep_len = c->ep_len; a.resets = c->resets;
  a.b_obs = c->b_obs; a.b_next = c->b_next; a.b_act = c->b_act; a.b_rew = c->b_rew; a.b_term = c->b_term; a.dev = c->dev;
  a.seed = g.seed; a.it0 = (unsigned long long)(c->it + 1); a.learning_starts = g.learning_starts;
  a.sigma = (float)(g.exploration_noise * (double)DD_MAX_TORQUE);
  a.N = N; a.C = C; a.ptr = c->ptr; a.max_steps = g.max_episode_steps;
  int ns = 0;
  learn = false;
  while (k < iterations && ns < ACT_MAX_STEPS && (long long)(ns + 1) * N <= (long long)C && !learn) {
    c->it += 1;
    k += 1;
    ns += 1;
    c->ptr = (int)(((long long)c->ptr + N) % C);
    c->size = c->size + N > C ? C : c->size + N;
    const long long gs = c->it * (long long)N;
    learn = gs > (long long)g.learning_starts && c->it % g.train_freq == 0 && c->size >= g.batch_size;
  }
  a.n_steps = ns;
  kernel<<<(N + ACT_E - 1) / ACT_E, ACT_T, smem, c->stream>>>(a);
  DCK(cudaGetLastError());
  c->launches += 1;
  return CRL_OK;
}

// the learning step's batch: Philox stream 6 keyed by the learning-step index, over the ring's current size
static LearnArgs learn_args(const crl_ddpg_ctx* c, const Scratch& s) {
  LearnArgs l;
  memset(&l, 0, sizeof(l));
  l.actor = c->actor; l.critic = c->critic; l.actor_tgt = c->actor_tgt; l.critic_tgt = c->critic_tgt;
  l.b_obs = c->b_obs; l.b_next = c->b_next; l.b_act = c->b_act; l.b_rew = c->b_rew; l.b_term = c->b_term;
  l.seed = c->cfg.seed; l.learn_step = (unsigned long long)c->learn_steps; l.gamma = c->cfg.gamma; l.B = c->cfg.batch_size;
  l.size = c->size; l.s = s; l.loss_part = c->loss_part;
  return l;
}

// every policy_frequency-th learning step, on the same batch and against the critic just updated: the actor's step,
// then Polyak averaging of the actor's and the critic's targets
static int actor_step(crl_ddpg_ctx* c, const LearnArgs& l) {
  UpdArgs u;
  memset(&u, 0, sizeof(u));
  u.params = c->actor; u.m = c->am; u.v = c->av; u.loss_out = &c->dev->actor_loss; u.lr = c->cfg.lr; u.bp1 = c->abp1; u.bp2 = c->abp2;
  DCK(launch_net_step(false, l, u, c->stream));
  ddpg_polyak_kernel<<<(ANet::P + CNet::P + 255) / 256, 256, 0, c->stream>>>(c->actor, c->actor_tgt, c->critic, c->critic_tgt, c->cfg.tau);
  DCK(cudaGetLastError());
  c->abp1 *= 0.9; c->abp2 *= 0.999;
  c->launches += 3;
  c->actor_steps += 1;
  return CRL_OK;
}

extern "C" CRL_API int crl_ddpg_run(crl_ddpg_ctx* c, int64_t iterations, crl_ddpg_stats* stats) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  if (iterations < 0) return dfail(CRL_ERR_INVALID, "iterations must be >= 0");
  if (!c->params_set) return dfail(CRL_ERR_STATE, "crl_ddpg_run called before crl_ddpg_set_params");
  if (!c->reset_done) return dfail(CRL_ERR_STATE, "crl_ddpg_run called before crl_ddpg_reset");
  DCK(cudaSetDevice(c->cfg.device));
  // per-call episode aggregate: clear the three accumulators, keep the last losses
  DCK(cudaMemsetAsync(&c->dev->sum_return, 0, sizeof(double) * 2 + sizeof(unsigned long long), c->stream));
  const Scratch s = carve(c->scratch);
  int64_t k = 0;
  while (k < iterations) {
    bool learn = false;
    if (int rc = act_launch(c, c->actor, ddpg_act_kernel, ACT_SMEM, iterations, k, learn)) return rc;
    if (!learn) continue;
    const LearnArgs l = learn_args(c, s);
    UpdArgs u;
    memset(&u, 0, sizeof(u));
    u.params = c->critic; u.m = c->cm; u.v = c->cv; u.loss_out = &c->dev->critic_loss; u.lr = c->cfg.lr; u.bp1 = c->cbp1; u.bp2 = c->cbp2;
    DCK(launch_net_step(true, l, u, c->stream));
    c->cbp1 *= 0.9; c->cbp2 *= 0.999;
    c->launches += 2;
    c->learn_steps += 1;
    if (c->learn_steps % c->cfg.policy_frequency == 0)
      if (int rc = actor_step(c, l)) return rc;
  }
  if (stats) {
    DdpgDev d;
    DCK(cudaMemcpyAsync(&d, c->dev, sizeof(d), cudaMemcpyDeviceToHost, c->stream));
    DCK(cudaStreamSynchronize(c->stream));
    stats->critic_loss = d.critic_loss; stats->actor_loss = d.actor_loss; stats->sum_return = d.sum_return;
    stats->sum_length = d.sum_length; stats->episodes = (int64_t)d.episodes; stats->learn_steps = c->learn_steps;
    stats->actor_steps = c->actor_steps; stats->iterations = c->it; stats->kernel_launches = c->launches;
  }
  return CRL_OK;
}

extern "C" CRL_API int crl_ddpg_read_buffer(crl_ddpg_ctx* c, float* obs, float* action, float* reward, float* next_obs,
                                            uint8_t* terminal, int32_t* size, int32_t* ptr) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  DCK(cudaSetDevice(c->cfg.device));
  const size_t C = c->cfg.buffer_size;
  if (obs) DCK(cudaMemcpyAsync(obs, c->b_obs, C * DD_D * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  if (next_obs) DCK(cudaMemcpyAsync(next_obs, c->b_next, C * DD_D * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  if (action) DCK(cudaMemcpyAsync(action, c->b_act, C * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  if (reward) DCK(cudaMemcpyAsync(reward, c->b_rew, C * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  if (terminal) DCK(cudaMemcpyAsync(terminal, c->b_term, C, cudaMemcpyDeviceToHost, c->stream));
  DCK(cudaStreamSynchronize(c->stream));
  if (size) *size = c->size;
  if (ptr) *ptr = c->ptr;
  return CRL_OK;
}

// ---- raw entry points (device pointers)
static int ddpg_raw_device_check() {
  int dev = 0;
  DCK(cudaGetDevice(&dev));
  if (int rc = ddpg_device_check(dev)) return rc;
  DCK(set_smem_attrs());
  return CRL_OK;
}

extern "C" CRL_API int crl_ddpg_forward_raw(const float* actor, const float* critic, const float* obs, const float* action,
                                            float* mu_out, float* q_out, int64_t n, void* stream) {
  if (n < 0 || (n > 0 && (!actor || !critic || !obs || !action || !mu_out || !q_out))) return dfail(CRL_ERR_INVALID, "NULL argument or n < 0");
  if (((uintptr_t)actor | (uintptr_t)critic) % 16) return dfail(CRL_ERR_INVALID, "actor and critic must be 16-byte aligned");
  if (n == 0) return CRL_OK;
  if (int rc = ddpg_raw_device_check()) return rc;
  const int64_t grid = (n + ACT_E - 1) / ACT_E;
  if (grid > 0x7fffffff) return dfail(CRL_ERR_INVALID, "n too large");
  ddpg_forward_raw_kernel<<<(unsigned)grid, ACT_T, FWD_RAW_SMEM, (cudaStream_t)stream>>>(actor, critic, obs, action, mu_out, q_out, n);
  DCK(cudaGetLastError());
  return CRL_OK;
}

// one net's step of the learning step on rows 0..B-1 (nothing sampled), gradient out instead of Adam
static int ddpg_loss_raw(bool critic, LearnArgs& l, float* grads_out, double* loss_out, cudaStream_t s) {
  if (l.B < 1 || l.B > LEARN_B) return dfail(CRL_ERR_INVALID, "B must be in [1, 256]");
  if (int rc = ddpg_raw_device_check()) return rc;
  float* scratch = nullptr;
  double* dscratch = nullptr;
  DCK(cudaMalloc(reinterpret_cast<void**>(&scratch), SCRATCH_FLOATS * sizeof(float)));
  if (cudaMalloc(reinterpret_cast<void**>(&dscratch), LF_MAX_BLOCKS * sizeof(double)) != cudaSuccess) {
    cudaFree(scratch);
    return dfail(CRL_ERR_CUDA, "cudaMalloc failed (crl_ddpg loss raw)");
  }
  l.in_order = 1; l.size = l.B; l.s = carve(scratch); l.loss_part = dscratch;
  UpdArgs u;
  memset(&u, 0, sizeof(u));
  u.grads_out = grads_out; u.loss_out = loss_out;
  cudaError_t e = launch_net_step(critic, l, u, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);   // the scratch is freed below
  cudaFree(scratch);
  cudaFree(dscratch);
  if (e != cudaSuccess) return dfail(CRL_ERR_CUDA, std::string("crl_ddpg loss raw failed: ") + cudaGetErrorString(e));
  return CRL_OK;
}

extern "C" CRL_API int crl_ddpg_critic_loss_raw(const float* actor_target, const float* critic, const float* critic_target, int32_t B,
                                                const float* obs, const float* action, const float* reward, const float* next_obs,
                                                const uint8_t* terminal, double gamma, float* grads_out, double* loss_out, void* stream) {
  if (!actor_target || !critic || !critic_target || !obs || !action || !reward || !next_obs || !terminal || !grads_out || !loss_out)
    return dfail(CRL_ERR_INVALID, "NULL argument");
  if (((uintptr_t)actor_target | (uintptr_t)critic | (uintptr_t)critic_target) % 16)
    return dfail(CRL_ERR_INVALID, "parameter vectors must be 16-byte aligned");
  LearnArgs l;
  memset(&l, 0, sizeof(l));
  l.actor_tgt = actor_target; l.critic = critic; l.critic_tgt = critic_target;
  l.b_obs = obs; l.b_act = action; l.b_rew = reward; l.b_next = next_obs; l.b_term = terminal; l.gamma = gamma; l.B = B;
  return ddpg_loss_raw(true, l, grads_out, loss_out, (cudaStream_t)stream);
}

extern "C" CRL_API int crl_ddpg_actor_loss_raw(const float* actor, const float* critic, int32_t B, const float* obs, float* grads_out,
                                               double* loss_out, void* stream) {
  if (!actor || !critic || !obs || !grads_out || !loss_out) return dfail(CRL_ERR_INVALID, "NULL argument");
  if (((uintptr_t)actor | (uintptr_t)critic) % 16) return dfail(CRL_ERR_INVALID, "parameter vectors must be 16-byte aligned");
  LearnArgs l;
  memset(&l, 0, sizeof(l));
  l.actor = actor; l.critic = critic; l.b_obs = obs; l.B = B;
  return ddpg_loss_raw(false, l, grads_out, loss_out, (cudaStream_t)stream);
}

// ---- TD3 (include/cleanrl_td3.h). The DDPG context carries everything the two share: envs, ring, actor, qf1 (as the
// critic), the actor's and qf1's targets, their Adam state and the counters. Both critics share one step count, so
// qf2's Adam uses the critic's beta powers.
struct crl_td3_ctx {
  crl_ddpg_ctx* d;
  crl_td3_config cfg;
  float *critic2, *critic2_tgt, *c2m, *c2v;
  float* scratch2;
  double *loss_part2, *qf2_loss;
};

static crl_ddpg_config td3_ddpg_config(const crl_td3_config& t) {
  crl_ddpg_config g;
  memset(&g, 0, sizeof(g));
  g.struct_size = (int32_t)sizeof(crl_ddpg_config);
  g.num_envs = t.num_envs; g.buffer_size = t.buffer_size; g.learning_starts = t.learning_starts; g.batch_size = t.batch_size;
  g.train_freq = t.train_freq; g.policy_frequency = t.policy_frequency; g.max_episode_steps = t.max_episode_steps;
  g.device = t.device; g.gamma = t.gamma; g.tau = t.tau; g.lr = t.lr; g.exploration_noise = t.exploration_noise; g.seed = t.seed;
  return g;
}

static int td3_validate_noise(double policy_noise, double noise_clip) {
  if (!(policy_noise >= 0.0 && isfinite(policy_noise)) || !(noise_clip >= 0.0 && isfinite(noise_clip)))
    return dfail(CRL_ERR_INVALID, "policy_noise and noise_clip must be finite and >= 0");
  return CRL_OK;
}

extern "C" CRL_API int crl_td3_destroy(crl_td3_ctx* c) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  if (c->d) {
    cudaSetDevice(c->cfg.device);
    cudaStreamSynchronize(c->d->stream);
  }
  void* ptrs[] = {c->critic2, c->critic2_tgt, c->c2m, c->c2v, c->scratch2, c->loss_part2, c->qf2_loss};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (c->d) crl_ddpg_destroy(c->d);
  delete c;
  return CRL_OK;
}

extern "C" CRL_API int crl_td3_create(const crl_td3_config* cfg, crl_td3_ctx** out) {
  if (!cfg || !out) return dfail(CRL_ERR_INVALID, "NULL argument");
  *out = nullptr;
  if (cfg->struct_size != (int32_t)sizeof(crl_td3_config)) return dfail(CRL_ERR_INVALID, "crl_td3_config.struct_size mismatch");
  if (int rc = td3_validate_noise(cfg->policy_noise, cfg->noise_clip)) return rc;
  const crl_ddpg_config g = td3_ddpg_config(*cfg);
  if (int rc = ddpg_validate(&g)) return rc;
  crl_ddpg_ctx* d = nullptr;
  if (int rc = crl_ddpg_create(&g, &d)) return rc;   // checks the device, then allocates
  crl_td3_ctx* c = new crl_td3_ctx();
  memset(c, 0, sizeof(*c));
  c->d = d;
  c->cfg = *cfg;
#define TCKC(call)                                                                                            \
  do {                                                                                                        \
    cudaError_t e__ = (call);                                                                                 \
    if (e__ != cudaSuccess) {                                                                                 \
      crl_td3_destroy(c);                                                                                     \
      return dfail(CRL_ERR_CUDA, std::string(#call) + " failed: " + cudaGetErrorString(e__) + " (ddpg.cu)"); \
    }                                                                                                         \
  } while (0)
  TCKC(dzalloc(&c->critic2, CNet::PP)); TCKC(dzalloc(&c->critic2_tgt, CNet::PP)); TCKC(dzalloc(&c->c2m, CNet::P));
  TCKC(dzalloc(&c->c2v, CNet::P)); TCKC(dzalloc(&c->scratch2, SCRATCH_FLOATS)); TCKC(dzalloc(&c->loss_part2, LF_MAX_BLOCKS));
  TCKC(dzalloc(&c->qf2_loss, 1));
#undef TCKC
  *out = c;
  return CRL_OK;
}

extern "C" CRL_API int crl_td3_set_params(crl_td3_ctx* c, const float* actor, int32_t n_actor, const float* qf1, int32_t n_qf1,
                                          const float* qf2, int32_t n_qf2) {
  if (!c || !actor || !qf1 || !qf2) return dfail(CRL_ERR_INVALID, "NULL argument");
  if (n_actor != ANet::P || n_qf1 != CNet::P || n_qf2 != CNet::P)
    return dfail(CRL_ERR_INVALID, "TD3 parameter vectors must have 4481 (actor) and 4545 (qf1, qf2) floats");
  if (int rc = crl_ddpg_set_params(c->d, actor, n_actor, qf1, n_qf1)) return rc;
  c->d->params_set = false;   // until qf2 is in place as well
  const cudaStream_t s = c->d->stream;
  DCK(cudaMemcpyAsync(c->critic2, qf2, sizeof(float) * CNet::P, cudaMemcpyHostToDevice, s));
  DCK(cudaMemcpyAsync(c->critic2_tgt, c->critic2, sizeof(float) * CNet::P, cudaMemcpyDeviceToDevice, s));
  DCK(cudaMemsetAsync(c->c2m, 0, sizeof(float) * CNet::P, s)); DCK(cudaMemsetAsync(c->c2v, 0, sizeof(float) * CNet::P, s));
  DCK(cudaMemsetAsync(c->qf2_loss, 0, sizeof(double), s));
  DCK(cudaStreamSynchronize(s));
  c->d->params_set = true;
  return CRL_OK;
}

extern "C" CRL_API int crl_td3_get_params(crl_td3_ctx* c, float* actor, float* qf1, float* qf2, float* actor_target, float* qf1_target,
                                          float* qf2_target) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  if (int rc = crl_ddpg_get_params(c->d, actor, qf1, actor_target, qf1_target)) return rc;
  if (qf2) DCK(cudaMemcpyAsync(qf2, c->critic2, sizeof(float) * CNet::P, cudaMemcpyDeviceToHost, c->d->stream));
  if (qf2_target) DCK(cudaMemcpyAsync(qf2_target, c->critic2_tgt, sizeof(float) * CNet::P, cudaMemcpyDeviceToHost, c->d->stream));
  DCK(cudaStreamSynchronize(c->d->stream));
  return CRL_OK;
}

extern "C" CRL_API int crl_td3_get_adam_state(crl_td3_ctx* c, float* actor_m, float* actor_v, float* qf1_m, float* qf1_v, float* qf2_m,
                                              float* qf2_v, double* beta_pow) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  if (int rc = crl_ddpg_get_adam_state(c->d, actor_m, actor_v, qf1_m, qf1_v, beta_pow)) return rc;
  if (qf2_m) DCK(cudaMemcpyAsync(qf2_m, c->c2m, sizeof(float) * CNet::P, cudaMemcpyDeviceToHost, c->d->stream));
  if (qf2_v) DCK(cudaMemcpyAsync(qf2_v, c->c2v, sizeof(float) * CNet::P, cudaMemcpyDeviceToHost, c->d->stream));
  DCK(cudaStreamSynchronize(c->d->stream));
  return CRL_OK;
}

extern "C" CRL_API int crl_td3_reset(crl_td3_ctx* c) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  return crl_ddpg_reset(c->d);
}

extern "C" CRL_API int crl_td3_run(crl_td3_ctx* t, int64_t iterations, crl_td3_stats* stats) {
  if (!t) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  if (iterations < 0) return dfail(CRL_ERR_INVALID, "iterations must be >= 0");
  crl_ddpg_ctx* c = t->d;
  if (!c->params_set) return dfail(CRL_ERR_STATE, "crl_td3_run called before crl_td3_set_params");
  if (!c->reset_done) return dfail(CRL_ERR_STATE, "crl_td3_run called before crl_td3_reset");
  DCK(cudaSetDevice(c->cfg.device));
  DCK(cudaMemsetAsync(&c->dev->sum_return, 0, sizeof(double) * 2 + sizeof(unsigned long long), c->stream));
  const Scratch s1 = carve(c->scratch), s2 = carve(t->scratch2);
  int64_t k = 0;
  while (k < iterations) {
    bool learn = false;
    if (int rc = act_launch(c, c->actor, ddpg_act_kernel, ACT_SMEM, iterations, k, learn)) return rc;
    if (!learn) continue;
    Td3Args a;
    memset(&a, 0, sizeof(a));
    a.l = learn_args(c, s1);
    a.critic2 = t->critic2; a.critic2_tgt = t->critic2_tgt; a.s2 = s2; a.loss_part2 = t->loss_part2;
    a.policy_noise = (float)t->cfg.policy_noise; a.noise_clip = (float)t->cfg.noise_clip;
    UpdArgs u1, u2;
    memset(&u1, 0, sizeof(u1));
    u1.lr = c->cfg.lr; u1.bp1 = c->cbp1; u1.bp2 = c->cbp2;
    u2 = u1;
    u1.params = c->critic; u1.m = c->cm; u1.v = c->cv; u1.loss_out = &c->dev->critic_loss;
    u2.params = t->critic2; u2.m = t->c2m; u2.v = t->c2v; u2.loss_out = t->qf2_loss;
    DCK(launch_td3_critic_step(a, u1, u2, c->stream));
    c->cbp1 *= 0.9; c->cbp2 *= 0.999;
    c->launches += 2;
    c->learn_steps += 1;
    if (c->learn_steps % c->cfg.policy_frequency == 0) {
      if (int rc = actor_step(c, a.l)) return rc;   // actor against qf1, Polyak of actor' and qf1'
      td3_polyak_kernel<<<(CNet::P + 255) / 256, 256, 0, c->stream>>>(t->critic2, t->critic2_tgt, c->cfg.tau);
      DCK(cudaGetLastError());
      c->launches += 1;
    }
  }
  if (stats) {
    DdpgDev d;
    double q2 = 0.0;
    DCK(cudaMemcpyAsync(&d, c->dev, sizeof(d), cudaMemcpyDeviceToHost, c->stream));
    DCK(cudaMemcpyAsync(&q2, t->qf2_loss, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    DCK(cudaStreamSynchronize(c->stream));
    stats->qf1_loss = d.critic_loss; stats->qf2_loss = q2; stats->actor_loss = d.actor_loss; stats->sum_return = d.sum_return;
    stats->sum_length = d.sum_length; stats->episodes = (int64_t)d.episodes; stats->learn_steps = c->learn_steps;
    stats->actor_steps = c->actor_steps; stats->iterations = c->it; stats->kernel_launches = c->launches;
  }
  return CRL_OK;
}

extern "C" CRL_API int crl_td3_read_buffer(crl_td3_ctx* c, float* obs, float* action, float* reward, float* next_obs, uint8_t* terminal,
                                           int32_t* size, int32_t* ptr) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  return crl_ddpg_read_buffer(c->d, obs, action, reward, next_obs, terminal, size, ptr);
}

extern "C" CRL_API int crl_td3_critic_loss_raw(const float* actor_target, const float* qf1, const float* qf2, const float* qf1_target,
                                               const float* qf2_target, int32_t B, const float* obs, const float* action,
                                               const float* reward, const float* next_obs, const uint8_t* terminal, double gamma,
                                               double policy_noise, double noise_clip, uint64_t seed, uint64_t learn_step,
                                               float* qf1_grads_out, float* qf2_grads_out, double* qf1_loss_out,
                                               double* qf2_loss_out, void* stream) {
  if (!actor_target || !qf1 || !qf2 || !qf1_target || !qf2_target || !obs || !action || !reward || !next_obs || !terminal ||
      !qf1_grads_out || !qf2_grads_out || !qf1_loss_out || !qf2_loss_out)
    return dfail(CRL_ERR_INVALID, "NULL argument");
  if (((uintptr_t)actor_target | (uintptr_t)qf1 | (uintptr_t)qf2 | (uintptr_t)qf1_target | (uintptr_t)qf2_target) % 16)
    return dfail(CRL_ERR_INVALID, "parameter vectors must be 16-byte aligned");
  if (B < 1 || B > LEARN_B) return dfail(CRL_ERR_INVALID, "B must be in [1, 256]");
  if (int rc = td3_validate_noise(policy_noise, noise_clip)) return rc;
  if (int rc = ddpg_raw_device_check()) return rc;
  float* scratch = nullptr;
  double* dscratch = nullptr;
  DCK(cudaMalloc(reinterpret_cast<void**>(&scratch), 2 * SCRATCH_FLOATS * sizeof(float)));
  if (cudaMalloc(reinterpret_cast<void**>(&dscratch), 2 * LF_MAX_BLOCKS * sizeof(double)) != cudaSuccess) {
    cudaFree(scratch);
    return dfail(CRL_ERR_CUDA, "cudaMalloc failed (crl_td3_critic_loss_raw)");
  }
  Td3Args a;
  memset(&a, 0, sizeof(a));
  LearnArgs& l = a.l;
  l.actor_tgt = actor_target; l.critic = qf1; l.critic_tgt = qf1_target;
  l.b_obs = obs; l.b_act = action; l.b_rew = reward; l.b_next = next_obs; l.b_term = terminal;
  l.seed = seed; l.learn_step = learn_step; l.gamma = gamma; l.B = B; l.size = B; l.in_order = 1;
  l.s = carve(scratch); l.loss_part = dscratch;
  a.critic2 = qf2; a.critic2_tgt = qf2_target; a.s2 = carve(scratch + SCRATCH_FLOATS); a.loss_part2 = dscratch + LF_MAX_BLOCKS;
  a.policy_noise = (float)policy_noise; a.noise_clip = (float)noise_clip;
  UpdArgs u1, u2;
  memset(&u1, 0, sizeof(u1));
  u2 = u1;
  u1.grads_out = qf1_grads_out; u1.loss_out = qf1_loss_out;
  u2.grads_out = qf2_grads_out; u2.loss_out = qf2_loss_out;
  const cudaStream_t s = (cudaStream_t)stream;
  cudaError_t e = launch_td3_critic_step(a, u1, u2, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);   // the scratch is freed below
  cudaFree(scratch);
  cudaFree(dscratch);
  if (e != cudaSuccess) return dfail(CRL_ERR_CUDA, std::string("crl_td3_critic_loss_raw failed: ") + cudaGetErrorString(e));
  return CRL_OK;
}

// ---- SAC (include/cleanrl_sac.h). The DDPG context carries the envs, the ring, qf1 (as the critic), qf1' and qf1's
// Adam state, the counters and both optimisers' beta powers: the critics share the critic's, and the actor and log_alpha
// the actor's. Its own actor buffers are not used: SAC's 4,546-float actor lives here. actor_steps counts actor iterations.
struct crl_sac_ctx {
  crl_ddpg_ctx* d;
  crl_sac_config cfg;
  float *actor, *am, *av;
  float *critic2, *critic2_tgt, *c2m, *c2v;
  float* scratch2;     // qf2's scratch in the critic step, the actor's in the actor step
  double* loss_part2;
  SacDev* sdev;
};

static int sac_validate(const crl_sac_config* cfg) {
  if (cfg->struct_size != (int32_t)sizeof(crl_sac_config)) return dfail(CRL_ERR_INVALID, "crl_sac_config.struct_size mismatch");
  if (!(cfg->policy_lr > 0.0 && isfinite(cfg->policy_lr)) || !(cfg->q_lr > 0.0 && isfinite(cfg->q_lr)))
    return dfail(CRL_ERR_INVALID, "policy_lr and q_lr must be finite and > 0");
  if (!(cfg->alpha >= 0.0 && isfinite(cfg->alpha))) return dfail(CRL_ERR_INVALID, "alpha must be finite and >= 0");
  if (cfg->target_network_frequency < 1) return dfail(CRL_ERR_INVALID, "target_network_frequency must be >= 1");
  if (cfg->autotune != 0 && cfg->autotune != 1) return dfail(CRL_ERR_INVALID, "autotune must be 0 or 1");
  return CRL_OK;
}

static crl_ddpg_config sac_ddpg_config(const crl_sac_config& t) {
  crl_ddpg_config g;
  memset(&g, 0, sizeof(g));
  g.struct_size = (int32_t)sizeof(crl_ddpg_config);
  g.num_envs = t.num_envs; g.buffer_size = t.buffer_size; g.learning_starts = t.learning_starts; g.batch_size = t.batch_size;
  g.train_freq = t.train_freq; g.policy_frequency = t.policy_frequency; g.max_episode_steps = t.max_episode_steps;
  g.device = t.device; g.gamma = t.gamma; g.tau = t.tau; g.lr = t.q_lr; g.exploration_noise = 0.0; g.seed = t.seed;
  return g;
}

extern "C" CRL_API int crl_sac_destroy(crl_sac_ctx* c) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  if (c->d) {
    cudaSetDevice(c->cfg.device);
    cudaStreamSynchronize(c->d->stream);
  }
  void* ptrs[] = {c->actor, c->am, c->av, c->critic2, c->critic2_tgt, c->c2m, c->c2v, c->scratch2, c->loss_part2, c->sdev};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (c->d) crl_ddpg_destroy(c->d);
  delete c;
  return CRL_OK;
}

extern "C" CRL_API int crl_sac_create(const crl_sac_config* cfg, crl_sac_ctx** out) {
  if (!cfg || !out) return dfail(CRL_ERR_INVALID, "NULL argument");
  *out = nullptr;
  if (int rc = sac_validate(cfg)) return rc;
  const crl_ddpg_config g = sac_ddpg_config(*cfg);
  if (int rc = ddpg_validate(&g)) return rc;
  crl_ddpg_ctx* d = nullptr;
  if (int rc = crl_ddpg_create(&g, &d)) return rc;   // checks the device, then allocates
  crl_sac_ctx* c = new crl_sac_ctx();
  memset(c, 0, sizeof(*c));
  c->d = d;
  c->cfg = *cfg;
#define SCKC(call)                                                                                            \
  do {                                                                                                        \
    cudaError_t e__ = (call);                                                                                 \
    if (e__ != cudaSuccess) {                                                                                 \
      crl_sac_destroy(c);                                                                                     \
      return dfail(CRL_ERR_CUDA, std::string(#call) + " failed: " + cudaGetErrorString(e__) + " (ddpg.cu)"); \
    }                                                                                                         \
  } while (0)
  SCKC(dzalloc(&c->actor, SNet::PP)); SCKC(dzalloc(&c->am, SNet::P)); SCKC(dzalloc(&c->av, SNet::P));
  SCKC(dzalloc(&c->critic2, CNet::PP)); SCKC(dzalloc(&c->critic2_tgt, CNet::PP)); SCKC(dzalloc(&c->c2m, CNet::P));
  SCKC(dzalloc(&c->c2v, CNet::P)); SCKC(dzalloc(&c->scratch2, SAC_SCRATCH_FLOATS)); SCKC(dzalloc(&c->loss_part2, LF_MAX_BLOCKS));
  SCKC(dzalloc(&c->sdev, 1));
#undef SCKC
  *out = c;
  return CRL_OK;
}

extern "C" CRL_API int crl_sac_set_params(crl_sac_ctx* t, const float* actor, int32_t n_actor, const float* qf1, int32_t n_qf1,
                                          const float* qf2, int32_t n_qf2) {
  if (!t || !actor || !qf1 || !qf2) return dfail(CRL_ERR_INVALID, "NULL argument");
  if (n_actor != SNet::P || n_qf1 != CNet::P || n_qf2 != CNet::P)
    return dfail(CRL_ERR_INVALID, "SAC parameter vectors must have 4546 (actor) and 4545 (qf1, qf2) floats");
  crl_ddpg_ctx* c = t->d;
  DCK(cudaSetDevice(c->cfg.device));
  const cudaStream_t s = c->stream;
  c->params_set = false;
  DCK(cudaMemcpyAsync(t->actor, actor, sizeof(float) * SNet::P, cudaMemcpyHostToDevice, s));
  DCK(cudaMemcpyAsync(c->critic, qf1, sizeof(float) * CNet::P, cudaMemcpyHostToDevice, s));
  DCK(cudaMemcpyAsync(c->critic_tgt, c->critic, sizeof(float) * CNet::P, cudaMemcpyDeviceToDevice, s));
  DCK(cudaMemcpyAsync(t->critic2, qf2, sizeof(float) * CNet::P, cudaMemcpyHostToDevice, s));
  DCK(cudaMemcpyAsync(t->critic2_tgt, t->critic2, sizeof(float) * CNet::P, cudaMemcpyDeviceToDevice, s));
  DCK(cudaMemsetAsync(t->am, 0, sizeof(float) * SNet::P, s)); DCK(cudaMemsetAsync(t->av, 0, sizeof(float) * SNet::P, s));
  DCK(cudaMemsetAsync(c->cm, 0, sizeof(float) * CNet::P, s)); DCK(cudaMemsetAsync(c->cv, 0, sizeof(float) * CNet::P, s));
  DCK(cudaMemsetAsync(t->c2m, 0, sizeof(float) * CNet::P, s)); DCK(cudaMemsetAsync(t->c2v, 0, sizeof(float) * CNet::P, s));
  DdpgDev d;
  memset(&d, 0, sizeof(d));
  SacDev sd;
  memset(&sd, 0, sizeof(sd));
  sd.alpha = t->cfg.autotune ? 1.0 : t->cfg.alpha;
  DCK(cudaMemcpyAsync(c->dev, &d, sizeof(d), cudaMemcpyHostToDevice, s));
  DCK(cudaMemcpyAsync(t->sdev, &sd, sizeof(sd), cudaMemcpyHostToDevice, s));
  DCK(cudaStreamSynchronize(s));
  c->abp1 = c->cbp1 = 0.9; c->abp2 = c->cbp2 = 0.999;
  c->params_set = true;
  return CRL_OK;
}

extern "C" CRL_API int crl_sac_get_params(crl_sac_ctx* t, float* actor, float* qf1, float* qf2, float* qf1_target, float* qf2_target,
                                          float* log_alpha) {
  if (!t) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  if (int rc = crl_ddpg_get_params(t->d, nullptr, qf1, nullptr, qf1_target)) return rc;
  const cudaStream_t s = t->d->stream;
  if (actor) DCK(cudaMemcpyAsync(actor, t->actor, sizeof(float) * SNet::P, cudaMemcpyDeviceToHost, s));
  if (qf2) DCK(cudaMemcpyAsync(qf2, t->critic2, sizeof(float) * CNet::P, cudaMemcpyDeviceToHost, s));
  if (qf2_target) DCK(cudaMemcpyAsync(qf2_target, t->critic2_tgt, sizeof(float) * CNet::P, cudaMemcpyDeviceToHost, s));
  if (log_alpha) DCK(cudaMemcpyAsync(log_alpha, &t->sdev->log_alpha, sizeof(float), cudaMemcpyDeviceToHost, s));
  DCK(cudaStreamSynchronize(s));
  return CRL_OK;
}

extern "C" CRL_API int crl_sac_get_adam_state(crl_sac_ctx* t, float* actor_m, float* actor_v, float* qf1_m, float* qf1_v, float* qf2_m,
                                              float* qf2_v, float* log_alpha_mv, double* beta_pow) {
  if (!t) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  if (int rc = crl_ddpg_get_adam_state(t->d, nullptr, nullptr, qf1_m, qf1_v, beta_pow)) return rc;
  const cudaStream_t s = t->d->stream;
  if (actor_m) DCK(cudaMemcpyAsync(actor_m, t->am, sizeof(float) * SNet::P, cudaMemcpyDeviceToHost, s));
  if (actor_v) DCK(cudaMemcpyAsync(actor_v, t->av, sizeof(float) * SNet::P, cudaMemcpyDeviceToHost, s));
  if (qf2_m) DCK(cudaMemcpyAsync(qf2_m, t->c2m, sizeof(float) * CNet::P, cudaMemcpyDeviceToHost, s));
  if (qf2_v) DCK(cudaMemcpyAsync(qf2_v, t->c2v, sizeof(float) * CNet::P, cudaMemcpyDeviceToHost, s));
  if (log_alpha_mv) DCK(cudaMemcpyAsync(log_alpha_mv, &t->sdev->la_m, 2 * sizeof(float), cudaMemcpyDeviceToHost, s));
  DCK(cudaStreamSynchronize(s));
  return CRL_OK;
}

extern "C" CRL_API int crl_sac_reset(crl_sac_ctx* t) {
  if (!t) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  return crl_ddpg_reset(t->d);
}

extern "C" CRL_API int crl_sac_run(crl_sac_ctx* t, int64_t iterations, crl_sac_stats* stats) {
  if (!t) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  if (iterations < 0) return dfail(CRL_ERR_INVALID, "iterations must be >= 0");
  crl_ddpg_ctx* c = t->d;
  if (!c->params_set) return dfail(CRL_ERR_STATE, "crl_sac_run called before crl_sac_set_params");
  if (!c->reset_done) return dfail(CRL_ERR_STATE, "crl_sac_run called before crl_sac_reset");
  const crl_sac_config& g = t->cfg;
  DCK(cudaSetDevice(g.device));
  DCK(cudaMemsetAsync(&c->dev->sum_return, 0, sizeof(double) * 2 + sizeof(unsigned long long), c->stream));
  const Scratch s1 = carve(c->scratch), s2 = carve(t->scratch2);
  const int fwd_blocks = (g.batch_size + LF_S - 1) / LF_S;
  int64_t k = 0;
  while (k < iterations) {
    bool learn = false;
    if (int rc = act_launch(c, t->actor, sac_act_kernel, SACT_SMEM, iterations, k, learn)) return rc;
    if (!learn) continue;
    SacArgs a;
    memset(&a, 0, sizeof(a));
    a.l = learn_args(c, s1);
    a.l.actor = t->actor; a.l.actor_tgt = nullptr;
    a.critic2 = t->critic2; a.critic2_tgt = t->critic2_tgt; a.s2 = s2; a.loss_part2 = t->loss_part2;
    a.alpha = &t->sdev->alpha; a.draw = (unsigned long long)c->learn_steps;
    UpdArgs u1, u2;
    memset(&u1, 0, sizeof(u1));
    u1.lr = g.q_lr; u1.bp1 = c->cbp1; u1.bp2 = c->cbp2;
    u2 = u1;
    u1.params = c->critic; u1.m = c->cm; u1.v = c->cv; u1.loss_out = &c->dev->critic_loss;
    u2.params = t->critic2; u2.m = t->c2m; u2.v = t->c2v; u2.loss_out = &t->sdev->qf2_loss;
    DCK(launch_sac_critic_step(a, u1, u2, c->stream));
    c->cbp1 *= 0.9; c->cbp2 *= 0.999;
    c->launches += 2;
    c->learn_steps += 1;
    if (c->learn_steps % g.policy_frequency == 0) {
      // the actor iterations reuse the batch, qf2's scratch for the actor's and the first loss parts
      SacArgs b = a;
      b.l.s = s2; b.loss_part2 = nullptr;
      for (int u = 0; u < g.policy_frequency; u++) {
        b.draw = (unsigned long long)c->actor_steps;
        UpdArgs ua;
        memset(&ua, 0, sizeof(ua));
        ua.params = t->actor; ua.m = t->am; ua.v = t->av; ua.loss_out = &c->dev->actor_loss;
        ua.lr = g.policy_lr; ua.bp1 = c->abp1; ua.bp2 = c->abp2;
        DCK(launch_sac_actor_step(b, ua, nullptr, c->stream));
        c->launches += 2;
        if (g.autotune) {
          sac_alpha_fwd_kernel<<<fwd_blocks, LF_T, SAL_SMEM, c->stream>>>(b);
          DCK(cudaGetLastError());
          AlphaArgs al;
          al.part = b.l.loss_part; al.n_parts = fwd_blocks; al.B = g.batch_size; al.dev = t->sdev;
          al.lr = g.q_lr; al.bp1 = c->abp1; al.bp2 = c->abp2;
          sac_alpha_update_kernel<<<1, 1, 0, c->stream>>>(al);
          DCK(cudaGetLastError());
          c->launches += 2;
        }
        c->abp1 *= 0.9; c->abp2 *= 0.999;
        c->actor_steps += 1;
      }
    }
    if (c->learn_steps % g.target_network_frequency == 0) {
      sac_polyak_kernel<<<(2 * CNet::P + 255) / 256, 256, 0, c->stream>>>(c->critic, c->critic_tgt, t->critic2, t->critic2_tgt, g.tau);
      DCK(cudaGetLastError());
      c->launches += 1;
    }
  }
  if (stats) {
    DdpgDev d;
    SacDev sd;
    DCK(cudaMemcpyAsync(&d, c->dev, sizeof(d), cudaMemcpyDeviceToHost, c->stream));
    DCK(cudaMemcpyAsync(&sd, t->sdev, sizeof(sd), cudaMemcpyDeviceToHost, c->stream));
    DCK(cudaStreamSynchronize(c->stream));
    stats->qf1_loss = d.critic_loss; stats->qf2_loss = sd.qf2_loss; stats->actor_loss = d.actor_loss;
    stats->alpha_loss = sd.alpha_loss; stats->alpha = sd.alpha; stats->sum_return = d.sum_return;
    stats->sum_length = d.sum_length; stats->episodes = (int64_t)d.episodes; stats->learn_steps = c->learn_steps;
    stats->actor_steps = c->actor_steps; stats->iterations = c->it; stats->kernel_launches = c->launches;
  }
  return CRL_OK;
}

extern "C" CRL_API int crl_sac_read_buffer(crl_sac_ctx* t, float* obs, float* action, float* reward, float* next_obs, uint8_t* terminal,
                                           int32_t* size, int32_t* ptr) {
  if (!t) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  return crl_ddpg_read_buffer(t->d, obs, action, reward, next_obs, terminal, size, ptr);
}

extern "C" CRL_API int crl_sac_forward_raw(const float* actor, const float* qf, const float* obs, const float* action, float* mean_out,
                                           float* log_std_out, float* q_out, int64_t n, void* stream) {
  if (n < 0 || (n > 0 && (!actor || !qf || !obs || !action || !mean_out || !log_std_out || !q_out)))
    return dfail(CRL_ERR_INVALID, "NULL argument or n < 0");
  if (((uintptr_t)actor | (uintptr_t)qf) % 16) return dfail(CRL_ERR_INVALID, "actor and qf must be 16-byte aligned");
  if (n == 0) return CRL_OK;
  if (int rc = ddpg_raw_device_check()) return rc;
  const int64_t grid = (n + ACT_E - 1) / ACT_E;
  if (grid > 0x7fffffff) return dfail(CRL_ERR_INVALID, "n too large");
  sac_forward_raw_kernel<<<(unsigned)grid, ACT_T, SFWD_RAW_SMEM, (cudaStream_t)stream>>>(actor, qf, obs, action, mean_out, log_std_out,
                                                                                          q_out, n);
  DCK(cudaGetLastError());
  return CRL_OK;
}

// scratch of one raw SAC call: two nets' scratch (SAC-sized), 2 x LF_MAX_BLOCKS loss parts and alpha
struct SacRawScratch {
  float* f = nullptr;
  double* d = nullptr;
  ~SacRawScratch() { if (f) cudaFree(f); if (d) cudaFree(d); }
};

static int sac_raw_begin(int32_t B, double alpha, SacRawScratch& r, SacArgs& a, cudaStream_t s) {
  if (B < 1 || B > LEARN_B) return dfail(CRL_ERR_INVALID, "B must be in [1, 256]");
  if (!(alpha >= 0.0 && isfinite(alpha))) return dfail(CRL_ERR_INVALID, "alpha must be finite and >= 0");
  if (int rc = ddpg_raw_device_check()) return rc;
  DCK(cudaMalloc(reinterpret_cast<void**>(&r.f), 2 * SAC_SCRATCH_FLOATS * sizeof(float)));
  DCK(cudaMalloc(reinterpret_cast<void**>(&r.d), (2 * LF_MAX_BLOCKS + 1) * sizeof(double)));
  DCK(cudaMemcpyAsync(r.d + 2 * LF_MAX_BLOCKS, &alpha, sizeof(double), cudaMemcpyHostToDevice, s));
  memset(&a, 0, sizeof(a));
  a.l.B = B; a.l.size = B; a.l.in_order = 1;
  a.l.s = carve(r.f); a.l.loss_part = r.d;
  a.s2 = carve(r.f + SAC_SCRATCH_FLOATS); a.loss_part2 = r.d + LF_MAX_BLOCKS;
  a.alpha = r.d + 2 * LF_MAX_BLOCKS;
  return CRL_OK;
}

extern "C" CRL_API int crl_sac_critic_loss_raw(const float* actor, const float* qf1, const float* qf2, const float* qf1_target,
                                               const float* qf2_target, int32_t B, const float* obs, const float* action,
                                               const float* reward, const float* next_obs, const uint8_t* terminal, double gamma,
                                               double alpha, uint64_t seed, uint64_t learn_step, float* qf1_grads_out,
                                               float* qf2_grads_out, double* qf1_loss_out, double* qf2_loss_out, void* stream) {
  if (!actor || !qf1 || !qf2 || !qf1_target || !qf2_target || !obs || !action || !reward || !next_obs || !terminal ||
      !qf1_grads_out || !qf2_grads_out || !qf1_loss_out || !qf2_loss_out)
    return dfail(CRL_ERR_INVALID, "NULL argument");
  if (((uintptr_t)actor | (uintptr_t)qf1 | (uintptr_t)qf2 | (uintptr_t)qf1_target | (uintptr_t)qf2_target) % 16)
    return dfail(CRL_ERR_INVALID, "parameter vectors must be 16-byte aligned");
  const cudaStream_t s = (cudaStream_t)stream;
  SacRawScratch r;
  SacArgs a;
  if (int rc = sac_raw_begin(B, alpha, r, a, s)) return rc;
  LearnArgs& l = a.l;
  l.actor = actor; l.critic = qf1; l.critic_tgt = qf1_target;
  l.b_obs = obs; l.b_act = action; l.b_rew = reward; l.b_next = next_obs; l.b_term = terminal;
  l.seed = seed; l.gamma = gamma;
  a.critic2 = qf2; a.critic2_tgt = qf2_target; a.draw = learn_step;
  UpdArgs u1, u2;
  memset(&u1, 0, sizeof(u1));
  u2 = u1;
  u1.grads_out = qf1_grads_out; u1.loss_out = qf1_loss_out;
  u2.grads_out = qf2_grads_out; u2.loss_out = qf2_loss_out;
  cudaError_t e = launch_sac_critic_step(a, u1, u2, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);   // the scratch is freed on return
  if (e != cudaSuccess) return dfail(CRL_ERR_CUDA, std::string("crl_sac_critic_loss_raw failed: ") + cudaGetErrorString(e));
  return CRL_OK;
}

extern "C" CRL_API int crl_sac_actor_loss_raw(const float* actor, const float* qf1, const float* qf2, int32_t B, const float* obs,
                                              double alpha, uint64_t seed, uint64_t actor_step, float* grads_out, double* loss_out,
                                              double* mean_log_pi_out, void* stream) {
  if (!actor || !qf1 || !qf2 || !obs || !grads_out || !loss_out || !mean_log_pi_out) return dfail(CRL_ERR_INVALID, "NULL argument");
  if (((uintptr_t)actor | (uintptr_t)qf1 | (uintptr_t)qf2) % 16) return dfail(CRL_ERR_INVALID, "parameter vectors must be 16-byte aligned");
  const cudaStream_t s = (cudaStream_t)stream;
  SacRawScratch r;
  SacArgs a;
  if (int rc = sac_raw_begin(B, alpha, r, a, s)) return rc;
  a.l.actor = actor; a.l.critic = qf1; a.l.b_obs = obs; a.l.seed = seed;
  a.critic2 = qf2; a.draw = actor_step;
  UpdArgs u;
  memset(&u, 0, sizeof(u));
  u.grads_out = grads_out; u.loss_out = loss_out;
  cudaError_t e = launch_sac_actor_step(a, u, mean_log_pi_out, s);
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return dfail(CRL_ERR_CUDA, std::string("crl_sac_actor_loss_raw failed: ") + cudaGetErrorString(e));
  return CRL_OK;
}
