// dqn.cu — vectorised DQN (SURVEY 8f-2; src/algorithms/dqn.jl) behind the crl_dqn_* entry points of
// include/cleanrl_cuda.h: N CartPole envs stepping in lockstep with an epsilon-greedy Q-network, an HBM-resident
// ring replay buffer, and one learning step (sample without replacement -> TD target from the target net -> MSE on
// the taken action -> backward -> Adam -> optional target copy) every train_freq iterations.
//
// The 4-120-84-2 network is evaluated out of shared memory as register tiles of 4 neurons x 4 samples (q_forward):
// per k one 128-bit weight load and one 128-bit activation load feed 16 independent FMA chains, software-pipelined.
// With one neuron per thread and one sample per lane the kernels were bound by shared-memory wavefronts (ncu:
// profiles/r1_v7_ncu_dqn_summary.csv); every neuron is still ONE fmaf chain over ascending k, so results do not
// depend on the tiling. What is left in the 120 -> 84 layer is the FMA pipe of the busiest scheduler: 21 x 8 tiles are
// 5.25 warps, so two schedulers carry two warps each (measured 44 cycles per k for 32 envs, -DDQN_TRACE).
//
//   dqn_act_kernel        32 envs per CTA of 256 threads. Warp 0 (one lane per env, state in registers) draws epsilon /
//                         the random action from Philox, steps CartPole, appends the transition at
//                         (ptr + step * N + env) % capacity and resets a finished env on the spot. The parameters only
//                         change at a learning step, so ONE launch runs every iteration up to the next learning step
//                         (train_freq of them, at most ACT_MAX_STEPS).
//   dqn_learn_fwd_kernel  the learning step, part 1: CTA c owns samples 16c..16c+15 of the batch: gather, target and q
//                         forward, TD target, loss, dz2, dz1; everything the weight gradients need is written
//                         sample-major to a global scratch (L2-resident, 220 KB).
//   dqn_learn_upd_kernel  part 2: a block stages the scratch columns it needs in shared memory, one thread per 4x4
//                         tile of dW2 (or per element of the small arrays) sums over the batch in ascending sample
//                         order (deterministic, the oracle's order) and applies Adam to the parameters it has just
//                         differentiated (plus the target copy), so gradients never leave registers.
// crl_dqn_forward_raw and crl_dqn_loss_raw run the acting kernel's forward pass and the two learning kernels (gradient
// out instead of Adam) on rows the caller passes in, so that each can be compared with a reference on its own.
// Every decision that only depends on counters (epsilon, "learn on this iteration?", "copy the target?", Adam's beta
// powers) is taken on the host, so a run is a plain sequence of launches on one stream without any device-to-host read.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <string>

#include "device_math.cuh"
#include "kernels.h"

namespace {

// -DDQN_TRACE: clock stamps of one CTA printed from the kernels (development aid, like TC_TRACE in update_tc.cu)
#ifdef DQN_TRACE
#define DTR(i) do { if (dtrace) dtr[i] = clock64(); } while (0)
#else
#define DTR(i) do { } while (0)
#endif

constexpr int DQ_D = 4, DQ_H1 = 120, DQ_H2 = 84, DQ_A = 2;
constexpr int DQ_W1 = 0, DQ_B1 = DQ_W1 + DQ_H1 * DQ_D, DQ_W2 = DQ_B1 + DQ_H1, DQ_B2 = DQ_W2 + DQ_H2 * DQ_H1,
              DQ_W3 = DQ_B2 + DQ_H2, DQ_B3 = DQ_W3 + DQ_A * DQ_H2, DQ_P = DQ_B3 + DQ_A;
constexpr int DQ_PP = (DQ_P + 3) & ~3;
static_assert(DQ_P == CRL_DQN_PARAMS, "parameter count");
static_assert(DQ_H2 % 4 == 0 && DQ_H1 % 4 == 0 && DQ_W2 % 4 == 0, "128-bit weight loads of the second layer");
constexpr uint32_t STREAM_DQN_ACT = 3u, STREAM_DQN_BATCH = 4u;
constexpr int ACT_E = 32;           // envs per CTA in dqn_act_kernel
constexpr int ACT_SP = ACT_E + 4;   // activation row stride (floats): rows stay 16-byte aligned
constexpr int ACT_T = 256;          // forward threads of dqn_act_kernel; two speculation warps follow them
constexpr int ACT_THREADS = ACT_T + 64;
constexpr int ACT_MAX_STEPS = 16;   // iterations per dqn_act_kernel launch (bounded by the next learning step)
constexpr int LEARN_B = 128;        // max batch size
constexpr int LF_S = 16, LF_SP = LF_S + 4, LF_T = 256;   // dqn_learn_fwd_kernel: samples per CTA, row stride, threads
constexpr int LF_MAX_BLOCKS = LEARN_B / LF_S;
// dqn_learn_upd_kernel: block kinds (A) dW2 tiles of 4 input columns, (B) dW1/db1 of 24 neurons, (C) dW3/db2(/db3)
// of 28 neurons
constexpr int LU_T = 256;
constexpr int LU_KA = 4, LU_A_BLOCKS = DQ_H1 / LU_KA;    // 30 blocks x (21 neuron quads x 1 input quad) = 630 tiles
constexpr int LU_JB = 24, LU_B_BLOCKS = DQ_H1 / LU_JB;   // 5 blocks x 24 neurons x (4 inputs + bias)
constexpr int LU_KC = 28, LU_C_BLOCKS = DQ_H2 / LU_KC;   // 3 blocks x 28 neurons x (2 outputs + bias)
static_assert(DQ_H1 % LU_KA == 0 && DQ_H1 % LU_JB == 0 && DQ_H2 % LU_KC == 0, "upd block decomposition");
static_assert((DQ_H2 / 4) * (LU_KA / 4) <= LU_T && LU_JB * (DQ_D + 1) <= LU_T && LU_KC * (DQ_A + 1) + DQ_A <= LU_T, "upd block size");

struct DqnDev {               // device-resident scalars
  double last_loss;
  double sum_return, sum_length;
  unsigned long long episodes;
};

struct ActArgs {
  const float* q;
  float* env_state; int* env_t; double* ep_ret; int* ep_len; uint32_t* resets;
  float *b_state, *b_next, *b_reward; int* b_action; uint8_t* b_term;
  DqnDev* dev;
  unsigned long long seed, it0;   // it0 = iteration number (1-based) of step 0 of this launch
  double eps[ACT_MAX_STEPS];      // epsilon of each step (dqn.jl:52, evaluated on the host)
  int n_steps;
  int N, C, ptr, max_steps;
  int env_id_base;                // global id of local env 0 (data-parallel shards; 0 on one GPU)
};

// global -> shared copy of one parameter vector (128-bit loads; cudaMalloc'ed source, 16-byte aligned destination)
template <int NT> __device__ __forceinline__ void load_q_params(const float* __restrict__ g, float* sp, int tid) {
  const float4* g4 = reinterpret_cast<const float4*>(g);
  float4* s4 = reinterpret_cast<float4*>(sp);
  constexpr int N4 = DQ_P / 4, PER = (N4 + NT - 1) / NT;
  float4 tmp[PER];   // every load is in flight before the first store: one L2 round trip instead of PER
#pragma unroll
  for (int u = 0; u < PER; u++) if (tid + u * NT < N4) tmp[u] = g4[tid + u * NT];
#pragma unroll
  for (int u = 0; u < PER; u++) if (tid + u * NT < N4) s4[tid + u * NT] = tmp[u];
  if (tid < DQ_P % 4) sp[N4 * 4 + tid] = g[N4 * 4 + tid];
}

// Dense -> relu -> Dense -> relu -> Dense for a tile of NS samples by NT threads (CTA-wide barriers between the
// layers: every thread of the CTA must call this). p: parameters in shared memory (16-byte aligned); xs [4][SP] the
// inputs, h1 [120][SP], h2 [84][SP], qo [2][SP] (SP a multiple of 4). A thread owns 4 consecutive samples of one
// first-layer neuron, then 4 neurons x 4 samples of the second layer (one 128-bit weight load + one 128-bit activation
// load per k for 16 FMAs), then one (output, sample) chain of the head.
// BAR = 0: __syncthreads (all NT threads of the CTA call this); BAR > 0: named barrier BAR over the first NT threads
// (the acting kernel has two more warps that do not take part)
template <int BAR, int NT> __device__ __forceinline__ void q_barrier() {
  if (BAR == 0) __syncthreads();
  else asm volatile("bar.sync %0, %1;" ::"n"(BAR), "n"(NT) : "memory");
}
template <int NS, int SP, int NT, int BAR = 0>
__device__ __forceinline__ void q_forward(const float* __restrict__ p, const float* xs, float* h1, float* h2, float* qo, int tid) {
  constexpr int EQ = NS / 4;   // sample quads
  static_assert(NS % 4 == 0 && SP % 4 == 0 && SP >= NS, "tile geometry");
#ifdef DQN_TRACE
  const long long q_t0 = clock64();
#endif
  static_assert((DQ_H2 / 4) * EQ <= NT && DQ_A * NS <= NT, "one pass for the second layer and the head");
  for (int w = tid; w < DQ_H1 * EQ; w += NT) {
    const int eq = w % EQ, j = w / EQ;
    float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll
    for (int k = 0; k < DQ_D; k++) {
      const float wt = p[DQ_W1 + j + DQ_H1 * k];
      const float4 x = *reinterpret_cast<const float4*>(xs + k * SP + 4 * eq);
      acc.x = fmaf(wt, x.x, acc.x); acc.y = fmaf(wt, x.y, acc.y); acc.z = fmaf(wt, x.z, acc.z); acc.w = fmaf(wt, x.w, acc.w);
    }
    const float b = p[DQ_B1 + j];
    *reinterpret_cast<float4*>(h1 + j * SP + 4 * eq) =
        make_float4(fmaxf(acc.x + b, 0.0f), fmaxf(acc.y + b, 0.0f), fmaxf(acc.z + b, 0.0f), fmaxf(acc.w + b, 0.0f));
  }
#ifdef DQN_TRACE
  const long long q_t1 = clock64();
#endif
  q_barrier<BAR, NT>();
#ifdef DQN_TRACE
  const long long q_t2 = clock64();
#endif
  if (tid < (DQ_H2 / 4) * EQ) {
    const int eq = tid % EQ, j = 4 * (tid / EQ);
    // 16 independent scalar chains (packed FP32 would need a register-pair move per operand, and with one or two
    // warps per scheduler and in-order issue each move stalls the FMA behind it: measured 45 cycles per k).
    // Software pipeline: the operands of the next U values of k are loaded while the current U are multiplied.
    float acc[4][4];
#pragma unroll
    for (int n = 0; n < 4; n++)
#pragma unroll
      for (int c = 0; c < 4; c++) acc[n][c] = 0.0f;
    constexpr int U = 4;
    static_assert(DQ_H1 % (2 * U) == 0, "pipeline depth");
    const float* wp = p + DQ_W2 + j;
    const float* hp = h1 + 4 * eq;
    float4 wn[U], hn[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      wn[u] = *reinterpret_cast<const float4*>(wp + DQ_H2 * u);
      hn[u] = *reinterpret_cast<const float4*>(hp + SP * u);
    }
#pragma unroll 2
    for (int k0 = 0; k0 < DQ_H1; k0 += U) {
      float4 wc[U], hc[U];
#pragma unroll
      for (int u = 0; u < U; u++) { wc[u] = wn[u]; hc[u] = hn[u]; }
      if (k0 + U < DQ_H1) {
#pragma unroll
        for (int u = 0; u < U; u++) {
          wn[u] = *reinterpret_cast<const float4*>(wp + DQ_H2 * (k0 + U + u));
          hn[u] = *reinterpret_cast<const float4*>(hp + SP * (k0 + U + u));
        }
      }
#pragma unroll
      for (int u = 0; u < U; u++) {
        const float wv[4] = {wc[u].x, wc[u].y, wc[u].z, wc[u].w}, hv[4] = {hc[u].x, hc[u].y, hc[u].z, hc[u].w};
#pragma unroll
        for (int n = 0; n < 4; n++)
#pragma unroll
          for (int c = 0; c < 4; c++) acc[n][c] = fmaf(wv[n], hv[c], acc[n][c]);
      }
    }
#pragma unroll
    for (int n = 0; n < 4; n++) {
      const float b = p[DQ_B2 + j + n];
      *reinterpret_cast<float4*>(h2 + (j + n) * SP + 4 * eq) =
          make_float4(fmaxf(acc[n][0] + b, 0.0f), fmaxf(acc[n][1] + b, 0.0f), fmaxf(acc[n][2] + b, 0.0f), fmaxf(acc[n][3] + b, 0.0f));
    }
  }
#ifdef DQN_TRACE
  const long long q_t3 = clock64();
#endif
  q_barrier<BAR, NT>();
#ifdef DQN_TRACE
  const long long q_t4 = clock64();
#endif
  if (tid < DQ_A * NS) {
    const int l = tid % NS, o = tid / NS;
    // one chain of 84 dependent FMAs: the next 12 operand pairs are loaded under the current 12 FMAs
    constexpr int UH = 12;
    static_assert(DQ_H2 % UH == 0, "head pipeline depth");
    const float* wp = p + DQ_W3 + o;
    const float* hp = h2 + l;
    float wn[UH], hn[UH];
#pragma unroll
    for (int u = 0; u < UH; u++) { wn[u] = wp[DQ_A * u]; hn[u] = hp[SP * u]; }
    float acc = 0.0f;
#pragma unroll
    for (int k0 = 0; k0 < DQ_H2; k0 += UH) {
      float wc[UH], hc[UH];
#pragma unroll
      for (int u = 0; u < UH; u++) { wc[u] = wn[u]; hc[u] = hn[u]; }
      if (k0 + UH < DQ_H2) {
#pragma unroll
        for (int u = 0; u < UH; u++) { wn[u] = wp[DQ_A * (k0 + UH + u)]; hn[u] = hp[SP * (k0 + UH + u)]; }
      }
#pragma unroll
      for (int u = 0; u < UH; u++) acc = fmaf(wc[u], hc[u], acc);
    }
    qo[o * SP + l] = acc + p[DQ_B3 + o];
  }
#ifdef DQN_TRACE
  const long long q_t5 = clock64();
#endif
  q_barrier<BAR, NT>();
#ifdef DQN_TRACE
  if (tid == 0 && blockIdx.x == 0)
    printf("q_forward<%d>: layer1 %lld | barrier %lld | layer2 %lld | barrier %lld | head %lld | barrier %lld\n", NS, q_t1 - q_t0,
           q_t2 - q_t1, q_t3 - q_t2, q_t4 - q_t3, q_t5 - q_t4, clock64() - q_t5);
#endif
}

// Warps 0-7 evaluate the Q-network for the CTA's 32 envs; warp 0 (one lane per env) then chooses the action, records the
// transition and advances its env. As in rollout_kernel, two more warps work in the shadow of the forward pass on what
// does not depend on the chosen action: warp 8 the step's Philox draw (epsilon test + random action) and the successor
// state for action 0, warp 9 the successor for action 1 and the state each env takes at its next reset. Warp 0 picks
// the successor of its action: same device function, same inputs, same bits as stepping afterwards.
__global__ void __launch_bounds__(ACT_THREADS, 1) dqn_act_kernel(ActArgs a) {
  extern __shared__ __align__(16) float smem[];
  constexpr int SP = ACT_SP;
  constexpr int BAR_Q = 1, BAR_SPEC = 2;   // named barriers: forward threads | speculation warps -> warp 0
  float* p = smem;                       // [DQ_PP]
  float* h1 = p + DQ_PP;                 // [120][SP]
  float* h2 = h1 + DQ_H1 * SP;           // [84][SP]
  float* qo = h2 + DQ_H2 * SP;           // [2][SP]
  float* xs = qo + DQ_A * SP;            // [4][SP] current observation of the CTA's envs
  float* st_s = xs + DQ_D * SP;          // [4][ACT_E] env state for the speculation warps (= xs without the padding)
  float* spec_s = st_s + 4 * ACT_E;      // [2][4][ACT_E] successor states
  float* rst_s = spec_s + 8 * ACT_E;     // [4][ACT_E] state at the next reset
  double* u_s = reinterpret_cast<double*>(rst_s + 4 * ACT_E);          // [ACT_E] uniform of the epsilon test
  uint32_t* bit_s = reinterpret_cast<uint32_t*>(rst_s + 6 * ACT_E);    // [ACT_E] random action
  int* used_s = reinterpret_cast<int*>(rst_s + 7 * ACT_E);             // [ACT_E] warp 0 consumed the reset state
  static_assert(((DQ_PP + (DQ_H1 + DQ_H2 + DQ_A + DQ_D) * ACT_SP + 16 * ACT_E) % 2) == 0, "the Float64 uniforms need 8-byte alignment");
  const int tid = threadIdx.x, warp = tid >> 5;
  load_q_params<ACT_THREADS>(a.q, p, tid);
  const int e = tid & 31;                // env lane of warps 0, 8 and 9
  const int n = blockIdx.x * ACT_E + e;
  const bool fwd = tid < ACT_T, owner = tid < ACT_E, in_range = n < a.N, valid = owner && in_range;
  const uint32_t gid = (uint32_t)(a.env_id_base + n);         // Philox is keyed by the global env id
  float st[4] = {0.0f, 0.0f, 0.0f, 0.0f};
  int t = 0, len = 0;
  double ret = 0.0;
  uint32_t rc = 0;                       // warp 0: the env's reset counter; warp 9: the counter its prepared state was drawn for
  if (owner) {
    if (valid) {
      const float4 s4 = reinterpret_cast<const float4*>(a.env_state)[n];
      st[0] = s4.x; st[1] = s4.y; st[2] = s4.z; st[3] = s4.w;
      t = a.env_t[n];
      ret = a.ep_ret[n];
      len = a.ep_len[n];
      rc = a.resets[n];
    }
#pragma unroll
    for (int k = 0; k < 4; k++) { xs[k * SP + e] = st[k]; st_s[k * ACT_E + e] = st[k]; }
    used_s[e] = 0;
  }
  auto prepare_reset = [&]() {           // warp 9
    float u4[4], rs[4];
    int rt;
    rng_reset_uniforms(a.seed, gid, rc, u4);
    cartpole_reset(rs, rt, u4);
#pragma unroll
    for (int k = 0; k < 4; k++) rst_s[k * ACT_E + e] = rs[k];
  };
  if (warp == 9) {
    if (in_range) rc = a.resets[n];
    prepare_reset();
  }
  __syncthreads();
#ifdef DQN_TRACE
  long long dtr[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#endif
  for (int s = 0; s < a.n_steps; s++) {
#ifdef DQN_TRACE
    const bool dtrace = blockIdx.x == 0 && s == 5 && (tid == 0 || tid == 5 * 32);
#endif
    DTR(0);
    if (!fwd) {
      // ---- speculation warps
      if (warp == 9 && used_s[e]) {
        rc += 1;
        prepare_reset();
        used_s[e] = 0;
      }
      if (warp == 8) {
        uint32_t r[4];
        philox_draw(a.seed, gid, a.it0 + (unsigned long long)s, STREAM_DQN_ACT, r);
        u_s[e] = (double)((((uint64_t)r[0] << 32) | r[1]) >> 11) * (1.0 / 9007199254740992.0);
        bit_s[e] = r[2] & 1u;
      }
      float s4[4];
#pragma unroll
      for (int k = 0; k < 4; k++) s4[k] = st_s[k * ACT_E + e];
      cartpole_dynamics(s4, warp - 8);
#pragma unroll
      for (int k = 0; k < 4; k++) spec_s[((warp - 8) * 4 + k) * ACT_E + e] = s4[k];
      __threadfence_block();
      asm volatile("bar.arrive %0, %1;" ::"n"(BAR_SPEC), "n"(ACT_E + 64) : "memory");
    } else {
      q_forward<ACT_E, SP, ACT_T, BAR_Q>(p, xs, h1, h2, qo, tid);   // q_net(obs), dqn.jl:56 (used only where the epsilon test fails)
      DTR(1);
      if (owner) {
        asm volatile("bar.sync %0, %1;" ::"n"(BAR_SPEC), "n"(ACT_E + 64) : "memory");   // this step's speculation has arrived
        if (valid) {
          const float4 obs = make_float4(st[0], st[1], st[2], st[3]);   // deepcopy(state(env)), dqn.jl:50
          int action;
          if (u_s[e] < a.eps[s]) action = (int)bit_s[e];              // rand(action_space(env)), dqn.jl:54
          else action = qo[1 * SP + e] > qo[0 * SP + e] ? 1 : 0;     // argmax: first maximum, dqn.jl:56-57
          DTR(2);
          float rew;
          bool done;
#pragma unroll
          for (int k = 0; k < 4; k++) st[k] = spec_s[(action * 4 + k) * ACT_E + e];   // cartpole_step, evaluated ahead
          t += 1;
          cartpole_outcome(st, t, a.max_steps, rew, done);
          DTR(3);
          const int slot = (int)(((long long)a.ptr + (long long)s * a.N + n) % a.C);   // add!, replay_buffer.jl:23-37, envs in order
          reinterpret_cast<float4*>(a.b_state)[slot] = obs;
          reinterpret_cast<float4*>(a.b_next)[slot] = make_float4(st[0], st[1], st[2], st[3]);
          a.b_action[slot] = action;
          a.b_reward[slot] = rew;
          a.b_term[slot] = done ? 1 : 0;
          ret += (double)rew;
          len += 1;
          if (done) {                          // dqn.jl:80-86
            atomicAdd(&a.dev->episodes, 1ull);
            atomicAdd(&a.dev->sum_return, ret);
            atomicAdd(&a.dev->sum_length, (double)len);
            ret = 0.0;
            len = 0;
#pragma unroll
            for (int k = 0; k < 4; k++) st[k] = rst_s[k * ACT_E + e];   // cartpole_reset with this env's next draw (warp 9)
            t = 0;
            rc += 1;
            used_s[e] = 1;
          }
#pragma unroll
          for (int k = 0; k < 4; k++) { xs[k * SP + e] = st[k]; st_s[k * ACT_E + e] = st[k]; }
        }
      }
    }
    DTR(4);
    __syncthreads();
    DTR(5);
#ifdef DQN_TRACE
    if (dtrace)
      printf("act warp %d: forward %lld | choice %lld | outcome %lld | store+reset %lld | barrier %lld | step %lld\n",
             tid >> 5, dtr[1] - dtr[0], dtr[2] - dtr[1], dtr[3] - dtr[2], dtr[4] - dtr[3], dtr[5] - dtr[4], dtr[5] - dtr[0]);
#endif
  }
  if (valid) {
    a.ep_ret[n] = ret;
    a.ep_len[n] = len;
    a.env_t[n] = t;
    a.resets[n] = rc;
    reinterpret_cast<float4*>(a.env_state)[n] = make_float4(st[0], st[1], st[2], st[3]);
  }
}

// crl_dqn_forward_raw: the acting kernel's forward pass alone (same instantiation of q_forward, 32 samples per CTA, named
// barrier), so that its Q-values can be compared with a reference; rows past n are zero and not written back
__global__ void __launch_bounds__(ACT_T, 1) dqn_forward_raw_kernel(const float* q, const float* obs, float* q_out, int64_t n) {
  extern __shared__ __align__(16) float smem[];
  constexpr int SP = ACT_SP;
  float* p = smem;                       // [DQ_PP]
  float* h1 = p + DQ_PP;                 // [120][SP]
  float* h2 = h1 + DQ_H1 * SP;           // [84][SP]
  float* qo = h2 + DQ_H2 * SP;           // [2][SP]
  float* xs = qo + DQ_A * SP;            // [4][SP]
  const int tid = threadIdx.x;
  load_q_params<ACT_T>(q, p, tid);
  const int64_t i = (int64_t)blockIdx.x * ACT_E + tid;
  if (tid < ACT_E) {
    float4 x = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (i < n) x = reinterpret_cast<const float4*>(obs)[i];
    xs[0 * SP + tid] = x.x; xs[1 * SP + tid] = x.y; xs[2 * SP + tid] = x.z; xs[3 * SP + tid] = x.w;
  }
  __syncthreads();
  q_forward<ACT_E, SP, ACT_T, 1>(p, xs, h1, h2, qo, tid);
  if (tid < ACT_E && i < n) reinterpret_cast<float2*>(q_out)[i] = make_float2(qo[0 * SP + tid], qo[1 * SP + tid]);
}

struct LearnArgs {
  float* q; float* tgt; float* m; float* v;
  const float *b_state, *b_next, *b_reward; const int* b_action; const uint8_t* b_term;
  DqnDev* dev;
  unsigned long long seed, learn_step;
  double gamma, lr;
  int B, size, copy_target;
  int in_order;           // sample b is row b of the b_* arrays (crl_dqn_loss_raw), not entry b of the keyed permutation
  // sample-major scratch between the two kernels: [128][120], [128][84], [128][84], [128][120], [128][4], [128][2]
  float *h1T, *h2T, *z2T, *z1T, *xT, *dqT;
  double* loss_part;      // [LF_MAX_BLOCKS]
  double bp1, bp2;        // beta1^t, beta2^t of Adam, kept on the host
  // data-parallel shards: the mean is over B_scale = world * B samples, the batch permutation is keyed by the rank, and
  // the update kernel leaves its gradient in gbuf / its squared-error sum in lbuf for the allreduce (dqn_adam_kernel)
  int B_scale, rank;
  float* gbuf;            // [DQ_P]
  double* lbuf;           // [1]
  // peer-memory exchange (crl_dqn_comm_init): the update kernel also PUSHES every gradient element (and the loss sum)
  // into every peer's exchange buffer as a flag-in-data packet; dqn_adam_kernel polls this rank's own buffer and adds
  // the world values in rank order (the oracle's order). Row layout [2 slots][world][x_stride] packets of 16 bytes.
  unsigned char* const* x_peers;   // device array [world] of all ranks' exchange buffers, or nullptr (NCCL allreduce)
  const unsigned char* x_local;
  int x_world, x_stride, x_slot;
  unsigned int x_flag;
  int* x_err;
  long long x_timeout;
};

// push element k of this rank's contribution (gradient k < DQ_P, squared-error sum k = DQ_P) to every peer
__device__ __forceinline__ void x_push(const LearnArgs& a, int k, double v) {
  if (!a.x_peers) return;
  for (int r = 0; r < a.x_world; r++) {
    if (r == a.rank) continue;
    uint4* dst = reinterpret_cast<uint4*>(a.x_peers[r]) + ((size_t)a.x_slot * a.x_world + a.rank) * a.x_stride + k;
    ll_store(dst, v, a.x_flag);
  }
}

__global__ void __launch_bounds__(LF_T) dqn_learn_fwd_kernel(LearnArgs a) {
  extern __shared__ __align__(16) float smem[];
  constexpr int SP = LF_SP, EQ = LF_S / 4;
  float* pq = smem;                       // q_net parameters
  float* pt = pq + DQ_PP;                 // target_net parameters
  float* h1 = pt + DQ_PP;                 // [120][SP]
  float* h2 = h1 + DQ_H1 * SP;            // [84][SP]   (later dz2 in place)
  float* qo = h2 + DQ_H2 * SP;            // [2][SP]
  float* dq = qo + DQ_A * SP;             // [2][SP]
  float* xin = dq + DQ_A * SP;            // [8][SP]: rows 0-3 state, rows 4-7 next_state
  __shared__ float s_rew[LF_S];
  __shared__ int s_act[LF_S], s_term[LF_S];
  const int tid = threadIdx.x, B = a.B;
  const int b0 = blockIdx.x * LF_S;       // first sample of this CTA
#ifdef DQN_TRACE
  long long dtr[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  const bool dtrace = blockIdx.x == 0 && (tid == 0 || tid == 5 * 32);
#endif
  DTR(0);
  // the gather (HBM latency) is issued first and completes under the parameter loads
  float4 s4 = make_float4(0.f, 0.f, 0.f, 0.f), n4 = s4;
  int act = 0, term = 0;
  float rew = 0.0f;
  if (tid < LF_S && b0 + tid < B) {
    // sample(1:size, B, replace=false), replay_buffer.jl:43: the first B entries of a keyed permutation of [0,size)
    uint32_t idx = (uint32_t)(b0 + tid);
    if (!a.in_order) {
      uint32_t keys[8];
      philox_draw(a.seed, (uint32_t)a.rank, a.learn_step, STREAM_DQN_BATCH, keys);
      philox_draw(a.seed, 0x80000000u | (uint32_t)a.rank, a.learn_step, STREAM_DQN_BATCH, keys + 4);
      idx = perm_index(idx, (uint32_t)a.size, perm_half_bits((uint32_t)a.size), keys);
    }
    s4 = reinterpret_cast<const float4*>(a.b_state)[idx];
    n4 = reinterpret_cast<const float4*>(a.b_next)[idx];
    act = a.b_action[idx];
    rew = a.b_reward[idx];
    term = a.b_term[idx];
  }
  load_q_params<LF_T>(a.q, pq, tid);
  load_q_params<LF_T>(a.tgt, pt, tid);
  if (tid < LF_S) {
    const int i = tid, b = b0 + i;
    if (b < B) reinterpret_cast<float4*>(a.xT)[b] = s4;
    xin[0 * SP + i] = s4.x; xin[1 * SP + i] = s4.y; xin[2 * SP + i] = s4.z; xin[3 * SP + i] = s4.w;
    xin[4 * SP + i] = n4.x; xin[5 * SP + i] = n4.y; xin[6 * SP + i] = n4.z; xin[7 * SP + i] = n4.w;
    s_rew[i] = rew; s_act[i] = act; s_term[i] = term;
  }
  DTR(1);
  __syncthreads();
  DTR(2);
  q_forward<LF_S, SP, LF_T>(pt, xin + 4 * SP, h1, h2, qo, tid);      // target_net(next_state), dqn.jl:99
  DTR(3);
  double td = 0.0;
  if (tid < LF_S) {
    const float next_q = fmaxf(qo[0 * SP + tid], qo[1 * SP + tid]);
    td = (double)s_rew[tid] + a.gamma * (double)next_q * (1.0 - (double)s_term[tid]);   // dqn.jl:100
  }
  __syncthreads();
  q_forward<LF_S, SP, LF_T>(pq, xin, h1, h2, qo, tid);               // q_net(state), dqn.jl:105
  DTR(4);
  if (tid < LF_S) {                                                  // lanes 0-15 of warp 0
    const int i = tid, b = b0 + i;
    float d0 = 0.0f, d1 = 0.0f;
    double sq = 0.0;
    if (b < B) {
      const int act = s_act[i];
      const double diff = td - (double)qo[act * SP + i];
      sq = diff * diff;                                              // Flux.mse, dqn.jl:107
      const float dd = (float)(-2.0 * diff / (double)a.B_scale);
      if (act == 0) d0 = dd; else d1 = dd;
      reinterpret_cast<float2*>(a.dqT)[b] = make_float2(d0, d1);
    }
    dq[0 * SP + i] = d0;
    dq[1 * SP + i] = d1;
#pragma unroll
    for (int o = LF_S / 2; o > 0; o >>= 1) sq += __shfl_xor_sync(0x0000ffffu, sq, o);
    if (i == 0) a.loss_part[blockIdx.x] = sq;
  }
  __syncthreads();
  DTR(5);
  // dz2 = (W3^T dq) .* (h2 > 0), in place; h1, h2 (activations) and dz2 go to the scratch, neuron fastest
  for (int w = tid; w < DQ_H2 * LF_S; w += LF_T) {
    const int k = w % DQ_H2, i = w / DQ_H2, b = b0 + i;
    const float hv = h2[k * SP + i];
    const float dh = fmaf(pq[DQ_W3 + 1 + DQ_A * k], dq[1 * SP + i], pq[DQ_W3 + 0 + DQ_A * k] * dq[0 * SP + i]);
    const float z = hv > 0.0f ? dh : 0.0f;
    h2[k * SP + i] = z;
    if (b < B) { a.h2T[b * DQ_H2 + k] = hv; a.z2T[b * DQ_H2 + k] = z; }
  }
  for (int w = tid; w < DQ_H1 * LF_S; w += LF_T) {
    const int k = w % DQ_H1, i = w / DQ_H1, b = b0 + i;
    if (b < B) a.h1T[b * DQ_H1 + k] = h1[k * SP + i];
  }
  __syncthreads();
  DTR(6);
  // dz1 = (W2^T dz2) .* (h1 > 0): a thread owns inputs k, k + 60 for 4 samples; four consecutive j are one 128-bit
  // weight load (each chain in ascending j)
  if (tid < (DQ_H1 / 2) * EQ) {
    const int eq = tid % EQ, k = tid / EQ;
    float4 d[2];
    d[0] = d[1] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll 3
    for (int j = 0; j < DQ_H2; j += 4) {
      float4 z[4];
#pragma unroll
      for (int t = 0; t < 4; t++) z[t] = *reinterpret_cast<const float4*>(h2 + (j + t) * SP + 4 * eq);
#pragma unroll
      for (int c = 0; c < 2; c++) {
        const float4 w = *reinterpret_cast<const float4*>(pq + DQ_W2 + j + DQ_H2 * (k + (DQ_H1 / 2) * c));
        d[c].x = fmaf(w.x, z[0].x, d[c].x); d[c].y = fmaf(w.x, z[0].y, d[c].y); d[c].z = fmaf(w.x, z[0].z, d[c].z); d[c].w = fmaf(w.x, z[0].w, d[c].w);
        d[c].x = fmaf(w.y, z[1].x, d[c].x); d[c].y = fmaf(w.y, z[1].y, d[c].y); d[c].z = fmaf(w.y, z[1].z, d[c].z); d[c].w = fmaf(w.y, z[1].w, d[c].w);
        d[c].x = fmaf(w.z, z[2].x, d[c].x); d[c].y = fmaf(w.z, z[2].y, d[c].y); d[c].z = fmaf(w.z, z[2].z, d[c].z); d[c].w = fmaf(w.z, z[2].w, d[c].w);
        d[c].x = fmaf(w.w, z[3].x, d[c].x); d[c].y = fmaf(w.w, z[3].y, d[c].y); d[c].z = fmaf(w.w, z[3].z, d[c].z); d[c].w = fmaf(w.w, z[3].w, d[c].w);
      }
    }
#pragma unroll
    for (int c = 0; c < 2; c++) {
      const int kc = k + (DQ_H1 / 2) * c;
      const float4 hv = *reinterpret_cast<const float4*>(h1 + kc * SP + 4 * eq);
      const float dv[4] = {d[c].x, d[c].y, d[c].z, d[c].w}, hh[4] = {hv.x, hv.y, hv.z, hv.w};
#pragma unroll
      for (int t = 0; t < 4; t++) {
        const int b = b0 + 4 * eq + t;
        if (b < B) a.z1T[b * DQ_H1 + kc] = hh[t] > 0.0f ? dv[t] : 0.0f;
      }
    }
  }
  DTR(7);
#ifdef DQN_TRACE
  if (dtrace)
    printf("learn_fwd warp %d: params+gather %lld | barrier %lld | target fwd %lld | q fwd %lld | loss %lld | dz2+export %lld | dz1 %lld | total %lld\n",
           tid >> 5, dtr[1] - dtr[0], dtr[2] - dtr[1], dtr[3] - dtr[2], dtr[4] - dtr[3], dtr[5] - dtr[4], dtr[6] - dtr[5], dtr[7] - dtr[6], dtr[7] - dtr[0]);
#endif
}

// Flux.Adam(lr) (dqn.jl:41,109) for NP parameters of one thread, Float64 scalars as in clip_adam_kernel; then the
// target copy (dqn.jl:111-113). All loads are issued before the first store (the compiler cannot prove that the
// arrays do not alias).
template <int NP>
__device__ __forceinline__ void dqn_adam(const LearnArgs& a, const int (&idx)[NP], const float (&g)[NP], const bool (&ok)[NP]) {
  const double b1 = 0.9, b2 = 0.999, eps = 1e-8;
  float m0[NP], v0[NP], q0[NP];
#pragma unroll
  for (int i = 0; i < NP; i++) {
    m0[i] = v0[i] = q0[i] = 0.0f;
    if (ok[i]) { m0[i] = a.m[idx[i]]; v0[i] = a.v[idx[i]]; q0[i] = a.q[idx[i]]; }
  }
  const double c1 = 1.0 - a.bp1, c2 = 1.0 - a.bp2;
#pragma unroll
  for (int i = 0; i < NP; i++) {
    if (!ok[i]) continue;
    const float d = g[i];
    const float mt = (float)__dadd_rn(__dmul_rn(b1, (double)m0[i]), __dmul_rn(1.0 - b1, (double)d));
    const float vt = (float)__dadd_rn(__dmul_rn(b2, (double)v0[i]), __dmul_rn(__dmul_rn(1.0 - b2, (double)d), (double)d));
    const double den = __dadd_rn(sqrt(__ddiv_rn((double)vt, c2)), eps);
    const float step = (float)__dmul_rn(__ddiv_rn(__ddiv_rn((double)mt, c1), den), a.lr);
    const float pn = __fsub_rn(q0[i], step);
    a.m[idx[i]] = mt;
    a.v[idx[i]] = vt;
    a.q[idx[i]] = pn;
    if (a.copy_target) a.tgt[idx[i]] = pn;
  }
}

// block-wide copy of `cols` consecutive columns starting at column c0 of a sample-major [rows][ld] scratch array into
// shared memory [rows][cols] (128-bit loads; c0, cols, ld multiples of 4)
__device__ __forceinline__ void stage_cols(const float* __restrict__ src, int ld, int c0, int cols, int rows, float* dst, int tid) {
  const int q = cols / 4, total = rows * q;
  constexpr int BATCH = 8;   // loads in flight per thread before the first store
  for (int base = 0; base < total; base += BATCH * LU_T) {
    float4 tmp[BATCH];
#pragma unroll
    for (int u = 0; u < BATCH; u++) {
      const int i = base + u * LU_T + tid;
      if (i < total) tmp[u] = *reinterpret_cast<const float4*>(src + (i / q) * ld + c0 + 4 * (i % q));
    }
#pragma unroll
    for (int u = 0; u < BATCH; u++) {
      const int i = base + u * LU_T + tid;
      if (i < total) reinterpret_cast<float4*>(dst)[i] = tmp[u];
    }
  }
}

// EXCH = false: Adam on the spot (one GPU). EXCH = true: the gradient goes to a.gbuf and the squared-error sum to a.lbuf;
// after the allreduce dqn_adam_kernel finishes the step.
template <bool EXCH>
__global__ void __launch_bounds__(LU_T) dqn_learn_upd_kernel(LearnArgs a, int n_fwd_blocks) {
  extern __shared__ __align__(16) float smem[];
  const int B = a.B, tid = threadIdx.x;
  if (blockIdx.x == 0 && tid == LU_T - 1) {
    double sq = 0.0;
    for (int c = 0; c < n_fwd_blocks; c++) sq += a.loss_part[c];
    if (EXCH) { a.lbuf[0] = sq; x_push(a, DQ_P, sq); }
    else a.dev->last_loss = sq / (double)B;
  }
#ifdef DQN_TRACE
  long long dtr[4] = {0, 0, 0, 0};
  const bool dtrace = (blockIdx.x == 1 || blockIdx.x == LU_A_BLOCKS || blockIdx.x == LU_A_BLOCKS + LU_B_BLOCKS) && tid == 0;
#endif
  DTR(0);
  if (blockIdx.x < LU_A_BLOCKS) {
    // (A) dW2(j,k) for the 4 inputs k0..k0+3: thread = neurons j, j+21, j+42, j+63 x 4 consecutive inputs; the block's
    // 336 parameters W2(:, k0..k0+3) are contiguous in the flat vector, so Adam then runs block-wide and coalesced
    constexpr int JQ = DQ_H2 / 4, NPAR = DQ_H2 * LU_KA, PER = (NPAR + LU_T - 1) / LU_T;
    const int k0 = blockIdx.x * LU_KA;
    float* zs = smem;                     // [B][84]  dz2
    float* hs = zs + LEARN_B * DQ_H2;     // [B][4]   h1 columns k0..
    float* gs = hs + LEARN_B * LU_KA;     // [4][84]  gradient of this block's parameters
    stage_cols(a.z2T, DQ_H2, 0, DQ_H2, B, zs, tid);
    stage_cols(a.h1T, DQ_H1, k0, LU_KA, B, hs, tid);
    __syncthreads();
    DTR(1);
    if (tid < JQ * (LU_KA / 4)) {
      const int j = tid % JQ, kq = tid / JQ;
      float acc[4][4];   // 16 independent scalar chains (see q_forward)
#pragma unroll
      for (int t = 0; t < 4; t++)
#pragma unroll
        for (int u = 0; u < 4; u++) acc[t][u] = 0.0f;
#pragma unroll 4
      for (int b = 0; b < B; b++) {
        const float4 hh = *reinterpret_cast<const float4*>(hs + b * LU_KA + 4 * kq);
        const float hv[4] = {hh.x, hh.y, hh.z, hh.w};
#pragma unroll
        for (int t = 0; t < 4; t++) {
          const float z = zs[b * DQ_H2 + j + JQ * t];
#pragma unroll
          for (int u = 0; u < 4; u++) acc[t][u] = fmaf(z, hv[u], acc[t][u]);
        }
      }
#pragma unroll
      for (int t = 0; t < 4; t++)
#pragma unroll
        for (int u = 0; u < 4; u++) gs[(4 * kq + u) * DQ_H2 + j + JQ * t] = acc[t][u];
    }
    __syncthreads();
    DTR(2);
    {
      int idx[PER];
      float g[PER];
      bool ok[PER];
#pragma unroll
      for (int u = 0; u < PER; u++) {
        const int i = tid + u * LU_T;
        ok[u] = i < NPAR;
        idx[u] = DQ_W2 + DQ_H2 * k0 + i;
        g[u] = ok[u] ? gs[i] : 0.0f;
        if (EXCH && ok[u]) { a.gbuf[idx[u]] = g[u]; x_push(a, idx[u], (double)g[u]); }
      }
      if (!EXCH) dqn_adam<PER>(a, idx, g, ok);
    }
    DTR(3);
#ifdef DQN_TRACE
    if (dtrace) printf("learn_upd A: stage %lld | reduce %lld | adam x2 %lld\n", dtr[1] - dtr[0], dtr[2] - dtr[1], dtr[3] - dtr[2]);
#endif
    return;
  }
  if (blockIdx.x < LU_A_BLOCKS + LU_B_BLOCKS) {
    // (B) dW1(j, 0..3) and db1(j) for the 24 first-layer neurons j0..j0+23
    const int j0 = (blockIdx.x - LU_A_BLOCKS) * LU_JB;
    float* z1s = smem;                    // [B][24]  dz1 columns j0..
    float* xs = z1s + LEARN_B * LU_JB;    // [B][4]
    stage_cols(a.z1T, DQ_H1, j0, LU_JB, B, z1s, tid);
    stage_cols(a.xT, DQ_D, 0, DQ_D, B, xs, tid);
    __syncthreads();
    DTR(1);
    if (tid >= LU_JB * (DQ_D + 1)) return;
    const int jl = tid % LU_JB, kind = tid / LU_JB, j = j0 + jl;
    float acc = 0.0f;
    int idx[1];
    if (kind < DQ_D) {
#pragma unroll 8
      for (int b = 0; b < B; b++) acc = fmaf(z1s[b * LU_JB + jl], xs[b * DQ_D + kind], acc);
      idx[0] = DQ_W1 + j + DQ_H1 * kind;
    } else {
#pragma unroll 8
      for (int b = 0; b < B; b++) acc += z1s[b * LU_JB + jl];
      idx[0] = DQ_B1 + j;
    }
    DTR(2);
    const float g[1] = {acc};
    const bool ok[1] = {true};
    if (EXCH) { a.gbuf[idx[0]] = acc; x_push(a, idx[0], (double)acc); }
    else dqn_adam<1>(a, idx, g, ok);
    DTR(3);
#ifdef DQN_TRACE
    if (dtrace) printf("learn_upd B: stage %lld | reduce %lld | adam %lld\n", dtr[1] - dtr[0], dtr[2] - dtr[1], dtr[3] - dtr[2]);
#endif
    return;
  }
  {
    // (C) dW3(0,k), dW3(1,k), db2(k) for the 28 second-layer neurons k0..k0+27; db3 in the first of these blocks
    const int c = blockIdx.x - LU_A_BLOCKS - LU_B_BLOCKS, k0 = c * LU_KC;
    float* h2s = smem;                    // [B][28]  h2 columns k0..
    float* z2s = h2s + LEARN_B * LU_KC;   // [B][28]  dz2 columns k0..
    float* dqs = z2s + LEARN_B * LU_KC;   // [B][2]
    stage_cols(a.h2T, DQ_H2, k0, LU_KC, B, h2s, tid);
    stage_cols(a.z2T, DQ_H2, k0, LU_KC, B, z2s, tid);
    for (int i = tid; i < B * DQ_A; i += LU_T) dqs[i] = a.dqT[i];
    __syncthreads();
    DTR(1);
    const int n_main = LU_KC * (DQ_A + 1);
    if (tid >= n_main + (c == 0 ? DQ_A : 0)) return;
    float acc = 0.0f;
    int idx[1];
    if (tid < n_main) {
      const int kl = tid % LU_KC, kind = tid / LU_KC, k = k0 + kl;
      if (kind < DQ_A) {
#pragma unroll 8
        for (int b = 0; b < B; b++) acc = fmaf(dqs[b * DQ_A + kind], h2s[b * LU_KC + kl], acc);
        idx[0] = DQ_W3 + kind + DQ_A * k;
      } else {
#pragma unroll 8
        for (int b = 0; b < B; b++) acc += z2s[b * LU_KC + kl];
        idx[0] = DQ_B2 + k;
      }
    } else {
      const int o = tid - n_main;
#pragma unroll 8
      for (int b = 0; b < B; b++) acc += dqs[b * DQ_A + o];
      idx[0] = DQ_B3 + o;
    }
    DTR(2);
    const float g[1] = {acc};
    const bool ok[1] = {true};
    if (EXCH) { a.gbuf[idx[0]] = acc; x_push(a, idx[0], (double)acc); }
    else dqn_adam<1>(a, idx, g, ok);
    DTR(3);
#ifdef DQN_TRACE
    if (dtrace) printf("learn_upd C: stage %lld | reduce %lld | adam %lld\n", dtr[1] - dtr[0], dtr[2] - dtr[1], dtr[3] - dtr[2]);
#endif
  }
}

// data-parallel shards: Adam on the summed gradient (every rank holds the same sums, so the replicas stay identical).
// With the peer-memory exchange this kernel IS the second half of the allreduce: thread k waits for every peer's packet
// k of this learning step in this rank's own memory and adds the world values in rank order, Float32 as the oracle's
// group run does (the loss sum in Float64). Without it (x_local == nullptr) gbuf / lbuf hold NCCL's sums.
__global__ void __launch_bounds__(256) dqn_adam_kernel(LearnArgs a) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k > DQ_P) return;
  float gsum = k < DQ_P ? a.gbuf[k] : 0.0f;
  double lsum = k == DQ_P ? a.lbuf[0] : 0.0;
  if (a.x_local) {
    const uint4* src = reinterpret_cast<const uint4*>(a.x_local) + (size_t)a.x_slot * a.x_world * a.x_stride + k;
    const float mine_g = gsum;
    const double mine_l = lsum;
    const long long t0 = clock64();
    bool bad = *reinterpret_cast<volatile int*>(a.x_err) != 0;   // sticky: an earlier exchange timed out
    for (int r = 0; r < a.x_world && !bad; r++) {
      double v;
      if (r == a.rank) {
        v = k < DQ_P ? (double)mine_g : mine_l;
      } else {
        uint4 pk = ll_load(src + (size_t)r * a.x_stride);
        while (pk.y != a.x_flag || pk.w != a.x_flag) {
          if (clock64() - t0 > a.x_timeout) { bad = true; break; }
          pk = ll_load(src + (size_t)r * a.x_stride);
        }
        v = __longlong_as_double((long long)(((unsigned long long)pk.z << 32) | pk.x));
      }
      if (k < DQ_P) gsum = r == 0 ? (float)v : __fadd_rn(gsum, (float)v);
      else lsum = r == 0 ? v : lsum + v;
    }
    if (bad) { atomicExch(a.x_err, 1); return; }   // no step on partial sums; the host reports CRL_ERR_NCCL
  }
  if (k == DQ_P) { a.dev->last_loss = lsum / (double)a.B_scale; return; }
  const int idx[1] = {k};
  const float g[1] = {gsum};
  const bool ok[1] = {true};
  dqn_adam<1>(a, idx, g, ok);
}

__global__ void dqn_loss_raw_finish_kernel(const double* sq, int B, double* loss_out) { *loss_out = sq[0] / (double)B; }

constexpr int ACT_SPEC_FLOATS = (4 + 2 * 4 + 4 + 2 + 1 + 1) * ACT_E;   // state | 2 successors | reset state | uniform (double) | random bit | used flag
constexpr size_t FWD_RAW_SMEM = (DQ_PP + (DQ_H1 + DQ_H2 + DQ_A + DQ_D) * ACT_SP) * sizeof(float);
constexpr size_t ACT_SMEM = FWD_RAW_SMEM + ACT_SPEC_FLOATS * sizeof(float);
constexpr size_t LF_SMEM = (2 * DQ_PP + (DQ_H1 + DQ_H2 + 2 * DQ_A + 2 * DQ_D) * LF_SP) * sizeof(float);
constexpr size_t LU_SMEM = ((size_t)LEARN_B * (DQ_H2 + LU_KA) + DQ_H2 * LU_KA) * sizeof(float);   // kind (A) is the largest
static_assert(LEARN_B * (LU_JB + DQ_D) <= LEARN_B * (DQ_H2 + LU_KA) && LEARN_B * (2 * LU_KC + DQ_A) <= LEARN_B * (DQ_H2 + LU_KA), "upd smem");
static_assert(ACT_SMEM <= 227 * 1024 && LF_SMEM <= 227 * 1024 && LU_SMEM <= 227 * 1024, "dqn shared memory");

int dfail(int code, const std::string& msg) { return crl_internal_fail(code, msg.c_str()); }
#define DCK(call)                                                                                          \
  do {                                                                                                     \
    cudaError_t e__ = (call);                                                                              \
    if (e__ != cudaSuccess)                                                                                \
      return dfail(CRL_ERR_CUDA, std::string(#call) + " failed: " + cudaGetErrorString(e__) + " (dqn.cu)"); \
  } while (0)

template <typename T> cudaError_t dzalloc(T** p, size_t n) {
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), (n ? n : 1) * sizeof(T));
  if (e != cudaSuccess) return e;
  return cudaMemset(*p, 0, (n ? n : 1) * sizeof(T));
}

}  // namespace

struct crl_dqn_ctx {
  crl_dqn_config cfg;
  cudaStream_t stream;
  float *q, *tgt, *m, *v;
  float* env_state; int* env_t; double* ep_ret; int* ep_len; uint32_t* resets;
  float *b_state, *b_next, *b_reward; int* b_action; uint8_t* b_term;
  DqnDev* dev;
  float *h1T, *h2T, *z2T, *z1T, *xT, *dqT;   // scratch between dqn_learn_fwd_kernel and dqn_learn_upd_kernel
  double* loss_part;
  double bp1, bp2;                            // beta1^t, beta2^t of Adam
  int world, rank, env_id_base;               // data-parallel shard (crl_dqn_comm_init); 1, 0, 0 on one GPU
  void* comm;                                 // NCCL communicator when world > 1
  float* gbuf; double* lbuf;                  // allreduce payload: gradient, squared-error sum
  // peer-memory exchange of that payload (NVLink): own buffer, the peers' mappings, device copy of the pointer table
  unsigned char* x_buf; unsigned char* x_peer[CRL_MAX_WORLD]; unsigned char** x_peers_dev; int* x_err; int x_stride; bool x_on;
  long long x_timeout;
  int size, ptr;
  long long it, learn_steps, launches;
  bool params_set, reset_done;
};

__global__ void dqn_reset_kernel(int N, unsigned long long seed, int env_id_base, float* env_state, int* env_t, double* ep_ret, int* ep_len,
                                 uint32_t* resets) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float u4[4], st[4];
  int t;
  rng_reset_uniforms(seed, (uint32_t)(env_id_base + n), 0, u4);
  cartpole_reset(st, t, u4);
  for (int k = 0; k < 4; k++) env_state[4 * n + k] = st[k];
  env_t[n] = t; ep_ret[n] = 0.0; ep_len[n] = 0; resets[n] = 1;
}

static double linear_schedule(double start_e, double end_e, double duration, double t) {  // dqn.jl:28-31
  const double slope = (end_e - start_e) / duration;
  const double e = slope * t + start_e;
  return e > end_e ? e : end_e;
}

extern "C" CRL_API int crl_dqn_create(const crl_dqn_config* cfg, crl_dqn_ctx** out) {
  if (!cfg || !out) return dfail(CRL_ERR_INVALID, "NULL argument");
  if (cfg->struct_size != (int32_t)sizeof(crl_dqn_config)) return dfail(CRL_ERR_INVALID, "crl_dqn_config.struct_size mismatch");
  if (cfg->num_envs < 1 || cfg->buffer_size < cfg->num_envs) return dfail(CRL_ERR_INVALID, "need 1 <= num_envs <= buffer_size");
  if (cfg->batch_size < 1 || cfg->batch_size > LEARN_B) return dfail(CRL_ERR_INVALID, "batch_size must be in [1, 128]");
  if (cfg->train_freq < 1 || cfg->target_net_freq < 1 || cfg->max_episode_steps < 1 || !(cfg->epsilon_duration > 0.0))
    return dfail(CRL_ERR_INVALID, "train_freq, target_net_freq, max_episode_steps, epsilon_duration must be positive");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) return dfail(CRL_ERR_CUDA, "no CUDA device: libcleanrl_cuda has no CPU fallback");
  if (cfg->device < 0 || cfg->device >= ndev) return dfail(CRL_ERR_INVALID, "device ordinal out of range");
  DCK(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  DCK(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10) return dfail(CRL_ERR_CUDA, "libcleanrl_cuda is built for sm_100a only");
  crl_dqn_ctx* c = new crl_dqn_ctx();
  memset(c, 0, sizeof(*c));
  // from here on a failure must release what was allocated so far (crl_dqn_destroy skips null members)
#define DCKC(call)                                                                                           \
  do {                                                                                                       \
    cudaError_t e__ = (call);                                                                                \
    if (e__ != cudaSuccess) {                                                                                \
      crl_dqn_destroy(c);                                                                                    \
      return dfail(CRL_ERR_CUDA, std::string(#call) + " failed: " + cudaGetErrorString(e__) + " (dqn.cu)"); \
    }                                                                                                        \
  } while (0)
  c->cfg = *cfg;
  const size_t N = cfg->num_envs, C = cfg->buffer_size;
  DCKC(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
  DCKC(dzalloc(&c->q, DQ_P)); DCKC(dzalloc(&c->tgt, DQ_P)); DCKC(dzalloc(&c->m, DQ_P)); DCKC(dzalloc(&c->v, DQ_P));
  DCKC(dzalloc(&c->env_state, 4 * N)); DCKC(dzalloc(&c->env_t, N)); DCKC(dzalloc(&c->ep_ret, N)); DCKC(dzalloc(&c->ep_len, N));
  DCKC(dzalloc(&c->resets, N));
  DCKC(dzalloc(&c->b_state, 4 * C)); DCKC(dzalloc(&c->b_next, 4 * C)); DCKC(dzalloc(&c->b_reward, C)); DCKC(dzalloc(&c->b_action, C));
  DCKC(dzalloc(&c->b_term, C)); DCKC(dzalloc(&c->dev, 1));
  DCKC(dzalloc(&c->h1T, (size_t)LEARN_B * DQ_H1)); DCKC(dzalloc(&c->h2T, (size_t)LEARN_B * DQ_H2)); DCKC(dzalloc(&c->z2T, (size_t)LEARN_B * DQ_H2));
  DCKC(dzalloc(&c->z1T, (size_t)LEARN_B * DQ_H1)); DCKC(dzalloc(&c->xT, (size_t)LEARN_B * DQ_D)); DCKC(dzalloc(&c->dqT, (size_t)LEARN_B * DQ_A));
  DCKC(dzalloc(&c->loss_part, LF_MAX_BLOCKS));
  DCKC(dzalloc(&c->gbuf, DQ_P)); DCKC(dzalloc(&c->lbuf, 1));
  c->world = 1; c->rank = 0; c->env_id_base = 0; c->comm = nullptr;
  DCKC(cudaFuncSetAttribute(dqn_learn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LF_SMEM));
  DCKC(cudaFuncSetAttribute(dqn_learn_upd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LU_SMEM));
  DCKC(cudaFuncSetAttribute(dqn_learn_upd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LU_SMEM));
  DCKC(cudaFuncSetAttribute(dqn_act_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ACT_SMEM));
#undef DCKC
  *out = c;
  return CRL_OK;
}

extern "C" CRL_API int crl_dqn_destroy(crl_dqn_ctx* c) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  cudaSetDevice(c->cfg.device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  void* ptrs[] = {c->q, c->tgt, c->m, c->v, c->env_state, c->env_t, c->ep_ret, c->ep_len, c->resets, c->b_state, c->b_next,
                  c->b_reward, c->b_action, c->b_term, c->dev, c->h1T, c->h2T, c->z2T, c->z1T, c->xT, c->dqT, c->loss_part, c->gbuf, c->lbuf};
  for (void* p : ptrs) if (p) cudaFree(p);
  for (int r = 0; r < CRL_MAX_WORLD; r++)
    if (c->x_peer[r] && c->x_peer[r] != c->x_buf) cudaIpcCloseMemHandle(c->x_peer[r]);
  { void* xp[] = {c->x_buf, c->x_peers_dev, c->x_err}; for (void* q : xp) if (q) cudaFree(q); }
  crl_internal_nccl_comm_destroy(c->comm);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
  return CRL_OK;
}

extern "C" CRL_API int crl_dqn_set_params(crl_dqn_ctx* c, const float* params, int32_t n) {
  if (!c || !params) return dfail(CRL_ERR_INVALID, "NULL argument");
  if (n != DQ_P) return dfail(CRL_ERR_INVALID, "DQN parameter vector must have 10934 floats");
  DCK(cudaSetDevice(c->cfg.device));
  DCK(cudaMemcpyAsync(c->q, params, sizeof(float) * DQ_P, cudaMemcpyHostToDevice, c->stream));
  DCK(cudaMemcpyAsync(c->tgt, c->q, sizeof(float) * DQ_P, cudaMemcpyDeviceToDevice, c->stream));   // deepcopy, dqn.jl:40
  DCK(cudaMemsetAsync(c->m, 0, sizeof(float) * DQ_P, c->stream));
  DCK(cudaMemsetAsync(c->v, 0, sizeof(float) * DQ_P, c->stream));
  DqnDev d;
  memset(&d, 0, sizeof(d));
  DCK(cudaMemcpyAsync(c->dev, &d, sizeof(d), cudaMemcpyHostToDevice, c->stream));
  DCK(cudaStreamSynchronize(c->stream));
  c->bp1 = 0.9; c->bp2 = 0.999;
  c->params_set = true;
  return CRL_OK;
}

extern "C" CRL_API int crl_dqn_get_params(crl_dqn_ctx* c, float* q_params, float* target_params, int32_t n) {
  if (!c || !q_params) return dfail(CRL_ERR_INVALID, "NULL argument");
  if (n != DQ_P) return dfail(CRL_ERR_INVALID, "DQN parameter vector must have 10934 floats");
  DCK(cudaSetDevice(c->cfg.device));
  DCK(cudaMemcpyAsync(q_params, c->q, sizeof(float) * DQ_P, cudaMemcpyDeviceToHost, c->stream));
  if (target_params) DCK(cudaMemcpyAsync(target_params, c->tgt, sizeof(float) * DQ_P, cudaMemcpyDeviceToHost, c->stream));
  DCK(cudaStreamSynchronize(c->stream));
  return CRL_OK;
}

extern "C" CRL_API int crl_dqn_reset(crl_dqn_ctx* c) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  DCK(cudaSetDevice(c->cfg.device));
  const int N = c->cfg.num_envs;
  dqn_reset_kernel<<<(N + 127) / 128, 128, 0, c->stream>>>(N, c->cfg.seed, c->env_id_base, c->env_state, c->env_t, c->ep_ret, c->ep_len, c->resets);
  DCK(cudaGetLastError());
  c->size = 0; c->ptr = 0; c->it = 0; c->learn_steps = 0;   /* launches keeps counting: it is a lifetime counter */
  c->reset_done = true;
  return CRL_OK;
}

extern "C" CRL_API int crl_dqn_comm_init(crl_dqn_ctx* c, const void* id128, int32_t world_size, int32_t rank, int32_t env_id_base) {
  if (!c || !id128) return dfail(CRL_ERR_INVALID, "NULL argument");
  if (world_size < 2 || rank < 0 || rank >= world_size || env_id_base < 0)
    return dfail(CRL_ERR_INVALID, "need world_size >= 2, 0 <= rank < world_size, env_id_base >= 0");
  if (c->comm) return dfail(CRL_ERR_STATE, "crl_dqn_comm_init called twice");
  if (c->reset_done) return dfail(CRL_ERR_STATE, "crl_dqn_comm_init must precede crl_dqn_reset (the env ids change)");
  DCK(cudaSetDevice(c->cfg.device));
  int rc = crl_internal_nccl_comm_init(&c->comm, world_size, rank, id128);
  if (rc != CRL_OK) return rc;
  c->world = world_size; c->rank = rank; c->env_id_base = env_id_base;
  // NCCL connects its channels lazily on the first collective: do that here, not inside the first learning step
  DCK(cudaMemsetAsync(c->lbuf, 0, sizeof(double), c->stream));
  rc = crl_internal_nccl_allreduce_sum(c->comm, c->lbuf, 1, 1, c->stream);
  if (rc != CRL_OK) return rc;
  DCK(cudaMemsetAsync(c->gbuf, 0, sizeof(float) * DQ_P, c->stream));
  rc = crl_internal_nccl_allreduce_sum(c->comm, c->gbuf, DQ_P, 0, c->stream);
  if (rc != CRL_OK) return rc;
  DCK(cudaStreamSynchronize(c->stream));
  if (world_size > CRL_MAX_WORLD) return dfail(CRL_ERR_INVALID, "world_size exceeds CRL_MAX_WORLD");
  if (getenv("CRL_NO_P2P") == nullptr) {
    // peer-memory exchange buffers (same scheme as crl_comm_init): cudaIpc handles travel through one NCCL all-gather,
    // every rank maps all peers; a failure anywhere leaves the NCCL allreduce in place on ALL ranks (one more collective
    // carries the verdict)
    const int W = world_size;
    c->x_stride = (DQ_P + 1 + 7) & ~7;
    const size_t bytes = (size_t)2 * W * c->x_stride * 16;
    bool ok = cudaMalloc(reinterpret_cast<void**>(&c->x_buf), bytes) == cudaSuccess && cudaMemset(c->x_buf, 0, bytes) == cudaSuccess;
    cudaIpcMemHandle_t mine;
    ok = ok && cudaIpcGetMemHandle(&mine, c->x_buf) == cudaSuccess;
    unsigned char* stage = nullptr;
    ok = ok && cudaMalloc(reinterpret_cast<void**>(&stage), (size_t)(W + 1) * sizeof(mine)) == cudaSuccess;
    cudaIpcMemHandle_t all[CRL_MAX_WORLD];
    if (ok) {
      ok = cudaMemcpy(stage, &mine, sizeof(mine), cudaMemcpyHostToDevice) == cudaSuccess;
      ok = ok && crl_internal_nccl_allgather(c->comm, stage, stage + sizeof(mine), sizeof(mine), c->stream) == CRL_OK;
      ok = ok && cudaStreamSynchronize(c->stream) == cudaSuccess;
      ok = ok && cudaMemcpy(all, stage + sizeof(mine), (size_t)W * sizeof(mine), cudaMemcpyDeviceToHost) == cudaSuccess;
    }
    if (stage) cudaFree(stage);
    for (int r = 0; r < W && ok; r++) {
      if (r == rank) { c->x_peer[r] = c->x_buf; continue; }
      void* ptr = nullptr;
      ok = cudaIpcOpenMemHandle(&ptr, all[r], cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
      c->x_peer[r] = static_cast<unsigned char*>(ptr);
    }
    ok = ok && cudaMalloc(reinterpret_cast<void**>(&c->x_peers_dev), CRL_MAX_WORLD * sizeof(void*)) == cudaSuccess;
    ok = ok && cudaMemcpy(c->x_peers_dev, c->x_peer, CRL_MAX_WORLD * sizeof(void*), cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && dzalloc(&c->x_err, 1) == cudaSuccess;
    double verdict = ok ? 1.0 : 0.0;
    DCK(cudaMemcpy(c->lbuf, &verdict, sizeof(double), cudaMemcpyHostToDevice));
    rc = crl_internal_nccl_allreduce_sum(c->comm, c->lbuf, 1, 1, c->stream);
    if (rc != CRL_OK) return rc;
    DCK(cudaStreamSynchronize(c->stream));
    DCK(cudaMemcpy(&verdict, c->lbuf, sizeof(double), cudaMemcpyDeviceToHost));
    cudaGetLastError();
    c->x_on = verdict > W - 0.5;
    const char* e = getenv("CRL_P2P_TIMEOUT_MS");
    int khz = 1965000;
    cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, c->cfg.device);
    c->x_timeout = (long long)((e ? atof(e) : 30000.0) * (double)khz);
  }
  return CRL_OK;
}

extern "C" CRL_API int crl_dqn_run(crl_dqn_ctx* c, int64_t iterations, crl_dqn_stats* stats) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  if (iterations < 0) return dfail(CRL_ERR_INVALID, "iterations must be >= 0");
  if (!c->params_set) return dfail(CRL_ERR_STATE, "crl_dqn_run called before crl_dqn_set_params");
  if (!c->reset_done) return dfail(CRL_ERR_STATE, "crl_dqn_run called before crl_dqn_reset");
  if (c->world > 1 && !c->comm) return dfail(CRL_ERR_STATE, "world_size > 1 but crl_dqn_comm_init did not complete");
  DCK(cudaSetDevice(c->cfg.device));
  const int N = c->cfg.num_envs, C = c->cfg.buffer_size;
  // per-call episode aggregate: clear the three accumulators, keep Adam's powers and the last loss
  DCK(cudaMemsetAsync(&c->dev->sum_return, 0, sizeof(double) * 2 + sizeof(unsigned long long), c->stream));
  double eps = 0.0;
  int64_t k = 0;
  while (k < iterations) {
    // One launch acts for every iteration up to (and including) the next learning step: the parameters are constant in
    // between. Bounded by ACT_MAX_STEPS and by the ring capacity (steps of one launch must not share a slot).
    ActArgs a;
    a.q = c->q; a.env_state = c->env_state; a.env_t = c->env_t; a.ep_ret = c->ep_ret; a.ep_len = c->ep_len; a.resets = c->resets;
    a.b_state = c->b_state; a.b_next = c->b_next; a.b_reward = c->b_reward; a.b_action = c->b_action; a.b_term = c->b_term;
    a.dev = c->dev; a.seed = c->cfg.seed; a.it0 = (unsigned long long)(c->it + 1); a.N = N; a.C = C; a.ptr = c->ptr;
    a.max_steps = c->cfg.max_episode_steps; a.env_id_base = c->env_id_base;
    int ns = 0;
    bool learn = false;
    while (k < iterations && ns < ACT_MAX_STEPS && (long long)(ns + 1) * N <= (long long)C && !learn) {
      c->it += 1;
      k += 1;
      const double gs = (double)c->it * (double)N * (double)c->world;   // global step over all shards
      eps = linear_schedule(c->cfg.epsilon_start, c->cfg.epsilon_end, c->cfg.epsilon_duration, gs);   // dqn.jl:52
      a.eps[ns++] = eps;
      c->ptr = (c->ptr + N) % C;
      c->size = c->size + N > C ? C : c->size + N;
      learn = gs > (double)c->cfg.min_buff_size && c->it % c->cfg.train_freq == 0 && c->size >= c->cfg.batch_size;   // dqn.jl:94
    }
    for (int i = ns; i < ACT_MAX_STEPS; i++) a.eps[i] = 0.0;
    a.n_steps = ns;
    dqn_act_kernel<<<(N + ACT_E - 1) / ACT_E, ACT_THREADS, ACT_SMEM, c->stream>>>(a);
    DCK(cudaGetLastError());
    c->launches += 1;
    if (learn) {
      LearnArgs l;
      memset(&l, 0, sizeof(l));
      l.q = c->q; l.tgt = c->tgt; l.m = c->m; l.v = c->v;
      l.b_state = c->b_state; l.b_next = c->b_next; l.b_reward = c->b_reward; l.b_action = c->b_action; l.b_term = c->b_term;
      l.dev = c->dev; l.seed = c->cfg.seed; l.learn_step = (unsigned long long)c->learn_steps; l.gamma = c->cfg.gamma;
      l.lr = c->cfg.lr; l.B = c->cfg.batch_size; l.size = c->size;
      l.copy_target = (c->it % c->cfg.target_net_freq == 0) ? 1 : 0;                                             // dqn.jl:111
      l.h1T = c->h1T; l.h2T = c->h2T; l.z2T = c->z2T; l.z1T = c->z1T; l.xT = c->xT; l.dqT = c->dqT;
      l.loss_part = c->loss_part; l.bp1 = c->bp1; l.bp2 = c->bp2;
      l.B_scale = l.B * c->world; l.rank = c->rank; l.gbuf = c->gbuf; l.lbuf = c->lbuf;
      const int fwd_blocks = (l.B + LF_S - 1) / LF_S;
      dqn_learn_fwd_kernel<<<fwd_blocks, LF_T, LF_SMEM, c->stream>>>(l);
      DCK(cudaGetLastError());
      if (c->world == 1) {
        dqn_learn_upd_kernel<false><<<LU_A_BLOCKS + LU_B_BLOCKS + LU_C_BLOCKS, LU_T, LU_SMEM, c->stream>>>(l, fwd_blocks);
        DCK(cudaGetLastError());
        c->launches += 2;
      } else {
        // one gradient exchange per learning step, then Adam on the sums. Peer memory (default): the update kernel pushes
        // its gradient into every peer's buffer and dqn_adam_kernel collects: no collective call, two launches.
        // Fallback (CRL_NO_P2P=1 or no peer access): two NCCL allreduces on the handle's stream in between.
        if (c->x_on) {
          l.x_peers = c->x_peers_dev; l.x_local = c->x_buf; l.x_world = c->world; l.x_stride = c->x_stride;
          l.x_flag = (unsigned int)(c->learn_steps + 1); l.x_slot = (int)((c->learn_steps + 1) & 1);
          l.x_err = c->x_err; l.x_timeout = c->x_timeout;
        }
        dqn_learn_upd_kernel<true><<<LU_A_BLOCKS + LU_B_BLOCKS + LU_C_BLOCKS, LU_T, LU_SMEM, c->stream>>>(l, fwd_blocks);
        DCK(cudaGetLastError());
        if (!c->x_on) {
          int rc = crl_internal_nccl_allreduce_sum(c->comm, c->gbuf, DQ_P, 0, c->stream);
          if (rc != CRL_OK) return rc;
          rc = crl_internal_nccl_allreduce_sum(c->comm, c->lbuf, 1, 1, c->stream);
          if (rc != CRL_OK) return rc;
        }
        dqn_adam_kernel<<<(DQ_P + 1 + 255) / 256, 256, 0, c->stream>>>(l);
        DCK(cudaGetLastError());
        c->launches += 3;
      }
      c->bp1 *= 0.9; c->bp2 *= 0.999;
      c->learn_steps += 1;
    }
  }
  if (stats) {
    DqnDev d;
    DCK(cudaMemcpyAsync(&d, c->dev, sizeof(d), cudaMemcpyDeviceToHost, c->stream));
    DCK(cudaStreamSynchronize(c->stream));
    stats->last_loss = d.last_loss; stats->sum_return = d.sum_return; stats->sum_length = d.sum_length; stats->epsilon = eps;
    stats->episodes = (int64_t)d.episodes; stats->learn_steps = c->learn_steps; stats->iterations = c->it;
    stats->kernel_launches = c->launches;
    if (c->x_on) {
      int err = 0;
      DCK(cudaMemcpy(&err, c->x_err, sizeof(int), cudaMemcpyDeviceToHost));
      if (err) return dfail(CRL_ERR_NCCL, "peer-memory gradient exchange timed out waiting for another rank");
    }
  }
  return CRL_OK;
}

extern "C" CRL_API int crl_dqn_read_buffer(crl_dqn_ctx* c, float* state, int32_t* action, float* reward, float* next_state,
                                           uint8_t* terminal, int32_t* size, int32_t* ptr) {
  if (!c) return dfail(CRL_ERR_INVALID, "ctx is NULL");
  DCK(cudaSetDevice(c->cfg.device));
  const size_t C = c->cfg.buffer_size;
  if (state) DCK(cudaMemcpyAsync(state, c->b_state, C * 16, cudaMemcpyDeviceToHost, c->stream));
  if (next_state) DCK(cudaMemcpyAsync(next_state, c->b_next, C * 16, cudaMemcpyDeviceToHost, c->stream));
  if (action) DCK(cudaMemcpyAsync(action, c->b_action, C * 4, cudaMemcpyDeviceToHost, c->stream));
  if (reward) DCK(cudaMemcpyAsync(reward, c->b_reward, C * 4, cudaMemcpyDeviceToHost, c->stream));
  if (terminal) DCK(cudaMemcpyAsync(terminal, c->b_term, C, cudaMemcpyDeviceToHost, c->stream));
  DCK(cudaStreamSynchronize(c->stream));
  if (size) *size = c->size;
  if (ptr) *ptr = c->ptr;
  return CRL_OK;
}

static int dqn_raw_device_check() {
  int dev = 0;
  DCK(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  DCK(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) return dfail(CRL_ERR_CUDA, "libcleanrl_cuda is built for sm_100a only");
  return CRL_OK;
}

extern "C" CRL_API int crl_dqn_forward_raw(const float* params, const float* obs, float* q_out, int64_t n, void* stream) {
  if (n < 0 || (n > 0 && (!params || !obs || !q_out))) return dfail(CRL_ERR_INVALID, "NULL argument or n < 0");
  if (((uintptr_t)params | (uintptr_t)obs) % 16 || (uintptr_t)q_out % 8)
    return dfail(CRL_ERR_INVALID, "params and obs must be 16-byte aligned, q_out 8-byte aligned");
  if (n == 0) return CRL_OK;
  if (int rc = dqn_raw_device_check()) return rc;
  DCK(cudaFuncSetAttribute(dqn_forward_raw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FWD_RAW_SMEM));
  const int64_t grid = (n + ACT_E - 1) / ACT_E;
  if (grid > 0x7fffffff) return dfail(CRL_ERR_INVALID, "n too large");
  dqn_forward_raw_kernel<<<(unsigned)grid, ACT_T, FWD_RAW_SMEM, (cudaStream_t)stream>>>(params, obs, q_out, n);
  DCK(cudaGetLastError());
  return CRL_OK;
}

extern "C" CRL_API int crl_dqn_loss_raw(const float* q, const float* tgt, int32_t B, const float* state, const int32_t* action,
                                        const float* reward, const float* next_state, const uint8_t* terminal, double gamma,
                                        float* grads_out, double* loss_out, void* stream) {
  if (!q || !tgt || !state || !action || !reward || !next_state || !terminal || !grads_out || !loss_out)
    return dfail(CRL_ERR_INVALID, "NULL argument");
  if (B < 1 || B > LEARN_B) return dfail(CRL_ERR_INVALID, "B must be in [1, 128]");
  if (((uintptr_t)q | (uintptr_t)tgt | (uintptr_t)state | (uintptr_t)next_state) % 16)
    return dfail(CRL_ERR_INVALID, "q, tgt, state and next_state must be 16-byte aligned");
  if (int rc = dqn_raw_device_check()) return rc;
  DCK(cudaFuncSetAttribute(dqn_learn_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LF_SMEM));
  DCK(cudaFuncSetAttribute(dqn_learn_upd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LU_SMEM));
  const cudaStream_t s = (cudaStream_t)stream;
  // the learning step of crl_dqn_run on rows 0..B-1, its update kernel in the variant that leaves the gradient in gbuf
  // (= grads_out) and the squared-error sum in lbuf instead of applying Adam (no peers: x_push does nothing)
  LearnArgs l;
  memset(&l, 0, sizeof(l));
  l.q = const_cast<float*>(q); l.tgt = const_cast<float*>(tgt);
  l.b_state = state; l.b_next = next_state; l.b_reward = reward; l.b_action = action; l.b_term = terminal;
  l.gamma = gamma; l.B = B; l.size = B; l.in_order = 1; l.B_scale = B; l.gbuf = grads_out;
  float* scratch = nullptr;
  double* dscratch = nullptr;
  const size_t nf = (size_t)LEARN_B * (2 * DQ_H1 + 2 * DQ_H2 + DQ_D + DQ_A);
  DCK(cudaMalloc(reinterpret_cast<void**>(&scratch), nf * sizeof(float)));
  if (cudaMalloc(reinterpret_cast<void**>(&dscratch), (LF_MAX_BLOCKS + 1) * sizeof(double)) != cudaSuccess) {
    cudaFree(scratch);
    return dfail(CRL_ERR_CUDA, "cudaMalloc failed (crl_dqn_loss_raw)");
  }
  l.h1T = scratch; l.z1T = l.h1T + LEARN_B * DQ_H1; l.h2T = l.z1T + LEARN_B * DQ_H1; l.z2T = l.h2T + LEARN_B * DQ_H2;
  l.xT = l.z2T + LEARN_B * DQ_H2; l.dqT = l.xT + LEARN_B * DQ_D;
  l.loss_part = dscratch; l.lbuf = dscratch + LF_MAX_BLOCKS;
  const int fwd_blocks = (B + LF_S - 1) / LF_S;
  dqn_learn_fwd_kernel<<<fwd_blocks, LF_T, LF_SMEM, s>>>(l);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) {
    dqn_learn_upd_kernel<true><<<LU_A_BLOCKS + LU_B_BLOCKS + LU_C_BLOCKS, LU_T, LU_SMEM, s>>>(l, fwd_blocks);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) {
    dqn_loss_raw_finish_kernel<<<1, 1, 0, s>>>(l.lbuf, B, loss_out);
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);   // the scratch is freed below
  cudaFree(scratch);
  cudaFree(dscratch);
  if (e != cudaSuccess) return dfail(CRL_ERR_CUDA, std::string("crl_dqn_loss_raw failed: ") + cudaGetErrorString(e));
  return CRL_OK;
}
