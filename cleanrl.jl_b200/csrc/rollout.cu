// rollout.cu — persistent rollout kernel (replaces the loop ppo.jl:123-166) and the raw
// env-step / policy-forward entry points.
//
// One launch runs all T steps. A CTA of 256 threads owns 32 envs for the whole rollout: the
// policy weights are constant during a rollout and nothing couples envs (SURVEY §3.5), so no
// grid-wide synchronisation is needed. Per step: the two 64-64 MLPs are evaluated for the 32
// envs as register-tiled FFMA layers out of shared memory (weights staged once per launch),
// then warp 0 (one lane per env) samples the action, steps the env in registers, writes the
// [T][N] rollout buffer with coalesced stores (state as one float4 per (t,n)), and resets
// finished envs on the spot.
#include "kernels.h"
#include "mlp_tile.cuh"

namespace {

constexpr int RE = 32;            // envs per CTA
constexpr int ROLL_FWD = CRL_THREADS;   // warps 0-7: the two MLPs; warp 0 also owns the envs (one lane per env)
constexpr int ROLL_THREADS = ROLL_FWD + 64;   // warps 8, 9: speculation warps (see rollout_kernel)
// grids larger than the GPU (BIG): 4 forward warps with 8 x 4 register tiles (see fwd_layer_8x4), 2 CTAs per SM
constexpr int BIG_FWD = 128, BIG_THREADS = BIG_FWD + 64;
constexpr int BAR_FWD = 1, BAR_SPEC = 2, BAR_BOOK = 3;      // named barriers: the forward threads / speculation warps -> warp 0 / bookkeeping warp -> output-layer threads

__device__ __forceinline__ void nbar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void nbar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

template <int ENV> struct RolloutSmem {
  using G = TileGeom<4, 2>;
  using E = EnvTraits<ENV>;
  static constexpr int SP = G::S_PAD;
  static constexpr int PARAMS = 0;
  static constexpr int X = PARAMS + SmemParams<ENV>::SIZE;
  static constexpr int H1 = X + CRL_MAXD * SP;
  static constexpr int H2 = H1 + G::ROWS * SP;
  static constexpr int OUT = H2 + G::ROWS * SP;
  static constexpr int ST = OUT + 4 * RE;          // [4][RE] env state as the speculation warps read it
  static constexpr int SPEC = ST + 4 * RE;         // [2 actions][4][RE] successor states (CartPole)
  static constexpr int RST = SPEC + 2 * 4 * RE;    // [4][RE] the state each env takes at its next reset
  static constexpr int NOISE = RST + 4 * RE;       // double[RE] uniform (Float64, StatsBase) or float[2][RE] normals
  static constexpr int USED = NOISE + 2 * RE;      // int[RE]: warp 0 consumed the prepared reset state
  static constexpr int BOOK = USED + RE;           // per env: action (int), action (float, Gaussian head), reward, done
  static constexpr int FLOATS = BOOK + 4 * RE;
  static constexpr size_t BYTES = FLOATS * sizeof(float);
  static_assert((NOISE % 2) == 0, "the Float64 uniforms need 8-byte alignment");
};

// -DROLL_TRACE: clock stamps of the phases of step 64 of CTA 0 (warps 0 and 5), printed from the kernel (development aid)
#ifdef ROLL_TRACE
#define RTR(i) do { if (tr) tr[i] = clock64(); } while (0)
#else
#define RTR(i) do { } while (0)
#endif

// this thread's row of the output layer in registers (threads < RE * (A + 1): output o = tid / RE of env tid % RE):
// constant during a launch, so the 64 broadcast loads per step become none
template <int ENV> struct HeadRow { float w[CRL_H]; float b; };
template <int ENV> __device__ __forceinline__ void load_head_row(const float* sp, HeadRow<ENV>& hr) {
  using E = EnvTraits<ENV>;
  const int o = threadIdx.x / RE;
#pragma unroll
  for (int k = 0; k < CRL_H; k++) hr.w[k] = 0.0f;
  hr.b = 0.0f;
  if (threadIdx.x >= RE * (E::A + 1)) return;
  if (o < E::A) {
    const float* a = sp + SmemParams<ENV>::ACTOR;
#pragma unroll
    for (int k = 0; k < CRL_H; k++) hr.w[k] = a[NetOff<E::D, E::A>::W3 + k * E::A + o];
    hr.b = a[NetOff<E::D, E::A>::B3 + o];
  } else {
    const float* c = sp + SmemParams<ENV>::CRITIC;
#pragma unroll
    for (int k = 0; k < CRL_H; k++) hr.w[k] = c[NetOff<E::D, 1>::W3 + k];
    hr.b = c[NetOff<E::D, 1>::B3];
  }
}

// both nets forward for the 32 samples whose observations sit in xs; heads -> so[o][e]
// (o < A: actor logits/mean, o == A: critic value). Called by the 256 forward threads only (named barrier BAR_FWD).
template <int ENV, bool BOOKSYNC = false>
__device__ __forceinline__ void forward32(const ThreadCoord<TileGeom<4, 2>>& tc, float* smem, const HeadRow<ENV>& hr,
                                          long long* tr = nullptr) {
  using G = TileGeom<4, 2>;
  using E = EnvTraits<ENV>;
  using SM = RolloutSmem<ENV>;
  constexpr int SP = G::S_PAD;
  float* sp = smem + SM::PARAMS;
  float* xs = smem + SM::X;
  float* h1 = smem + SM::H1;
  float* h2 = smem + SM::H2;
  float* so = smem + SM::OUT;
  const float* np = sp + net_base<ENV>(tc.net);
  using NO = NetOff<E::D, 1>;  // W1,B1,W2,B2,W3 offsets do not depend on the head width
  RTR(0);
  tile_layer_fwd4<G, E::D>(tc, np + NO::W1, np + NO::B1, xs, h1 + tc.net * CRL_H * SP);
  RTR(1);
  nbar_sync(BAR_FWD, ROLL_FWD);
  RTR(2);
  tile_layer_fwd4<G, CRL_H>(tc, np + NO::W2, np + NO::B2, h1 + tc.net * CRL_H * SP, h2 + tc.net * CRL_H * SP);
  RTR(3);
  nbar_sync(BAR_FWD, ROLL_FWD);
  RTR(4);
  if (threadIdx.x < RE * (E::A + 1)) {
    const int o = threadIdx.x / RE, e = threadIdx.x % RE;
    const float* hrow = h2 + (o < E::A ? 0 : CRL_H) * SP + e;
    float hv[CRL_H];
#pragma unroll
    for (int k = 0; k < CRL_H; k++) hv[k] = hrow[k * SP];   // all 64 loads in flight before the (serial) chain starts
    if (BOOKSYNC) nbar_sync(BAR_BOOK, RE * (E::A + 1) + 32);   // the bookkeeping warp has read the previous step's outputs
    float acc = 0.0f;
#pragma unroll
    for (int k = 0; k < CRL_H; k++) acc = fmaf(hr.w[k], hv[k], acc);
    acc += hr.b;
    so[o * RE + e] = acc;
  }
  RTR(5);
  nbar_sync(BAR_FWD, ROLL_FWD);
  RTR(6);
}

// The layers for grids larger than the GPU, where the rollout is bound by throughput and not by the latency of one
// step: 128 forward threads, thread (q, p) owns the 8 neurons 8q.. of net q / 8 and the 4 envs 4p.. (an 8 x 4 register
// tile: per k two 128-bit weight loads and one 128-bit activation load feed 16 packed FMAs, 1.5 B of shared-memory
// traffic per FMA instead of the 4 x 4 tile's 2 B; the shared-memory crossbar is what bounds these layers,
// profiles/r2_pipe_probe.txt). A warp is 4 q x 8 p with the 8 lanes of a quarter-warp on one q: its weight loads are
// one broadcast address, its activation loads and its stores 128 contiguous bytes. At 4096 envs (one CTA per SM,
// latency-bound) this variant is SLOWER than 4 x 4 tiles on 8 warps (0.541 vs 0.473 ms) and is not used there.
// Every accumulator is one fma chain over ascending k, as in tile_layer: same bits.
struct FwdCoord8x4 {
  int q, p, net, nb;   // neuron group, sample group, net, first neuron within the net
  __device__ FwdCoord8x4() {
    const int lane = threadIdx.x & 31, w = (threadIdx.x >> 5) & 3;
    q = w * 4 + (lane >> 3);
    p = lane & 7;
    net = q >> 3;
    nb = 8 * (q & 7);
  }
};
template <int K>
__device__ __forceinline__ void fwd_layer_8x4(const FwdCoord8x4& fc, const float* __restrict__ Wt, const float* __restrict__ bias,
                                              const float* __restrict__ in, float* __restrict__ out) {
  constexpr int SP = RE + 4, PF = 2;
  const float* wp = Wt + fc.nb;
  const float* ap = in + 4 * fc.p;
  const float4 b0 = *reinterpret_cast<const float4*>(bias + fc.nb), b1 = *reinterpret_cast<const float4*>(bias + fc.nb + 4);
  float2 acc[8][2];
#pragma unroll
  for (int j = 0; j < 8; j++) acc[j][0] = acc[j][1] = make_float2(0.0f, 0.0f);
  float4 w0[PF], w1[PF], av[PF];
#pragma unroll
  for (int i = 0; i < PF; i++) {
    if (i < K) {
      w0[i] = *reinterpret_cast<const float4*>(wp + i * CRL_H);
      w1[i] = *reinterpret_cast<const float4*>(wp + i * CRL_H + 4);
      av[i] = *reinterpret_cast<const float4*>(ap + i * SP);
    }
  }
#pragma unroll
  for (int k0 = 0; k0 < K; k0 += PF) {
    float4 w0n[PF], w1n[PF], avn[PF];
#pragma unroll
    for (int i = 0; i < PF; i++) {
      if (k0 + PF + i < K) {
        w0n[i] = *reinterpret_cast<const float4*>(wp + (k0 + PF + i) * CRL_H);
        w1n[i] = *reinterpret_cast<const float4*>(wp + (k0 + PF + i) * CRL_H + 4);
        avn[i] = *reinterpret_cast<const float4*>(ap + (k0 + PF + i) * SP);
      }
    }
#pragma unroll
    for (int i = 0; i < PF; i++) {
      if (k0 + i < K) {
        const float2 a01 = make_float2(av[i].x, av[i].y), a23 = make_float2(av[i].z, av[i].w);
#pragma unroll
        for (int j = 0; j < 8; j++) {
          const float wj = j < 4 ? f4_get(w0[i], j) : f4_get(w1[i], j - 4);
          const float2 ww = make_float2(wj, wj);
          acc[j][0] = __ffma2_rn(ww, a01, acc[j][0]);
          acc[j][1] = __ffma2_rn(ww, a23, acc[j][1]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < PF; i++) { w0[i] = w0n[i]; w1[i] = w1n[i]; av[i] = avn[i]; }
  }
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const float b = j < 4 ? f4_get(b0, j) : f4_get(b1, j - 4);
    const float2 t0 = tanh_fast2(__fadd2_rn(acc[j][0], make_float2(b, b)));
    const float2 t1 = tanh_fast2(__fadd2_rn(acc[j][1], make_float2(b, b)));
    *reinterpret_cast<float4*>(out + (fc.nb + j) * SP + 4 * fc.p) = make_float4(t0.x, t0.y, t1.x, t1.y);
  }
}
// forward32 for the BIG variant (output layer weights from shared memory)
template <int ENV>
__device__ __forceinline__ void forward32_big(const FwdCoord8x4& fc, float* smem) {
  using E = EnvTraits<ENV>;
  using SM = RolloutSmem<ENV>;
  constexpr int SP = RE + 4;
  static_assert(SP == TileGeom<4, 2>::S_PAD, "both forward variants share one activation layout");
  float* sp = smem + SM::PARAMS;
  float* xs = smem + SM::X;
  float* h1 = smem + SM::H1;
  float* h2 = smem + SM::H2;
  float* so = smem + SM::OUT;
  const float* np = sp + net_base<ENV>(fc.net);
  using NO = NetOff<E::D, 1>;
  fwd_layer_8x4<E::D>(fc, np + NO::W1, np + NO::B1, xs, h1 + fc.net * CRL_H * SP);
  nbar_sync(BAR_FWD, BIG_FWD);
  fwd_layer_8x4<CRL_H>(fc, np + NO::W2, np + NO::B2, h1 + fc.net * CRL_H * SP, h2 + fc.net * CRL_H * SP);
  nbar_sync(BAR_FWD, BIG_FWD);
  if (threadIdx.x < RE * (E::A + 1)) {
    const int o = threadIdx.x / RE, e = threadIdx.x % RE;
    const float* hrow = h2 + (o < E::A ? 0 : CRL_H) * SP + e;
    nbar_sync(BAR_BOOK, RE * (E::A + 1) + 32);   // the bookkeeping warp has read the previous step's outputs
    float acc = 0.0f;
    if (o < E::A) {
      const float* a = sp + SmemParams<ENV>::ACTOR;
#pragma unroll 16
      for (int k = 0; k < CRL_H; k++) acc = fmaf(a[NetOff<E::D, E::A>::W3 + k * E::A + o], hrow[k * SP], acc);
      acc += a[NetOff<E::D, E::A>::B3 + o];
    } else {
      const float* c = sp + SmemParams<ENV>::CRITIC;
#pragma unroll 16
      for (int k = 0; k < CRL_H; k++) acc = fmaf(c[NetOff<E::D, 1>::W3 + k], hrow[k * SP], acc);
      acc += c[NetOff<E::D, 1>::B3];
    }
    so[o * RE + e] = acc;
  }
  nbar_sync(BAR_FWD, BIG_FWD);
}

// Persistent rollout. Warps 0-7 evaluate the two MLPs for the CTA's 32 envs; warp 0 (one lane per env) then samples
// the action and advances its env. Only what the NEXT observation depends on stays on that serial phase (softmax
// probabilities, the inverse-CDF sample, picking the successor state, termination, reset): everything else is done by
// two extra warps in the shadow of the forward pass:
//   warp 8   the step's action noise (Philox: the Float64 uniform of StatsBase.sample, or the Gaussian head's normals)
//            and, CartPole, the successor state for action 0
//   warp 9   CartPole: the successor state for action 1; the state every env will take at its NEXT reset (Philox keyed
//            by the env's reset counter), refreshed after warp 0 consumed it; and the BOOKKEEPING of the previous step:
//            log-probability, the [T][N] buffer stores (Buffer.add!), episode length / return, episode records and
//            aggregates. Warp 0 hands it (action, reward, done) through shared memory; logits and value it reads from
//            the forward pass's outputs, the observation it read itself one step earlier.
// Warp 0 picks the successor of the action it sampled (same device function, same inputs: bit-identical to stepping
// after the fact). The injected-noise test modes (action_noise / reset_noise) read their draws on warp 0 as before.
// BIG = true: more CTAs than SMs (N / 32 > SM count): 4 forward warps with 8 x 4 tiles, two resident CTAs per SM (shared memory: 77 KB each).
template <int ENV, bool BIG>
__global__ void __launch_bounds__(BIG ? BIG_THREADS : ROLL_THREADS, BIG ? 2 : 1) rollout_kernel(RolloutArgs a) {
  constexpr int FWD = BIG ? BIG_FWD : ROLL_FWD;   // forward threads; the two speculation warps follow them
  constexpr int SW0 = FWD / 32;
  using G = TileGeom<4, 2>;
  using E = EnvTraits<ENV>;
  using SM = RolloutSmem<ENV>;
  constexpr int SP = G::S_PAD;
  constexpr int D = E::D, A = E::A, S = E::S;
  constexpr bool CART = ENV == CRL_ENV_CARTPOLE;
  extern __shared__ __align__(16) float smem[];
  float* sp = smem + SM::PARAMS;
  float* xs = smem + SM::X;
  float* so = smem + SM::OUT;
  float* st_s = smem + SM::ST;
  float* spec_s = smem + SM::SPEC;
  float* rst_s = smem + SM::RST;
  double* noise_d = reinterpret_cast<double*>(smem + SM::NOISE);
  float* noise_f = smem + SM::NOISE;
  int* used_s = reinterpret_cast<int*>(smem + SM::USED);
  int* act_s = reinterpret_cast<int*>(smem + SM::BOOK);
  float* actf_s = smem + SM::BOOK + RE;
  float* rew_s = smem + SM::BOOK + 2 * RE;
  int* done_s = reinterpret_cast<int*>(smem + SM::BOOK + 3 * RE);
  const ThreadCoord<G> tc;
  const FwdCoord8x4 fc;

  load_params<ENV>(a.params, sp);
  for (int i = threadIdx.x; i < CRL_MAXD * SP; i += blockDim.x) xs[i] = 0.0f;

  const int warp = threadIdx.x >> 5;
  const int e = threadIdx.x & 31;  // env lane of warps 0, 8 and 9
  const long long n = (long long)blockIdx.x * RE + e;
  const bool fwd = threadIdx.x < FWD;
  const bool owner = threadIdx.x < RE;
  const bool booker = warp == SW0 + 1;
  const bool in_range = n < a.N;
  const bool valid = owner && in_range;
  const unsigned long long step0 = a.ds->policy_step;
  const uint32_t gid = (uint32_t)(a.env_id_base + (int)n);

  // warp 0: the env itself
  float st[S];
  float obs[D];
  int env_t = 0;
  uint32_t resets = 0;  // warp 0: the env's counter; warp 9: the counter the prepared reset state was drawn for
  bool done_flag = false;  // Q3: ppo.jl:170 — is_terminated(env) after reset! is false
  // warp 9: the episode bookkeeping of the env
  int ep_len = 0;
  double ep_ret = 0.0;
  bool prev_done = false;   // next_done of the step being recorded (terminal[t], ppo.jl:139)
  float obs_b[D];           // the observation the step being recorded acted on
  unsigned long long agg_n = 0;
  double agg_ret = 0.0, agg_len = 0.0, agg_max = -INFINITY;
  // episode record whose slot is still on its way back from the atomic (stored one step later)
  bool rec_pending = false;
  unsigned int rec_slot = 0;
  crl_episode rec;
  rec.step = 0; rec.env = 0; rec.length = 0; rec._pad = 0; rec.episode_return = 0.0;

#pragma unroll
  for (int i = 0; i < S; i++) st[i] = 0.0f;
#pragma unroll
  for (int k = 0; k < D; k++) obs_b[k] = 0.0f;
  if (valid) {
#pragma unroll
    for (int i = 0; i < S; i++) st[i] = a.env_state[n * S + i];
    env_t = a.env_t[n];
    resets = a.reset_count[n];
  }
  if (booker && in_range) {
    ep_len = a.ep_length[n];
    ep_ret = a.ep_return[n];
    resets = a.reset_count[n];
  }
  __syncthreads();
  HeadRow<ENV> hr;
  if (!BIG) load_head_row<ENV>(sp, hr);
  if (owner) {
    env_obs<ENV>(st, obs);  // Q3: ppo.jl:169 — state(env) refreshed (post-reset state)
#pragma unroll
    for (int k = 0; k < D; k++) xs[k * SP + e] = obs[k];
#pragma unroll
    for (int i = 0; i < S; i++) st_s[i * RE + e] = st[i];
    used_s[e] = 0;
  }
  auto prepare_reset = [&]() {   // warp 9: the state env e takes at reset number `resets` (multi_thread_env.jl:105-111)
    float u4[4], rs[S];
    int rt;
    rng_reset_uniforms(a.seed, gid, resets, u4);
    env_reset<ENV>(rs, rt, u4);
#pragma unroll
    for (int i = 0; i < S; i++) rst_s[i * RE + e] = rs[i];
  };
  if (booker && !a.reset_noise) prepare_reset();

  // warp 9: everything of step tb that the next observation does not depend on (ppo.jl:125, 133-140, 145-165)
  auto book = [&](int tb, const float (&zv)[A + 1], int act_i, float act_f, float r, bool dn) {
    const long long b = (long long)tb * a.N + n;
    ep_len += 1;  // ppo.jl:125
    float logprob;
    if (!E::CONT) {
      // logsoftmax [NNlib], the same operations warp 0 ran for the probabilities
      float m = zv[0];
#pragma unroll
      for (int k = 1; k < A; k++) m = fmaxf(m, zv[k]);
      float sum = 0.0f;
#pragma unroll
      for (int k = 0; k < A; k++) sum = __fadd_rn(sum, expf(__fsub_rn(zv[k], m)));
      const float ls = logf(sum);
      logprob = __fsub_rn(__fsub_rn(zv[0], m), ls);
#pragma unroll
      for (int k = 1; k < A; k++) logprob = (act_i == k) ? __fsub_rn(__fsub_rn(zv[k], m), ls) : logprob;
    } else {
      float lps = 0.0f;
#pragma unroll
      for (int k = 0; k < A; k++) {
        const float mean = zv[k];
        const float logstd = sp[SmemParams<ENV>::LOGSTD + k];
        const float sd = expf(logstd);
        const float diff = __fsub_rn(act_f, mean);   // A = 1
        const float q = __fdiv_rn(-__fmul_rn(diff, diff), __fmul_rn(__fmul_rn(2.0f, sd), sd));
        lps = __fadd_rn(lps, __fsub_rn(__fsub_rn(q, logstd), 0.9189385332046727f));
      }
      logprob = lps;
    }
    if (rec_pending) {   // the previous record: its slot has long arrived
      if (rec_slot < (unsigned int)a.ep_capacity) a.records[rec_slot] = rec;
      rec_pending = false;
    }
    ep_ret += (double)r;    // ppo.jl:145
    if (in_range) {
      // Buffer.add!, ppo.jl:133-140: state = next_obs, terminal = next_done (previous step)
      if (D == 4) {
        reinterpret_cast<float4*>(a.state)[b] = make_float4(obs_b[0], obs_b[1], obs_b[2], obs_b[3]);
      } else {
#pragma unroll
        for (int k = 0; k < D; k++) a.state[b * D + k] = obs_b[k];
      }
      if (!E::CONT) reinterpret_cast<int32_t*>(a.action)[b] = act_i;
      else reinterpret_cast<float*>(a.action)[b * A] = act_f;
      a.logprob[b] = logprob;
      a.value[b] = zv[A];
      a.terminal[b] = prev_done ? 1 : 0;
      a.reward[b] = r;  // ppo.jl:132
      if (dn) {         // ppo.jl:147-165
        rec_slot = atomicAdd(&a.eb->count, 1u);
        rec_pending = true;
        rec.step = tb; rec.env = (int)n; rec.length = ep_len; rec._pad = 0; rec.episode_return = ep_ret;
        agg_n += 1; agg_ret += ep_ret; agg_len += (double)ep_len; agg_max = fmax(agg_max, ep_ret);
        ep_ret = 0.0;
        ep_len = 0;
      }
    }
    prev_done = dn;
  };
  static_assert(!E::CONT || A == 1, "the Gaussian head hands one action per env to the bookkeeping warp");
  __syncthreads();

  for (int t = 0; t < a.T; t++) {
    if (!fwd) {
      // ---- speculation / bookkeeping warps, in the shadow of the forward pass
      if (booker) {
        // what step t - 1 left behind: copied to registers before the output layer of this step may overwrite so[]
        float zv[A + 1];
#pragma unroll
        for (int k = 0; k <= A; k++) zv[k] = so[k * RE + e];
        const int act_i = act_s[e];
        const float act_f = actf_s[e], r = rew_s[e];
        const bool dn = done_s[e] != 0;
        nbar_arrive(BAR_BOOK, RE * (A + 1) + 32);
        if (t > 0) book(t - 1, zv, act_i, act_f, r, dn);
#pragma unroll
        for (int k = 0; k < D; k++) obs_b[k] = xs[k * SP + e];   // the observation step t acts on
        if (!a.reset_noise && used_s[e]) {
          resets += 1;
          prepare_reset();
          used_s[e] = 0;
        }
      }
      if (warp == SW0 && !a.action_noise) {
        if (!E::CONT) {
          noise_d[e] = in_range ? rng_action_uniform(a.seed, gid, step0 + (unsigned long long)t) : 0.0;
        } else {
          float zn[2] = {0.0f, 0.0f};
          if (in_range) rng_action_normals(a.seed, gid, step0 + (unsigned long long)t, zn);
          noise_f[e] = zn[0];
          noise_f[RE + e] = zn[1];
        }
      }
      if (CART) {
        float s4[4];
#pragma unroll
        for (int i = 0; i < 4; i++) s4[i] = st_s[i * RE + e];
        cartpole_dynamics(s4, warp - SW0);
#pragma unroll
        for (int i = 0; i < 4; i++) spec_s[((warp - SW0) * 4 + i) * RE + e] = s4[i];
      }
      __threadfence_block();
      nbar_arrive(BAR_SPEC, RE + 64);
    } else {
      // ends with a barrier of the forward threads; so[] is ready
      if (BIG) forward32_big<ENV>(fc, smem); else forward32<ENV, true>(tc, smem, hr);
      if (owner) {
        const long long b = (long long)t * a.N + n;
        int act_i = 0;
        float act_f = 0.0f;
        if (!E::CONT) {
          // get_action, ppo.jl:22-29: softmax [NNlib], then
          // StatsBase.sample(Weights(p)): t = rand()*sum(p); walk cw += p[i] while cw < t.
          float z[A], p[A];
#pragma unroll
          for (int k = 0; k < A; k++) z[k] = so[k * RE + e];
          float m = z[0];
#pragma unroll
          for (int k = 1; k < A; k++) m = fmaxf(m, z[k]);
          float ex[A], sum = 0.0f;
#pragma unroll
          for (int k = 0; k < A; k++) { ex[k] = expf(__fsub_rn(z[k], m)); sum = __fadd_rn(sum, ex[k]); }
          float psum = 0.0f;
#pragma unroll
          for (int k = 0; k < A; k++) {
            p[k] = __fdiv_rn(ex[k], sum);
            psum = __fadd_rn(psum, p[k]);
          }
          nbar_sync(BAR_SPEC, RE + 64);   // the speculation warps have delivered this step (and recorded the last one)
          double u = 0.0;
          if (valid) u = a.action_noise ? a.action_noise[b] : noise_d[e];
          const double tt = __dmul_rn(u, (double)psum);
          float cw = p[0];
          int i = 0;
#pragma unroll
          for (int k = 1; k < A; k++) {
            if ((double)cw < tt && i == k - 1) { i = k; cw = __fadd_rn(cw, p[k]); }
          }
          act_i = i;
        } else {
          // Gaussian head (CleanRL-Python convention; the reference has none)
          nbar_sync(BAR_SPEC, RE + 64);
          float zn = 0.0f;
          if (valid) zn = a.action_noise ? (float)a.action_noise[b * A] : noise_f[e];
          const float mean = so[e];
          const float sd = expf(sp[SmemParams<ENV>::LOGSTD]);
          act_f = __fadd_rn(mean, __fmul_rn(sd, zn));
        }
        // env(action), ppo.jl:130
        float r;
        bool dn;
        if (CART) {
          // the successor computed by warp 8 + act_i from this very state: cartpole_step without the wait
#pragma unroll
          for (int i = 0; i < 4; i++) st[i] = spec_s[(act_i * 4 + i) * RE + e];
          env_t += 1;
          cartpole_outcome(st, env_t, a.max_steps, r, dn);
        } else {
          pendulum_step(st, env_t, act_f, a.max_steps, r, dn);
        }
        env_obs<ENV>(st, obs);  // ppo.jl:143 — copied BEFORE reset! (Q2: stale terminal obs)
        done_flag = dn;         // ppo.jl:144
        act_s[e] = act_i; actf_s[e] = act_f; rew_s[e] = r; done_s[e] = dn ? 1 : 0;   // for the bookkeeping warp
        if (valid && dn) {      // ppo.jl:147-165
          if (a.reset_noise) {
            const float4 v = reinterpret_cast<const float4*>(a.reset_noise)[b];
            const float u4[4] = {v.x, v.y, v.z, v.w};
            env_reset<ENV>(st, env_t, u4);  // only terminated envs, multi_thread_env.jl:105-111
          } else {
#pragma unroll
            for (int i = 0; i < S; i++) st[i] = rst_s[i * RE + e];   // prepared by warp 9 for this reset counter
            env_t = 0;
            used_s[e] = 1;
          }
          resets += 1;
          if (a.fresh_obs_after_reset) env_obs<ENV>(st, obs);  // a2c.jl:108 then :52 (PPO: stale obs, Q2)
        }
#pragma unroll
        for (int k = 0; k < D; k++) xs[k * SP + e] = obs[k];
#pragma unroll
        for (int i = 0; i < S; i++) st_s[i * RE + e] = st[i];
      }
    }
    __syncthreads();
  }
  if (!fwd) {
    // the last step's bookkeeping, then the episode state and aggregates go back
    if (booker) {
      float zv[A + 1];
#pragma unroll
      for (int k = 0; k <= A; k++) zv[k] = so[k * RE + e];
      const int act_i = act_s[e];
      const float act_f = actf_s[e], r = rew_s[e];
      const bool dn = done_s[e] != 0;
      nbar_arrive(BAR_BOOK, RE * (A + 1) + 32);   // the bootstrap pass may overwrite so[] now
      book(a.T - 1, zv, act_i, act_f, r, dn);
      if (rec_pending && rec_slot < (unsigned int)a.ep_capacity) a.records[rec_slot] = rec;
      if (in_range) {
        a.ep_length[n] = ep_len;
        a.ep_return[n] = ep_ret;
      }
      const double sr = warp_sum(agg_ret), sl = warp_sum(agg_len), mx = warp_max(agg_max);
      unsigned long long cn = agg_n;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) cn += __shfl_xor_sync(0xffffffffu, cn, o);
      if (e == 0 && cn > 0) {
        atomicAdd(&a.eb->n_episodes, cn);
        atomicAdd(&a.eb->sum_return, sr);
        atomicAdd(&a.eb->sum_length, sl);
        unsigned long long* addr = reinterpret_cast<unsigned long long*>(&a.eb->max_return);
        unsigned long long old = *addr, assumed;
        do {
          assumed = old;
          if (__longlong_as_double((long long)assumed) >= mx) break;
          old = atomicCAS(addr, assumed, (unsigned long long)__double_as_longlong(mx));
        } while (assumed != old);
      }
    }
    return;   // only named barriers among the forward threads follow
  }

  // Bootstrap value for GAE: next_values = critic(state(env)) with the refreshed (post-reset)
  // observation, ppo.jl:169-171. The weights cannot change between here and crl_gae.
  float obs_last[D];
#pragma unroll
  for (int k = 0; k < D; k++) obs_last[k] = obs[k];
  if (owner) {
    float fresh[D];
    env_obs<ENV>(st, fresh);
#pragma unroll
    for (int k = 0; k < D; k++) xs[k * SP + e] = fresh[k];
  }
  nbar_sync(BAR_FWD, FWD);
  if (BIG) forward32_big<ENV>(fc, smem); else forward32<ENV, true>(tc, smem, hr);
  if (valid) {
    a.next_value[n] = so[A * RE + e];
#pragma unroll
    for (int i = 0; i < S; i++) a.env_state[n * S + i] = st[i];
    a.env_t[n] = env_t;
    a.reset_count[n] = resets;
#pragma unroll
    for (int k = 0; k < D; k++) a.next_obs[n * D + k] = obs_last[k];
    a.next_done[n] = done_flag ? 1 : 0;
  }
}

// ---- raw kernels (parity tests) --------------------------------------------------------
template <int ENV>
__global__ void env_step_raw_kernel(float* state, int* t, const void* action, float* reward, uint8_t* done,
                                    long long n, int max_steps) {
  constexpr int S = EnvTraits<ENV>::S;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float st[S];
#pragma unroll
  for (int k = 0; k < S; k++) st[k] = state[i * S + k];
  int tt = t[i];
  float r;
  bool dn;
  if (ENV == CRL_ENV_CARTPOLE) cartpole_step(st, tt, reinterpret_cast<const int32_t*>(action)[i], max_steps, r, dn);
  else pendulum_step(st, tt, reinterpret_cast<const float*>(action)[i], max_steps, r, dn);
#pragma unroll
  for (int k = 0; k < S; k++) state[i * S + k] = st[k];
  t[i] = tt;
  reward[i] = r;
  done[i] = dn ? 1 : 0;
}

// same tile code as the rollout: 32 observations per CTA
template <int ENV>
__global__ void __launch_bounds__(CRL_THREADS) policy_forward_raw_kernel(const float* params, const float* obs,
                                                                         float* out_policy, float* logp,
                                                                         float* value, long long n) {
  using G = TileGeom<4, 2>;
  using E = EnvTraits<ENV>;
  using SM = RolloutSmem<ENV>;
  constexpr int SP = G::S_PAD;
  constexpr int D = E::D, A = E::A;
  extern __shared__ __align__(16) float smem[];
  float* xs = smem + SM::X;
  float* so = smem + SM::OUT;
  const ThreadCoord<G> tc;
  load_params<ENV>(params, smem + SM::PARAMS);
  const int e = threadIdx.x;
  const long long i = (long long)blockIdx.x * RE + e;
  if (e < RE) {
#pragma unroll
    for (int k = 0; k < D; k++) xs[k * SP + e] = i < n ? obs[i * D + k] : 0.0f;
  }
  __syncthreads();
  HeadRow<ENV> hr;
  load_head_row<ENV>(smem + SM::PARAMS, hr);
  forward32<ENV>(tc, smem, hr);
  if (e < RE && i < n) {
    float z[A];
#pragma unroll
    for (int k = 0; k < A; k++) { z[k] = so[k * RE + e]; out_policy[i * A + k] = z[k]; }
    value[i] = so[A * RE + e];
    if (!E::CONT) {
      float m = z[0];
#pragma unroll
      for (int k = 1; k < A; k++) m = fmaxf(m, z[k]);
      float sum = 0.0f;
#pragma unroll
      for (int k = 0; k < A; k++) sum = __fadd_rn(sum, expf(__fsub_rn(z[k], m)));
      const float ls = logf(sum);
#pragma unroll
      for (int k = 0; k < A; k++) logp[i * A + k] = __fsub_rn(__fsub_rn(z[k], m), ls);
    }
  }
}

template <int ENV> cudaError_t launch_rollout_t(const RolloutArgs& a, cudaStream_t s) {
  const int grid = (a.N + RE - 1) / RE;
  static int sms = 0;
  if (sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  }
  if (grid > sms) rollout_kernel<ENV, true><<<grid, BIG_THREADS, RolloutSmem<ENV>::BYTES, s>>>(a);
  else rollout_kernel<ENV, false><<<grid, ROLL_THREADS, RolloutSmem<ENV>::BYTES, s>>>(a);
  return cudaGetLastError();
}

template <int ENV>
cudaError_t launch_policy_forward_t(const float* params, const float* obs, float* out_policy, float* logp,
                                    float* value, long long n, cudaStream_t s) {
  const long long grid = (n + RE - 1) / RE;
  if (grid == 0) return cudaSuccess;
  policy_forward_raw_kernel<ENV><<<(unsigned)grid, CRL_THREADS, RolloutSmem<ENV>::BYTES, s>>>(params, obs, out_policy,
                                                                                              logp, value, n);
  return cudaGetLastError();
}

__global__ void episode_buf_init_kernel(EpisodeBuf* eb) {
  eb->count = 0; eb->_pad = 0; eb->n_episodes = 0ull; eb->sum_return = 0.0; eb->sum_length = 0.0;
  eb->max_return = -INFINITY;
}

template <int ENV> cudaError_t init_attrs_t() {
  cudaError_t e = cudaFuncSetAttribute(rollout_kernel<ENV, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)RolloutSmem<ENV>::BYTES);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(rollout_kernel<ENV, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RolloutSmem<ENV>::BYTES);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(policy_forward_raw_kernel<ENV>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)RolloutSmem<ENV>::BYTES);
}

}  // namespace

// opt in to > 48 KB dynamic shared memory (per device; must run outside stream capture)
cudaError_t kernels_init_rollout() {
  cudaError_t e = init_attrs_t<CRL_ENV_CARTPOLE>();
  if (e != cudaSuccess) return e;
  return init_attrs_t<CRL_ENV_PENDULUM>();
}

cudaError_t launch_episode_buf_init(EpisodeBuf* eb, cudaStream_t s) {
  episode_buf_init_kernel<<<1, 1, 0, s>>>(eb);
  return cudaGetLastError();
}

cudaError_t launch_rollout(int env_kind, const RolloutArgs& a, cudaStream_t s) {
  return env_kind == CRL_ENV_CARTPOLE ? launch_rollout_t<CRL_ENV_CARTPOLE>(a, s) : launch_rollout_t<CRL_ENV_PENDULUM>(a, s);
}

cudaError_t launch_env_step_raw(int env_kind, float* state, int* t, const void* action, float* reward,
                                uint8_t* done, long long n, int max_steps, cudaStream_t s) {
  if (n == 0) return cudaSuccess;
  const unsigned grid = (unsigned)((n + 127) / 128);
  if (env_kind == CRL_ENV_CARTPOLE)
    env_step_raw_kernel<CRL_ENV_CARTPOLE><<<grid, 128, 0, s>>>(state, t, action, reward, done, n, max_steps);
  else
    env_step_raw_kernel<CRL_ENV_PENDULUM><<<grid, 128, 0, s>>>(state, t, action, reward, done, n, max_steps);
  return cudaGetLastError();
}

cudaError_t launch_policy_forward_raw(int env_kind, const float* params, const float* obs, float* out_policy,
                                      float* logp, float* value, long long n, cudaStream_t s) {
  return env_kind == CRL_ENV_CARTPOLE
             ? launch_policy_forward_t<CRL_ENV_CARTPOLE>(params, obs, out_policy, logp, value, n, s)
             : launch_policy_forward_t<CRL_ENV_PENDULUM>(params, obs, out_policy, logp, value, n, s);
}

// ---- env reset / refresh (ppo.jl:112-115) ------------------------------------------------
namespace {
template <int ENV>
__global__ void env_reset_kernel(int N, unsigned long long seed, int env_id_base, float* env_state, int* env_t,
                                 double* ep_return, int* ep_length, uint32_t* reset_count, float* next_obs,
                                 uint8_t* next_done) {
  constexpr int S = EnvTraits<ENV>::S, D = EnvTraits<ENV>::D;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float u4[4], st[S], obs[D];
  const uint32_t k = reset_count[n];
  rng_reset_uniforms(seed, (uint32_t)(env_id_base + n), k, u4);
  int t;
  env_reset<ENV>(st, t, u4);
  env_obs<ENV>(st, obs);
#pragma unroll
  for (int i = 0; i < S; i++) env_state[n * S + i] = st[i];
#pragma unroll
  for (int i = 0; i < D; i++) next_obs[n * D + i] = obs[i];
  env_t[n] = t;
  reset_count[n] = k + 1;
  next_done[n] = 0;
  ep_return[n] = 0.0;
  ep_length[n] = 0;
}
template <int ENV>
__global__ void env_refresh_kernel(int N, const float* env_state, float* next_obs, uint8_t* next_done) {
  constexpr int S = EnvTraits<ENV>::S, D = EnvTraits<ENV>::D;
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float st[S], obs[D];
#pragma unroll
  for (int i = 0; i < S; i++) st[i] = env_state[n * S + i];
  env_obs<ENV>(st, obs);
#pragma unroll
  for (int i = 0; i < D; i++) next_obs[n * D + i] = obs[i];
  next_done[n] = 0;
}
}  // namespace

cudaError_t launch_env_reset(int env_kind, int N, unsigned long long seed, int env_id_base, float* env_state,
                             int* env_t, double* ep_return, int* ep_length, uint32_t* reset_count, float* next_obs,
                             uint8_t* next_done, cudaStream_t s) {
  const int grid = (N + 127) / 128;
  if (env_kind == CRL_ENV_CARTPOLE)
    env_reset_kernel<CRL_ENV_CARTPOLE><<<grid, 128, 0, s>>>(N, seed, env_id_base, env_state, env_t, ep_return, ep_length,
                                                           reset_count, next_obs, next_done);
  else
    env_reset_kernel<CRL_ENV_PENDULUM><<<grid, 128, 0, s>>>(N, seed, env_id_base, env_state, env_t, ep_return, ep_length,
                                                           reset_count, next_obs, next_done);
  return cudaGetLastError();
}

cudaError_t launch_env_refresh(int env_kind, int N, const float* env_state, float* next_obs, uint8_t* next_done,
                               cudaStream_t s) {
  const int grid = (N + 127) / 128;
  if (env_kind == CRL_ENV_CARTPOLE) env_refresh_kernel<CRL_ENV_CARTPOLE><<<grid, 128, 0, s>>>(N, env_state, next_obs, next_done);
  else env_refresh_kernel<CRL_ENV_PENDULUM><<<grid, 128, 0, s>>>(N, env_state, next_obs, next_done);
  return cudaGetLastError();
}
