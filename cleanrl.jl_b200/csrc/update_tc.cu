// update_tc.cu — the PPO minibatch forward + loss + backward (ppo.jl:197-246) with every 64-wide contraction on
// the 5th-generation tensor cores (tcgen05.mma kind::tf32, accumulators in TMEM), as 3xTF32 so the results stay
// within fp32 tolerance of the oracle (operands are split x = hi + lo with hi = TF32(x); hi*hi + lo*hi + hi*lo).
//
// Work decomposition. Actor and critic gradients are independent given the rollout data, so a CTA owns ONE net and a
// persistent stride of 128-sample tiles; the first `tc_actor_ctas` CTAs take the actor, the rest the critic. Inside
// a CTA sample s of the tile IS TMEM lane s: warp w works on lanes 32*(w%4).. (the only lanes tcgen05.ld/st lets
// it touch) and on the feature half (w/4)*32.. of every 64-wide row, so each thread owns (1 sample, 32 features).
//
// Warp 0 also issues the MMAs: the other warps hand each operand set over with a NON-blocking named-barrier arrive
// (only warp 0 syncs on it) and everybody picks the results up on the mbarrier the issue is committed to, so the
// warps never wait for each other and the next tile's first layer is computed in the shadow of the current tile's
// first contraction. (A dedicated ninth issuer warp would cap the kernel at 168 registers per thread.)
//
// Per tile (the four contractions are the only cross-thread data flow besides one 2-float head exchange):
//   L1   h1 = tanh(W1 x + b1) on the CUDA cores (K = 4); hi/lo go to TMEM (A operand of G1, tcgen05.st) and,
//        feature-major, to shared memory (B operand of G2)
//   G1   z2[s][j] = sum_k h1[s][k] W2(j,k)            A = TMEM, B = weight image (rows j)          M128 N64 K64 x3
//   E1   h2 = tanh(z2 + b2); head; per-sample loss and d(loss)/d(head) in Float64 where Julia promotes (same code
//        as the FFMA kernel); dz2 = (W3^T dl) .* (1 - h2^2): hi/lo to TMEM (A of G3) and feature-major, hi rows
//        stacked over lo rows, to shared memory (A of G2); dW3/db2 by warp reduce-scatter shuffles
//   G3   dh1[s][k] = sum_j dz2[s][j] W2(j,k)          A = TMEM, B = weight image (rows k)          M128 N64 K64 x3
//   G2   dW2(j,k) += sum_s dz2[s][j] h1[s][k]         A = [dz2_hi ; dz2_lo] (M = 128), B = h1_hi then h1_lo: rows j
//        and 64+j of the accumulator add up to the full 4-term product; accumulates in TMEM over ALL tiles of the CTA
//   E3   dz1 = dh1 .* (1 - h1^2), hi/lo written in place over h1's feature-major copy
//   G4   dW1(k,d), db1(k) += sum_s dz1[s][k] x~[d][s]  A = [dz1_hi ; dz1_lo] (M = 128), B = x~^T hi then lo (rows
//        x_0..x_D-1, ones; N = 16 with the two 8-row groups aliased by SBO = 0); accumulates in TMEM over all tiles
// The weight-gradient accumulators are read out of TMEM once per launch.
//
// Shared memory (bytes): weight images 65,536 | dz2^T stacked 73,728 | h1^T/dz1^T hi,lo 73,728 | x~^T 8,192 |
// small parameters + scratch ~6 KB = ~222 KB: one CTA per SM. The feature-major operands use a 144-byte chunk
// stride (LBO) so that the 32 lanes of a warp (32 consecutive samples) store one feature conflict-free.
// Layouts and descriptor conventions were validated on a B200 by tools/tc_probe.cu and tools/tc_probe3.cu.
#include "kernels.h"
#include "mlp_tile.cuh"
#include "update_common.cuh"

#include <stdlib.h>

#include <type_traits>

namespace {
using namespace crl_upd;

// -DTC_TRACE: per-phase clock stamps of tile 3 of CTA 0 (warps 0 and 5), printed from the kernel (development aid)
#ifdef TC_TRACE
#define TR(i) do { if (trace_on) tr[i] = clock64(); } while (0)
#else
#define TR(i) do { } while (0)
#endif

constexpr int TC_S = 128;        // samples per tile = TMEM lanes
constexpr int TC_NG = 2;         // feature groups per sample (8 warps, 32 features per thread)
constexpr int TC_THREADS = 128 * TC_NG;  // 4 lane quadrants x TC_NG feature groups
constexpr int TC_WARPS = TC_THREADS / 32;
constexpr int TC_FG = CRL_H / TC_NG;     // features per thread
constexpr int F_LBO = 144, F_SBO = 32 * F_LBO;  // bytes; feature-major operand: rows r, K = 128 samples
__device__ __forceinline__ int f_off(int r, int s) { return (r & 7) * 4 + (r >> 3) * (F_SBO / 4) + (s >> 2) * (F_LBO / 4) + (s & 3); }
// x~^T (rows x_0..x_D-1, ones, zeros): two more 8-row groups (hi, lo) right behind h1^T, same strides, so that
// [h1_hi ; h1_lo ; x~_hi ; x~_lo] is ONE 144-row B operand
__device__ __forceinline__ int xt_off(int d, int s) { return d * 4 + (s >> 2) * (F_LBO / 4) + (s & 3); }
constexpr int XT_GROUP = F_SBO / 4;  // floats per 8-row group

// TMEM columns (fp32): z2/dh1 accumulator (A W_hi^T | A_hi W_lo^T: 128) | A operand hi (64) | A operand lo (64) |
// dW2 accumulator (x h1_hi | x h1_lo | x x~: 144) | dW1,db1 accumulator (x x~_hi | x x~_lo: 16)
constexpr uint32_t COL_D = 0, COL_AH = 128, COL_AL = 192, COL_D2 = 256, COL_D4 = 400, COL_P = 416, TMEM_COLS = 512;
// COL_P: h1^2 - 1 (the tanh derivative E3 needs) waits in 64 spare TMEM columns from the start of the tile instead of
// being rebuilt from the hi/lo rows of h1^T in shared memory (4 scalar loads + an add per feature pair)
// named barriers: 1-3 hand an operand set to the issuing warp (it syncs, the other warps only arrive), 4-7 = head exchange
// of lane quadrant 0-3
constexpr int BAR_G1 = 1, BAR_G3 = 2, BAR_G4 = 3, BAR_X = 4;
template <int ENV> struct TcSmem {
  static constexpr int WB = 0;                      // [4][4096] weight images of this CTA's net
  static constexpr int FZ = WB + 4 * TC_W_FLOATS;   // dz2^T, rows 0-63 hi, 64-127 lo
  static constexpr int FH = FZ + 16 * F_SBO / 4;    // h1^T (later dz1^T), rows 0-63 hi, 64-127 lo
  static constexpr int XT = FH + 16 * F_SBO / 4;    // [hi | lo] 8-row groups, directly behind FH
  static constexpr int W1P = XT + 2 * XT_GROUP;     // [32 pairs][4][2]: W1(2p + e, d)
  static constexpr int B1 = W1P + 4 * CRL_H;
  static constexpr int B2 = B1 + CRL_H;
  static constexpr int W3P = B2 + CRL_H;            // [2][64]: W3(o, f)
  static constexpr int B3 = W3P + 2 * CRL_H;        // b3[2], logstd[2]
  static constexpr int EXCH = B3 + 8;               // [TC_NG feature groups][2 outputs][128 samples]
  static constexpr int RED = EXCH + TC_NG * 2 * TC_S;   // 16 doubles (block sums) + 16 floats (block min)
  static constexpr int KEYS = RED + 48;
  static constexpr int FLOATS = KEYS + 8;
  static constexpr size_t BYTES = FLOATS * sizeof(float);
  static_assert(BYTES + 256 <= 227 * 1024, "loss_grad_tc shared memory exceeds 227 KB");
};

// ---------------------------------------------------------------- tcgen05 / mbarrier wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// kind::tf32, fp32 accumulate, both operands K-major
__device__ __forceinline__ constexpr uint32_t make_idesc(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void mma_ss(uint32_t d, uint64_t a, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
               ::"r"(d), "l"(a), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void mma_ts(uint32_t d, uint32_t a_tmem, uint64_t b, uint32_t idesc, uint32_t acc) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n"
               ::"r"(d), "r"(a_tmem), "l"(b), "r"(idesc), "r"(acc) : "memory");
}
// descriptors as (lo, hi) words: only the start-address field in lo changes between the K steps of one operand
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr, uint32_t lbo_bytes) { return ((saddr >> 4) & 0x3FFF) | ((lbo_bytes >> 4) << 16); }
__device__ __forceinline__ constexpr uint32_t desc_hi(uint32_t sbo_bytes) { return ((sbo_bytes >> 4) & 0x3FFF) | (1u << 14); }
__device__ __forceinline__ uint64_t pack64(uint32_t lo, uint32_t hi) {
  uint64_t d;
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
  return d;
}
__device__ __forceinline__ void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void mma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t done = 0;
  while (!done)
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                 : "=r"(done) : "r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void proxy_fence() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float* v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
               ::"r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
               "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
               "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
               "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15])) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float* v) {
  uint32_t r[16];
  __syncwarp();
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                 "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]) : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}

// two N-column rows (an accumulator's hi*W_hi and hi*W_lo halves) requested back to back behind ONE wait: the second
// load's latency hides behind the first instead of following it
__device__ __forceinline__ void tmem_ld16_issue(uint32_t taddr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                 "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]) : "r"(taddr));
}
template <int N> __device__ __forceinline__ void tmem_ld_pair(uint32_t ta, uint32_t tb, float* va, float* vb) {
  static_assert(N == 16 || N == 32, "");
  uint32_t ra[N], rb[N];
  __syncwarp();
#pragma unroll
  for (int i = 0; i < N; i += 16) tmem_ld16_issue(ta + i, ra + i);
#pragma unroll
  for (int i = 0; i < N; i += 16) tmem_ld16_issue(tb + i, rb + i);
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < N; i++) { va[i] = __uint_as_float(ra[i]); vb[i] = __uint_as_float(rb[i]); }
}

template <int N> __device__ __forceinline__ void tmem_ld_triple(uint32_t ta, uint32_t tb, uint32_t tc, float* va, float* vb, float* vc) {
  static_assert(N == 16 || N == 32, "");
  uint32_t ra[N], rb[N], rc[N];
  __syncwarp();
#pragma unroll
  for (int i = 0; i < N; i += 16) tmem_ld16_issue(ta + i, ra + i);
#pragma unroll
  for (int i = 0; i < N; i += 16) tmem_ld16_issue(tb + i, rb + i);
#pragma unroll
  for (int i = 0; i < N; i += 16) tmem_ld16_issue(tc + i, rc + i);
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < N; i++) { va[i] = __uint_as_float(ra[i]); vb[i] = __uint_as_float(rb[i]); vc[i] = __uint_as_float(rc[i]); }
}

template <int N> __device__ __forceinline__ void tmem_st_n(uint32_t taddr, const float* v) {
  static_assert(N == 16 || N == 32, "");
  tmem_st16(taddr, v);
  if (N == 32) tmem_st16(taddr + 16, v + 16);
}

// ---------------------------------------------------------------- packed FP32 helpers (f2, f2s, tanh_fast2: device_math.cuh)
// tanh_fast for this kernel: the same rational function, but (a) the argument is clamped to +-sqrt(66) instead of the
// result being replaced by +-1 beyond it (the rational is 1 - 1.2e-7 there; 4 min/max on the ALU pipe instead of 2
// compares + 2 selects + 2 sign copies) and (b) the reciprocal is MUFU.RCP without the Newton step (<= 1 ulp). Both are
// below the 3xTF32 error of the contractions around it (1.2e-6); the rollout and the FFMA kernel keep the exact form.
// A tanh_fast2 call costs ~35 issue cycles per warp (tools/pipe_probe.cu), 32 calls per thread and tile.
__device__ __forceinline__ float2 tanh_upd2(float2 x) {
  const float lim = 8.1240384f;   // sqrt(66)
  x.x = fminf(fmaxf(x.x, -lim), lim);
  x.y = fminf(fmaxf(x.y, -lim), lim);
  const float2 x2 = __fmul2_rn(x, x);
  float2 n = __ffma2_rn(x2, f2s(1.587199e-8f), f2s(2.2332108e-5f));
  n = __ffma2_rn(x2, n, f2s(0.0035974074f));
  n = __ffma2_rn(x2, n, f2s(0.1346604f));
  n = __ffma2_rn(x2, n, f2s(1.0f));
  float2 d = __ffma2_rn(x2, f2s(8.7767893e-7f), f2s(0.0003453992f));
  d = __ffma2_rn(x2, d, f2s(0.026262015f));
  d = __ffma2_rn(x2, d, f2s(0.4679937f));
  d = __ffma2_rn(x2, d, f2s(1.0f));
  float2 r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.x) : "f"(d.x));
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r.y) : "f"(d.y));
  return __fmul2_rn(x, __fmul2_rn(n, r));
}
// x = hi + lo with hi = TF32(x) (see tf32_hi), two values at once
__device__ __forceinline__ void split2(float2 v, float2& hi, float2& lo) {
  hi = f2(tf32_hi(v.x), tf32_hi(v.y));
  lo = __ffma2_rn(hi, f2s(-1.0f), v);
}

// Warp reduce-scatter: on return v[r] (r < V/32) holds the sum over the 32 lanes of the original element
// r + (V/32) * lane. V/2 + V/4 + ... shuffles instead of 5 V for V separate butterfly reductions.
template <int N, int OFF, int V> __device__ __forceinline__ void rs_step(float (&v)[V], int lane) {
  const bool up = (lane & OFF) != 0;
#pragma unroll
  for (int i = 0; i < N; i++) {
    const float keep = up ? v[i + N] : v[i];
    const float send = up ? v[i] : v[i + N];
    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, OFF);
  }
}
template <int V> __device__ __forceinline__ void warp_reduce_scatter(float (&v)[V], int lane) {
  rs_step<V / 2, 16>(v, lane);
  rs_step<V / 4, 8>(v, lane);
  rs_step<V / 8, 4>(v, lane);
  rs_step<V / 16, 2>(v, lane);
  rs_step<V / 32, 1>(v, lane);
}
// element index held in v[r] after warp_reduce_scatter<V>: bit b of the lane selects the upper half at step b
template <int V> __device__ __forceinline__ int rs_index(int lane, int r) {
  return r + (V / 32) * ((lane & 1) | (lane & 2) | (lane & 4) | (lane & 8) | (lane & 16));
}

template <int I> using IC = std::integral_constant<int, I>;

template <int ENV> struct Sample {
  float x[4];
  float adv, oldlp, R, V;
  float actf[EnvTraits<ENV>::A];
  int act;
  bool valid;
};
// buffer index of minibatch position m (-1 past the end); loaded one tile ahead of the fields that depend on it
__device__ __forceinline__ int load_index(const UpdateArgs& a, const uint32_t* keys, int m) {
  return m < a.M ? sample_index(a.idx, keys, m) : -1;
}
template <int ENV, int NET>
__device__ __forceinline__ void load_sample(const UpdateArgs& a, int b, Sample<ENV>& in) {
  using E = EnvTraits<ENV>;
  in.valid = b >= 0;
  in.x[0] = in.x[1] = in.x[2] = in.x[3] = 0.0f;
  in.adv = in.oldlp = in.R = in.V = 0.0f;
  in.act = 0;
#pragma unroll
  for (int k = 0; k < E::A; k++) in.actf[k] = 0.0f;
  if (!in.valid) return;
  if (E::D == 4) {
    const float4 x4 = __ldg(reinterpret_cast<const float4*>(a.states) + b);
    in.x[0] = x4.x; in.x[1] = x4.y; in.x[2] = x4.z; in.x[3] = x4.w;
  } else {
#pragma unroll
    for (int k = 0; k < E::D; k++) in.x[k] = __ldg(a.states + (long long)b * E::D + k);
  }
  if (NET == 0) {
    if (a.algo == 1) { in.R = __ldg(a.returns + b); in.V = __ldg(a.values + b); }
    in.adv = __ldg(a.advantages + b);
    in.oldlp = __ldg(a.logprobs + b);
    if (E::CONT) {
#pragma unroll
      for (int k = 0; k < E::A; k++) in.actf[k] = __ldg(reinterpret_cast<const float*>(a.actions) + (long long)b * E::A + k);
    } else {
      in.act = __ldg(reinterpret_cast<const int*>(a.actions) + b);
    }
  } else {
    in.R = __ldg(a.returns + b);
    in.V = __ldg(a.values + b);
  }
}

struct TcBars { unsigned long long pbar, g1, g2, g3, g4; };

template <int ENV, int NET>
__device__ __forceinline__ void tc_body(const UpdateArgs& a, float* smem, TcBars* bars, const uint32_t tmem) {
  using E = EnvTraits<ENV>;
  using SM = TcSmem<ENV>;
  using NO = NetOff<E::D, 1>;
  using NA = NetOff<E::D, E::A>;
  constexpr int D = E::D, A = E::A;
  constexpr int NOUT = NET == 0 ? A : 1;
  float* wb = smem + SM::WB;
  float* fz = smem + SM::FZ;
  float* fh = smem + SM::FH;
  float* xt = smem + SM::XT;
  const float4* w1v = reinterpret_cast<const float4*>(smem + SM::W1P);   // [pair][d][2] as two float4 per pair
  const float2* b1q = reinterpret_cast<const float2*>(smem + SM::B1);
  const float2* b2q = reinterpret_cast<const float2*>(smem + SM::B2);
  const float2* w3q = reinterpret_cast<const float2*>(smem + SM::W3P);   // [o][32 pairs]
  const float* b3s = smem + SM::B3;
  float* exch = smem + SM::EXCH;
  double* red = reinterpret_cast<double*>(smem + SM::RED);
  const uint32_t* keys = reinterpret_cast<const uint32_t*>(smem + SM::KEYS);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int q = warp & 3, g = warp >> 2;
  const int s = q * 32 + lane;   // sample of the tile = TMEM lane
  const int f0 = g * TC_FG;      // this thread's feature half
  const uint32_t lane_addr = tmem + ((uint32_t)(q * 32) << 16);
  const uint32_t bar1 = smem_u32(&bars->g1), bar2 = smem_u32(&bars->g2), bar3 = smem_u32(&bars->g3), bar4 = smem_u32(&bars->g4);

  const int n_cta = NET == 0 ? a.tc_actor_ctas : (int)gridDim.x - a.tc_actor_ctas;
  const int cta = NET == 0 ? (int)blockIdx.x : (int)blockIdx.x - a.tc_actor_ctas;
  const int n_tiles = (a.M + TC_S - 1) / TC_S;

  // minibatch scalars (same derivation as loss_grad_kernel)
  const bool spec = a.mode == LG_SPEC;
  const bool a2c = a.algo == 1;
  float mean_f, std_f, s_f;
  double Mg, cnt_over_M;
  if (spec) {
    double sa = 0.0, sa2 = 0.0;
#pragma unroll
    for (int i = 0; i < ADV_CHUNKS; i++) { sa += a.advparts[2 * i]; sa2 += a.advparts[2 * i + 1]; }
    Mg = (double)a.M * (double)a.world;
    const double mean = sa / Mg;
    double var = (sa2 - Mg * mean * mean) / (Mg - 1.0);
    if (var < 0.0) var = 0.0;
    mean_f = (float)mean; std_f = (float)sqrt(var); s_f = 0.0f; cnt_over_M = 0.0;
  } else {
    mean_f = a.fin->adv_mean; std_f = a.fin->adv_std; s_f = a.fin->s_unclipped;
    Mg = a.fin->M_global;
    cnt_over_M = (double)a.fin->cnt / Mg;
  }
  const float c = a.clip_coef;
  const float lo_c = 1.0f - c, hi_c = 1.0f + c;
  // loop-invariant Float64 factors, hoisted as reciprocals (one rounding in the 53rd bit instead of a division per
  // sample; invisible after the cast to Float32)
  const double inv_std = 1.0 / ((double)std_f + 1e-8), inv_Mg = 1.0 / Mg;
  const double ent_scale = (double)a.ent_coeff / ((double)A * Mg), v_scale = (double)a.v_coef * 0.5 / Mg;

  // accumulators that live for the whole kernel
  double st_pg = 0.0, st_vmax = 0.0, st_ent = 0.0, st_s = 0.0, g_logstd[A];
  float st_min = INFINITY;
  float2 gw3[NOUT][TC_FG / 2];  // dW3(o, f) summed over this thread's samples; reduced over the lanes at the end
  float gb3[NOUT];
#pragma unroll
  for (int k = 0; k < A; k++) g_logstd[k] = 0.0;
#pragma unroll
  for (int o = 0; o < NOUT; o++) {
    gb3[o] = 0.0f;
#pragma unroll
    for (int i = 0; i < TC_FG / 2; i++) gw3[o][i] = f2s(0.0f);
  }

  const uint32_t wb_a = smem_u32(wb), fz_a = smem_u32(fz), fh_a = smem_u32(fh), xt_a = smem_u32(xt);

  // ---- MMA issue (warp 0, one lane). Descriptor words are loop constants + an immediate per K step.
  // An MMA instruction costs ~50 cycles of operand fetch whatever its N, so the hi/lo products are stacked along N:
  // every operand is read once per K step.
  const uint32_t idesc64 = make_idesc(128, 64), idesc128 = make_idesc(128, 128), idesc144 = make_idesc(128, 144),
                 idesc16 = make_idesc(128, 16);
  const uint32_t w_hi = desc_hi(TC_W_SBO), f_hi = desc_hi(F_SBO);
  const uint32_t w1d = desc_lo(wb_a, TC_W_LBO), w3d = desc_lo(wb_a + 2 * TC_W_FLOATS * 4, TC_W_LBO);  // [W_hi ; W_lo], 128 rows
  const uint32_t fzd = desc_lo(fz_a, F_LBO), fhd = desc_lo(fh_a, F_LBO), xtd = desc_lo(xt_a, F_LBO);
  constexpr uint32_t WK = 2 * TC_W_LBO / 16, FK = 2 * F_LBO / 16;  // descriptor step per K = 8
  // hand-over point: the other warps only arrive, warp 0 waits for them and issues
  auto handover = [&](int bar_id, auto&& issue) {
    if (warp == 0) {
      bar_sync(bar_id, TC_THREADS);
      if (lane == 0) { tc_fence_after(); issue(); }
      __syncwarp();
    } else {
      bar_arrive(bar_id, TC_THREADS);
    }
  };
  // D[:, 0:64] = A_hi W_hi^T + A_lo W_hi^T, D[:, 64:128] = A_hi W_lo^T (added by the reader)
  auto issue_ts = [&](uint32_t wd, uint32_t bar) {
#pragma unroll
    for (int ks = 0; ks < 8; ks++) mma_ts(tmem + COL_D, tmem + COL_AH + ks * 8, pack64(wd + ks * WK, w_hi), idesc128, ks ? 1u : 0u);
#pragma unroll
    for (int ks = 0; ks < 8; ks++) mma_ts(tmem + COL_D, tmem + COL_AL + ks * 8, pack64(wd + ks * WK, w_hi), idesc64, 1u);
    mma_commit(bar);
  };
  auto issue_g1 = [&]() { issue_ts(w1d, bar1); };   // z2 = h1 W2^T
  auto issue_g3_g2 = [&](int it) {
    issue_ts(w3d, bar3);                              // -dh1 = (-dz2) W2
    // [-dz2_hi ; -dz2_lo]^T x [h1_hi ; h1_lo ; x~_hi ; x~_lo]: -dW2 (4 terms) and, through the ones row, -db2
#pragma unroll
    for (int ks = 0; ks < 16; ks++)
      mma_ss(tmem + COL_D2, pack64(fzd + ks * FK, f_hi), pack64(fhd + ks * FK, f_hi), idesc144, (it | ks) ? 1u : 0u);
    mma_commit(bar2);
  };
  auto issue_g4 = [&](int it) {   // [dz1_hi ; dz1_lo]^T x [x~_hi ; x~_lo]: dW1, db1
#pragma unroll
    for (int ks = 0; ks < 16; ks++)
      mma_ss(tmem + COL_D4, pack64(fhd + ks * FK, f_hi), pack64(xtd + ks * FK, f_hi), idesc16, (it | ks) ? 1u : 0u);
    mma_commit(bar4);
  };

  // L1 for one tile: h1 = tanh(W1 x + b1) for this thread's 16 feature pairs
  const int p0 = f0 / 2;
  auto layer1 = [&](const Sample<ENV>& in, float2 (&h)[TC_FG / 2], auto i0c, auto i1c) {
    constexpr int I0 = decltype(i0c)::value, I1 = decltype(i1c)::value;
    const float2 xb[4] = {f2s(in.x[0]), f2s(in.x[1]), f2s(in.x[2]), f2s(in.x[3])};
#pragma unroll
    for (int i = I0; i < I1; i++) {
      const float4 wa = w1v[(p0 + i) * 2], wc = w1v[(p0 + i) * 2 + 1];
      float2 acc = f2s(0.0f);
      acc = __ffma2_rn(f2(wa.x, wa.y), xb[0], acc);
      acc = __ffma2_rn(f2(wa.z, wa.w), xb[1], acc);
      acc = __ffma2_rn(f2(wc.x, wc.y), xb[2], acc);
      if (D == 4) acc = __ffma2_rn(f2(wc.z, wc.w), xb[3], acc);
      h[i] = tanh_upd2(__fadd2_rn(acc, b1q[p0 + i]));
    }
  };
  // hi/lo of 32 values: TMEM columns (A operand of G1/G3) and rows f0.. / 64+f0.. of a feature-major operand buffer
  auto split_to_tmem = [&](const float2 (&v)[TC_FG / 2], float (&vh)[TC_FG], float (&vl)[TC_FG]) {
#pragma unroll
    for (int i = 0; i < TC_FG / 2; i++) {
      float2 hi, lo;
      split2(v[i], hi, lo);
      vh[2 * i] = hi.x; vh[2 * i + 1] = hi.y; vl[2 * i] = lo.x; vl[2 * i + 1] = lo.y;
    }
    tmem_st_n<TC_FG>(lane_addr + COL_AH + f0, vh);
    tmem_st_n<TC_FG>(lane_addr + COL_AL + f0, vl);
  };
  auto split_to_smem = [&](const float (&vh)[TC_FG], const float (&vl)[TC_FG], float* buf) {
#pragma unroll
    for (int i = 0; i < TC_FG; i++) {
      buf[f_off(f0 + i, s)] = vh[i];
      buf[f_off(CRL_H + f0 + i, s)] = vl[i];
    }
  };

  // the next tile's first layer is spread over the shadows of G1, G3/G2 and G4 (pairs [0,A), [A,B), [B,end))
  constexpr int L1_A = TC_FG / 2 * 3 / 8, L1_B = TC_FG / 2 * 3 / 4;
  int it = 0;
  {
    Sample<ENV> cur, nxt;
    float2 h1[TC_FG / 2];
    int b_next = -1;  // buffer index of this thread's sample in the NEXT tile
    if (cta < n_tiles) {
      load_sample<ENV, NET>(a, load_index(a, keys, cta * TC_S + s), cur);
      if (cta + n_cta < n_tiles) b_next = load_index(a, keys, (cta + n_cta) * TC_S + s);
      layer1(cur, h1, IC<0>(), IC<TC_FG / 2>());
    }
#ifdef TC_TRACE
    long long tr[16];
    for (int i = 0; i < 16; i++) tr[i] = 0;
#endif
    for (int t = cta; t < n_tiles; t += n_cta, it++) {
#ifdef TC_TRACE
      const bool trace_on = (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1) && it == 3 && lane == 0 && (warp == 0 || warp == 5);
#endif
      TR(0);
      const uint32_t ph = it & 1;
      const int m0 = t * TC_S;
      const bool more = t + n_cta < n_tiles;
      // next tile's inputs (consumed in the shadow of G1 below) and the index for the tile after it
      if (more) {
        load_sample<ENV, NET>(a, b_next, nxt);
        if (t + 2 * n_cta < n_tiles) b_next = load_index(a, keys, (t + 2 * n_cta) * TC_S + s);
      }

      // ---- L1 hand-over, TMEM half: h1 hi/lo are the A operand of G1, which can start while the previous tile's
      //      G4 is still reading the shared-memory buffers
      float h1h[TC_FG], h1l[TC_FG];
      TR(1);
      split_to_tmem(h1, h1h, h1l);
      tmem_st_wait();
      tc_fence_before();
      TR(2);
      handover(BAR_G1, issue_g1);
      TR(3);
      {   // h1^2 - 1 is not an operand of G1: parked in its shadow (the previous tile's E3 has read its copy: program order)
        float dt[TC_FG];
#pragma unroll
        for (int i = 0; i < TC_FG / 2; i++) {
          const float2 d = __ffma2_rn(h1[i], h1[i], f2s(-1.0f));
          dt[2 * i] = d.x; dt[2 * i + 1] = d.y;
        }
        tmem_st_n<TC_FG>(lane_addr + COL_P + f0, dt);
      }
      // ---- in the shadow of G1: the shared-memory half (h1^T is the B operand of G2; x~^T), then part of the next
      //      tile's first layer (the rest follows G3 and G4)
      if (it > 0) mbar_wait(bar4, ph ^ 1);  // the previous tile's G4 has read dz1^T (same buffer as h1^T) and x~^T
      split_to_smem(h1h, h1l, fh);
      if (g == 0) {
#pragma unroll
        for (int d = 0; d < D; d++) {
          const float xh = tf32_hi(cur.x[d]);
          xt[xt_off(d, s)] = xh;
          xt[XT_GROUP + xt_off(d, s)] = cur.x[d] - xh;
        }
      }
      double adv_n = 0.0;  // (adv .- mean) ./ (std .+ 1e-8): Float32 numerator, Float64 quotient (Q6)
      if (NET == 0) adv_n = (double)__fsub_rn(cur.adv, mean_f) * inv_std;
      if (more) layer1(nxt, h1, IC<0>(), IC<L1_A>());
      TR(4);

      // ---- E1: h2, head, loss, dz2
      mbar_wait(bar1, ph);
      TR(5);
      tc_fence_after();
      float2 h2[TC_FG / 2];
      {
        float z2[TC_FG], z2b[TC_FG];
        tmem_ld_pair<TC_FG>(lane_addr + COL_D + f0, lane_addr + COL_D + CRL_H + f0, z2, z2b);
        float2 part[NOUT];
#pragma unroll
        for (int o = 0; o < NOUT; o++) part[o] = f2s(0.0f);
#pragma unroll
        for (int i = 0; i < TC_FG / 2; i++) {
          h2[i] = tanh_upd2(__fadd2_rn(__fadd2_rn(f2(z2[2 * i], z2[2 * i + 1]), f2(z2b[2 * i], z2b[2 * i + 1])), b2q[p0 + i]));
#pragma unroll
          for (int o = 0; o < NOUT; o++) part[o] = __ffma2_rn(w3q[o * (CRL_H / 2) + p0 + i], h2[i], part[o]);
        }
#pragma unroll
        for (int o = 0; o < NOUT; o++) exch[(g * 2 + o) * TC_S + s] = part[o].x + part[o].y;
      }
      TR(6);
      // only the TC_NG warps that share this lane quadrant exchange anything: one named barrier per quadrant instead of a
      // CTA-wide one, so that the quadrants do not wait for each other here (2.126 -> 2.115 ms per update)
      bar_sync(BAR_X + q, 32 * TC_NG);
      TR(7);
      float dl[NOUT];
#pragma unroll
      for (int o = 0; o < NOUT; o++) dl[o] = 0.0f;
      if (cur.valid) {
        float z[NOUT];
#pragma unroll
        for (int o = 0; o < NOUT; o++) {
          float acc = exch[(0 * 2 + o) * TC_S + s];
#pragma unroll
          for (int gg = 1; gg < TC_NG; gg++) acc += exch[(gg * 2 + o) * TC_S + s];
          z[o] = acc + b3s[o];
        }
        const bool own = g == 0;  // both feature halves evaluate the loss; only one of them accumulates its statistics
        if (NET == 0) {
          float newlp, p[A], lp[A];
          double ent_sum = 0.0;
          if (!E::CONT) {
            float m = z[0];
#pragma unroll
            for (int k = 1; k < A; k++) m = fmaxf(m, z[k]);
            float ex[A], sum = 0.0f;
#pragma unroll
            for (int k = 0; k < A; k++) { ex[k] = expf(__fsub_rn(z[k], m)); sum = __fadd_rn(sum, ex[k]); }
            const float ls = logf(sum);
            newlp = 0.0f;
#pragma unroll
            for (int k = 0; k < A; k++) {
              p[k] = __fdiv_rn(ex[k], sum);
              lp[k] = __fsub_rn(__fsub_rn(z[k], m), ls);
              ent_sum += (double)(-__fmul_rn(p[k], lp[k]));  // ppo.jl:42 (Q4: A x M matrix)
              if (k == cur.act) newlp = lp[k];
            }
          } else {
            float acc = 0.0f;
#pragma unroll
            for (int k = 0; k < A; k++) {
              const float logstd = b3s[2 + k];
              const float sd = expf(logstd);
              const float diff = __fsub_rn(cur.actf[k], z[k]);
              const float qq = __fdiv_rn(-__fmul_rn(diff, diff), __fmul_rn(__fmul_rn(2.0f, sd), sd));
              acc = __fadd_rn(acc, __fsub_rn(__fsub_rn(qq, logstd), 0.9189385332046727f));
              ent_sum += (double)__fadd_rn(__fadd_rn(0.5f, 0.9189385332046727f), logstd);
              p[k] = 0.0f; lp[k] = 0.0f;
            }
            newlp = acc;
          }
          double g_lp, ent_w = ent_scale;
          if (a2c) {
            // A2C (a2c.jl:88-97): actor_loss = -mean(logp .* advantage), advantage = R - critic(state) held constant.
            // The critic lives in other CTAs: its output for this sample is the value recorded by the rollout (same
            // parameters, A2C steps once per rollout; differs from a recomputation by fp32 summation order only).
            const double advd = (double)cur.R - (double)cur.V;
            if (own) st_pg += -(double)newlp * advd;
            g_lp = -advd * inv_Mg;
            ent_w = 0.0;
          } else {
          const float logratio = __fsub_rn(newlp, cur.oldlp);  // ppo.jl:224
          const float ratio = expf(logratio);                  // ppo.jl:225
          const float rc = ratio < lo_c ? lo_c : (ratio > hi_c ? hi_c : ratio);
          const double pg1 = -adv_n * (double)ratio;  // ppo.jl:226
          const double pg2 = -adv_n * (double)rc;     // ppo.jl:227
          double pgm, dratio;
          if (pg1 > pg2) { pgm = pg1; dratio = -adv_n; }
          else { pgm = pg2; dratio = (ratio >= lo_c && ratio <= hi_c) ? -adv_n : 0.0; }
          g_lp = dratio * (double)ratio * inv_Mg;
          if (own) { st_pg += pgm; st_ent += ent_sum; }
          }
          if (!E::CONT) {
#pragma unroll
            for (int k = 0; k < A; k++) {
              double dd = g_lp * ((k == cur.act ? 1.0 : 0.0) - (double)p[k]);
              dd += ent_w * (double)p[k] * ((double)lp[k] + ent_sum);
              dl[k] = (float)dd;
            }
          } else {
#pragma unroll
            for (int k = 0; k < A; k++) {
              const float sd = expf(b3s[2 + k]);
              const double diff = (double)__fsub_rn(cur.actf[k], z[k]);
              const double var = (double)sd * (double)sd;
              dl[k] = (float)(g_lp * diff / var);
              if (own) g_logstd[k] += g_lp * (diff * diff / var - 1.0) - ent_w;
            }
          }
        } else if (a2c) {
          // critic_loss = mean((R - v)^2) (a2c.jl:79-84)
          const double advd = (double)cur.R - (double)z[0];
          if (own) st_vmax += advd * advd;
          dl[0] = (float)(-2.0 * advd * inv_Mg);
        } else if (a.no_vclip) {
          // clip_value_loss = false: 0.5 * mean((newvalue - R).^2), ppo.jl:239-241 (no minibatch scalar, nothing to verify)
          const float d = __fsub_rn(z[0], cur.R);
          if (own) {
            st_vmax += (double)__fmul_rn(d, d);
            if (spec) a.vnew[m0 + s] = z[0];
          }
          dl[0] = (float)(v_scale * 2.0 * (double)d);
        } else {
          // value loss (Q5): 0.5*mean(max.(s, (clip - R)^2)), s a minibatch scalar
          const float v = z[0];
          float d_vcR, vlc;
          bool inside;
          value_clip(v, cur.V, cur.R, c, d_vcR, vlc, inside);
          const bool s_wins = !spec && s_f > vlc;
          if (own) {
            st_vmax += (double)(s_wins ? s_f : vlc);
            if (spec) {
              st_s += (double)__fsub_rn(v, __fmul_rn(cur.R, cur.R));  // newvalue .- mb_returns .^ 2, ppo.jl:232
              st_min = fminf(st_min, vlc);
              a.vnew[m0 + s] = v;
            }
          }
          double dv_d = cnt_over_M;
          if (!s_wins && inside) dv_d += 2.0 * (double)d_vcR;
          dl[0] = (float)(v_scale * dv_d);
        }
      }
      TR(8);
      // -dz2 = (W3^T dl) .* (h2^2 - 1): the sign is carried through G3/G2 and removed again by E3 / at the read-out,
      // which saves negating a packed operand here. dW3(o,f) += dl[o] h2[f] stays in registers.
      {
        float2 ndz2[TC_FG / 2];
#pragma unroll
        for (int i = 0; i < TC_FG / 2; i++) {
          float2 dh = __fmul2_rn(w3q[p0 + i], f2s(dl[0]));
#pragma unroll
          for (int o = 1; o < NOUT; o++) dh = __ffma2_rn(w3q[o * (CRL_H / 2) + p0 + i], f2s(dl[o]), dh);
          ndz2[i] = __fmul2_rn(dh, __ffma2_rn(h2[i], h2[i], f2s(-1.0f)));
#pragma unroll
          for (int o = 0; o < NOUT; o++) gw3[o][i] = __ffma2_rn(f2s(dl[o]), h2[i], gw3[o][i]);
        }
#pragma unroll
        for (int o = 0; o < NOUT; o++) if (g == 0) gb3[o] += dl[o];
        float zh[TC_FG], zl[TC_FG];
        split_to_tmem(ndz2, zh, zl);
        split_to_smem(zh, zl, fz);   // the previous tile's G2 was waited for in its E3
      }
      tmem_st_wait();
      proxy_fence();
      tc_fence_before();
      TR(9);
      handover(BAR_G3, [&]() { issue_g3_g2(it); });
      if (more) layer1(nxt, h1, IC<L1_A>(), IC<L1_B>());
      TR(10);

      // ---- E3: dz1 = (-dh1) .* (h1^2 - 1), in place over h1^T; h1^2 - 1 comes from the parked TMEM columns
      mbar_wait(bar3, ph);
      TR(11);
      tc_fence_after();
      float ndh1[TC_FG], ndh1b[TC_FG], dt[TC_FG];
      float2 dz1[TC_FG / 2];
      tmem_ld_triple<TC_FG>(lane_addr + COL_D + f0, lane_addr + COL_D + CRL_H + f0, lane_addr + COL_P + f0, ndh1, ndh1b, dt);
#pragma unroll
      for (int i = 0; i < TC_FG / 2; i++)
        dz1[i] = __fmul2_rn(__fadd2_rn(f2(ndh1[2 * i], ndh1[2 * i + 1]), f2(ndh1b[2 * i], ndh1b[2 * i + 1])), f2(dt[2 * i], dt[2 * i + 1]));
      TR(12);
      mbar_wait(bar2, ph);  // G2 has consumed h1^T and dz2^T
      TR(13);
#pragma unroll
      for (int i = 0; i < TC_FG / 2; i++) {
        float2 hi, lo;
        split2(dz1[i], hi, lo);
        fh[f_off(f0 + 2 * i, s)] = hi.x;
        fh[f_off(f0 + 2 * i + 1, s)] = hi.y;
        fh[f_off(CRL_H + f0 + 2 * i, s)] = lo.x;
        fh[f_off(CRL_H + f0 + 2 * i + 1, s)] = lo.y;
      }
      proxy_fence();
      tc_fence_before();
      TR(14);
      handover(BAR_G4, [&]() { issue_g4(it); });
      if (more) layer1(nxt, h1, IC<L1_B>(), IC<TC_FG / 2>());
      TR(15);
#ifdef TC_TRACE
      if (trace_on)
        printf("net %d warp %d: wait4 %lld | st_h1 %lld | hand1 %lld | L1next %lld | waitG1 %lld | E1a %lld | barX %lld | loss %lld | dz2+st %lld | "
               "hand3 %lld | waitG3 %lld | E3a %lld | waitG2 %lld | st_dz1 %lld | hand4 %lld | total %lld\n", NET, warp, tr[1] - tr[0],
               tr[2] - tr[1], tr[3] - tr[2], tr[4] - tr[3], tr[5] - tr[4], tr[6] - tr[5], tr[7] - tr[6], tr[8] - tr[7], tr[9] - tr[8],
               tr[10] - tr[9], tr[11] - tr[10], tr[12] - tr[11], tr[13] - tr[12], tr[14] - tr[13], tr[15] - tr[14], tr[15] - tr[0]);
#endif
      cur = nxt;
    }
  }

  // ---------------------------------------------------------------- epilogue: this CTA's partial gradient
#ifdef TC_TRACE
  const long long e_t0 = clock64();
#endif
  float* gp = a.gpart + (long long)blockIdx.x * E::P;
  const int nb = NET == 0 ? 0 : E::NET_A;
  using NN = NetOff<D, NOUT>;
  const bool has_tiles = cta < n_tiles;
  float* scr = fz;  // the operand buffers are free once the last G4 has completed
  if (has_tiles) {
    mbar_wait(bar4, (it - 1) & 1);  // the last commit covers every MMA issued before it
    tc_fence_after();
    // dW2(j,k) = -(D2[j][k] + D2[64+j][k]); dW1(k,d), db1(k) = D4[k][d] + D4[64+k][d]; db2(j) = -(D5[j][D] + D5[64+j][D]):
    // lanes 64.. hand their (lo) halves over through shared memory
    float d2[TC_FG], d4[16], d5[16];
    {
      float d2b[TC_FG];
      tmem_ld_pair<TC_FG>(lane_addr + COL_D2 + f0, lane_addr + COL_D2 + CRL_H + f0, d2, d2b);
#pragma unroll
      for (int i = 0; i < TC_FG; i++) d2[i] += d2b[i];
    }
    if (g == 0) { tmem_ld16(lane_addr + COL_D4, d4); tmem_ld16(lane_addr + COL_D2 + 2 * CRL_H, d5); }
    if (q >= 2) {
#pragma unroll
      for (int i = 0; i < TC_FG; i++) scr[(f0 + i) * CRL_H + (s - 64)] = d2[i];
      if (g == 0) {
#pragma unroll
        for (int d = 0; d <= D; d++) scr[CRL_H * CRL_H + d * CRL_H + (s - 64)] = d4[d] + d4[8 + d];
        scr[CRL_H * CRL_H + 7 * CRL_H + (s - 64)] = d5[D];
      }
    }
    __syncthreads();
    if (q < 2) {
#pragma unroll
      for (int i = 0; i < TC_FG; i++) gp[nb + NO::W2 + s + CRL_H * (f0 + i)] = -(d2[i] + scr[(f0 + i) * CRL_H + s]);
      if (g == 0) {
#pragma unroll
        for (int d = 0; d <= D; d++) {
          const float v = (d4[d] + d4[8 + d]) + scr[CRL_H * CRL_H + d * CRL_H + s];
          if (d < D) gp[nb + NO::W1 + s + CRL_H * d] = v;
          else gp[nb + NO::B1 + s] = v;
        }
        gp[nb + NO::B2 + s] = -(d5[D] + scr[CRL_H * CRL_H + 7 * CRL_H + s]);
      }
    }
  } else {
    for (int i = tid; i < CRL_H * CRL_H; i += TC_THREADS) gp[nb + NO::W2 + i] = 0.0f;
    for (int i = tid; i < CRL_H * (D + 1); i += TC_THREADS) gp[nb + NO::W1 + i] = 0.0f;  // W1 and b1 are adjacent
    for (int i = tid; i < CRL_H; i += TC_THREADS) gp[nb + NO::B2 + i] = 0.0f;
  }
  __syncthreads();
  // head partials: reduce-scatter over the 32 lanes (samples) of each warp, then sum the four lane quadrants
  {
    float* hs = scr + CRL_H * CRL_H + 8 * CRL_H;  // [NOUT][warps][32] (TC_FG = 32) or [warps][32] (TC_FG = 16)
    if (TC_FG == 32) {
#pragma unroll
      for (int o = 0; o < NOUT; o++) {
        float v[32];
#pragma unroll
        for (int i = 0; i < TC_FG / 2; i++) { v[(2 * i) & 31] = gw3[o][i].x; v[(2 * i + 1) & 31] = gw3[o][i].y; }
        warp_reduce_scatter<32>(v, lane);
        hs[(o * TC_WARPS + warp) * 32 + lane] = v[0];  // feature f0 + lane
      }
    } else {
      // 16 features per thread: both outputs share one 32-element reduce-scatter, element o * 16 + i
      float v[32];
#pragma unroll
      for (int e = 0; e < 32; e++) v[e] = 0.0f;
#pragma unroll
      for (int o = 0; o < NOUT; o++)
#pragma unroll
        for (int i = 0; i < TC_FG / 2; i++) {
          v[(o * 16 + 2 * i) & 31] = gw3[o][i].x;
          v[(o * 16 + 2 * i + 1) & 31] = gw3[o][i].y;
        }
      warp_reduce_scatter<32>(v, lane);
      hs[warp * 32 + lane] = v[0];  // output lane / 16, feature f0 + lane % 16
    }
    __syncthreads();
    if (tid < CRL_H) {
      const int gg = tid / TC_FG, ll = tid % TC_FG;  // feature tid lives in warps gg*4 .. gg*4+3
#pragma unroll
      for (int o = 0; o < NOUT; o++) {
        float sum = 0.0f;
#pragma unroll
        for (int qq = 0; qq < 4; qq++)
          sum += TC_FG == 32 ? hs[(o * TC_WARPS + gg * 4 + qq) * 32 + ll] : hs[(gg * 4 + qq) * 32 + o * 16 + ll];
        gp[nb + NN::W3 + o + NOUT * tid] = sum;  // Flux W3 is (out=o, in=f) at o + NOUT f
      }
    }
  }
  double t_b3[NOUT];
#pragma unroll
  for (int o = 0; o < NOUT; o++) t_b3[o] = block_sum<TC_WARPS>((double)gb3[o], red);
  const double t_pg = block_sum<TC_WARPS>(st_pg, red);
  const double t_vm = block_sum<TC_WARPS>(st_vmax, red);
  const double t_en = block_sum<TC_WARPS>(st_ent, red);
  const double t_ss = block_sum<TC_WARPS>(st_s, red);
  double t_ls[A];
#pragma unroll
  for (int k = 0; k < A; k++) t_ls[k] = block_sum<TC_WARPS>(g_logstd[k], red);
  float* mred = reinterpret_cast<float*>(red + 16);
  st_min = warp_min(st_min);
  __syncthreads();
  if (lane == 0) mred[warp] = st_min;
  __syncthreads();
  if (tid == 0) {
    float mn = mred[0];
#pragma unroll
    for (int w = 1; w < TC_WARPS; w++) mn = fminf(mn, mred[w]);
#pragma unroll
    for (int o = 0; o < NOUT; o++) gp[nb + NN::B3 + o] = (float)t_b3[o];
    double* spp = a.spart + (long long)blockIdx.x * 4;
    spp[0] = t_pg; spp[1] = t_vm; spp[2] = t_en; spp[3] = t_ss;
    if (spec) a.mpart[blockIdx.x] = mn;
    if (E::CONT && NET == 0) {
#pragma unroll
      for (int k = 0; k < A; k++) gp[E::NET_A + E::NET_C + k] = (float)t_ls[k];
    }
#ifdef TC_TRACE
    if (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1) printf("  net %d epilogue %lld tiles %d\n", NET, clock64() - e_t0, it);
#endif
  }
}


// ---------------------------------------------------------------- fused tail: reduce -> exchange -> clip + Adam
// Runs at the end of loss_grad_tc_kernel when UpdateArgs::fuse_tail is set (cooperative launch: all CTAs co-resident).
//   barrier 1   every CTA's partial gradient (gpart / spart / mpart) is in L2
//   reduce      CTA j owns the slab [j*slab, (j+1)*slab) of the P gradient elements + 4 loss sums and adds the partials
//               of all CTAs that hold them in the fixed order of grad_reduce_kernel (deterministic, same bits)
//   exchange    [multi-GPU] the slab is PUSHED into every peer's exchange buffer as 16-byte {lo, seq, hi, seq} packets
//               (the flag travels inside the data word, so no fence, no counter and no separate flag store is needed);
//               the same CTA on every rank then polls ITS OWN memory for the slab of every peer and adds the world
//               vectors in rank order: all ranks hold bit-identical sums. This rank's min (clip-R)^2 rides behind the
//               loss sums for the verification of the speculation.
//   barrier 2   the Float32 gradient of every array is complete in `grads_out`
//   clip+Adam   every CTA recomputes the norm of the arrays its slab touches (Float64 sum of squares in a fixed order:
//               identical in every CTA and on every rank), then Flux.Optimiser(ClipNorm, Adam) on its slab exactly as
//               clip_adam_kernel does it, parameter image included.
__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void grid_barrier(unsigned long long* ctr) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();  // cumulative: the CTA's writes (ordered before this point by the barrier above) become visible first
    const unsigned long long old = atomicAdd(ctr, 1ull);
    const unsigned long long target = (old / gridDim.x + 1ull) * gridDim.x;
    while (ld_acquire_u64(ctr) < target) { }
  }
  __syncthreads();
}
constexpr int FT_EL = 64;  // elements per reduction pass (x 4 partial groups = 256 threads)
constexpr int FT_BATCH = 10;  // partials per thread in flight in the slab reduction
// -DFT_TRACE: clock stamps of the tail's phases, printed by thread 0 of the first and the last CTA (development aid)
#ifdef FT_TRACE
__device__ __forceinline__ long long gtime() { long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define FTR(i) do { if (ft_on) ftr[i] = gtime(); } while (0)
#else
#define FTR(i) do { } while (0)
#endif

template <int ENV>
__device__ __noinline__ void fused_tail(const UpdateArgs& a, float* scratch, const unsigned long long seq) {
  using E = EnvTraits<ENV>;
  static_assert(TC_THREADS >= 4 * FT_EL, "the fused tail splits the partials over 4 thread groups of 64 elements");
  constexpr int P = E::P;
  const AdamArgs& f = a.adam;
  const int tid = threadIdx.x, G = (int)gridDim.x;
  const int lane_id = tid & 31, warp_id = tid >> 5;
  // CTA j owns the gradient elements [j*slab, (j+1)*slab); the LAST CTA (whose slab is empty at the benchmark sizes)
  // also owns the four loss sums and the min (clip-R)^2 of the verification, kept behind its gradient elements
  const int slab = (((P + G - 1) / G) + FT_EL - 1) & ~(FT_EL - 1);
  const int lo = (int)blockIdx.x * slab;
  const int ngrad = min(P, lo + slab) > lo ? min(P, lo + slab) - lo : 0;
  const bool tail_owner = (int)blockIdx.x == G - 1;
  const bool multi = f.ll_local != nullptr;
  const int W = multi ? f.world : 1;
  // scratch (the operand buffers are free): reduced sums (+ 4 loss sums + min) | 4 x 64 pass buffer | small per-array
  // state | Float32 gradient
  double* gs = reinterpret_cast<double*>(scratch);
  double* sh = gs + slab + 8;                          // [4][64]
  double* red = sh + 4 * FT_EL;                        // 16 doubles (block min)
  double* bp_s = red + 16;                             // [CRL_MAX_ARRAYS][2] beta powers BEFORE this step
  double* scale_s = bp_s + 2 * CRL_MAX_ARRAYS;         // [CRL_MAX_ARRAYS] clip factor, 1.0 = no clip
  float* gfl = reinterpret_cast<float*>(scale_s + CRL_MAX_ARRAYS);   // [slab]
  int* clip_s = reinterpret_cast<int*>(gfl + slab);    // [CRL_MAX_ARRAYS]
  __shared__ float all_min_s;
  Layout L;
  make_layout(ENV, &L);
#ifdef FT_TRACE
  const bool ft_on = tid == 0;
  long long ftr[8];
#endif
  FTR(0);
  if (tid < 2 * L.n_arrays) bp_s[tid] = f.beta_pow[tid];   // read before anybody can rewrite them (after barrier 2)
  const double lr = f.lr_host >= 0.0 ? f.lr_host : f.ds->lr;

  grid_barrier(f.grid_bar);
  FTR(1);
  if (a.p2p_seq && blockIdx.x == 0 && tid == 0) *a.p2p_seq = seq;   // every CTA has read the old value at kernel start

  // ---- reduce this slab over the per-CTA partials (order of grad_reduce_kernel)
  const int el = tid & (FT_EL - 1), g = tid >> 6;
  for (int base = 0; base < ngrad; base += FT_EL) {
    const int e = lo + base + el;
    double s = 0.0;
    if (g < 4 && base + el < ngrad) {
      int c_lo = 0, c_hi = G;
      const bool critic = e >= a.tc_net_a && e < a.tc_net_a + a.tc_net_c;
      if (critic) c_lo = a.tc_actor_ctas; else c_hi = a.tc_actor_ctas;
      // FT_BATCH partials requested before the first is added (one L2 round trip per batch); same summation order as the
      // plain loop: adding the +0.0f of a padded slot changes nothing
      for (int c0 = c_lo + g; c0 < c_hi; c0 += 4 * FT_BATCH) {
        float v[FT_BATCH];
#pragma unroll
        for (int j = 0; j < FT_BATCH; j++) {   // unconditional (clamped) loads: a predicated load would be a branch, i.e. serialised
          const int c = c0 + 4 * j;
          const float x = __ldcg(a.gpart + (long long)min(c, c_hi - 1) * P + e);
          v[j] = c < c_hi ? x : 0.0f;
        }
#pragma unroll
        for (int j = 0; j < FT_BATCH; j++) s += (double)v[j];
      }
    }
    if (g < 4) sh[g * FT_EL + el] = s;
    __syncthreads();
    if (g == 0 && base + el < ngrad) gs[base + el] = (sh[el] + sh[FT_EL + el]) + (sh[2 * FT_EL + el] + sh[3 * FT_EL + el]);
    __syncthreads();
  }
  int next = ngrad;   // entries of this CTA that take part in the exchange
  if (tail_owner) {
    // the four loss sums (same order as grad_reduce_kernel) and this rank's min_i (clip_i - R_i)^2 over all CTAs
    const int q = tid & 3, gg = (tid >> 2) & 3;      // threads 0..15: (sum q, group gg); the partials of a group in batches
    double s = 0.0;
    if (tid < 16) {
      for (int c0 = gg; c0 < G; c0 += 40) {
        double v[10];
#pragma unroll
        for (int j = 0; j < 10; j++) {
          const int c = c0 + 4 * j;
          const double x = __ldcg(a.spart + (long long)min(c, G - 1) * 4 + q);
          v[j] = c < G ? x : 0.0;
        }
#pragma unroll
        for (int j = 0; j < 10; j++) s += v[j];
      }
      sh[gg * 4 + q] = s;
    }
    float mn = INFINITY;
    if (f.verify) {
      for (int c = tid; c < G; c += TC_THREADS) mn = fminf(mn, __ldcg(a.mpart + c));
      mn = warp_min(mn);
      float* mred = reinterpret_cast<float*>(red);
      if (lane_id == 0) mred[warp_id] = mn;
    }
    __syncthreads();
    if (tid < 4) gs[ngrad + tid] = (sh[tid] + sh[4 + tid]) + (sh[8 + tid] + sh[12 + tid]);
    if (tid == 0) {
      const float* mred = reinterpret_cast<const float*>(red);
      float m8 = INFINITY;
      if (f.verify)
        for (int w = 0; w < TC_WARPS; w++) m8 = fminf(m8, mred[w]);
      all_min_s = m8;
      gs[ngrad + 4] = (double)m8;
    }
    next = ngrad + 5;
    __syncthreads();
  }
  FTR(2);

  // ---- exchange with the peers (NVLink peer memory, flag-in-data packets). Position in a rank's row: gradient element
  //      e at e, the loss sums at P..P+3, the min at P+4.
  if (multi) {
    const uint32_t flag = (uint32_t)seq;
    const int slot = (int)(seq & 1ull);
    auto pos = [&](int k) { return k < ngrad ? lo + k : P + (k - ngrad); };
    for (int i = tid; i < next * W; i += TC_THREADS) {
      const int r = i / next, k = i - r * next;
      if (r == f.rank) continue;
      uint4* dst = reinterpret_cast<uint4*>(f.ll_peers[r] + f.ll_off) + ((size_t)slot * W + f.rank) * f.ll_stride + pos(k);
      ll_store(dst, gs[k], flag);
    }
    __syncthreads();
    bool bad = false;
    for (int k = tid; k < next; k += TC_THREADS) {
      const uint4* src = reinterpret_cast<const uint4*>(f.ll_local + f.ll_off) + (size_t)slot * W * f.ll_stride + pos(k);
      uint4 pk[CRL_MAX_WORLD];
      const long long t0 = clock64();
      bool all = false;
      while (!all) {    // all peers' packets are requested before any is inspected: one round trip when they have arrived
        all = true;
#pragma unroll
        for (int r = 0; r < CRL_MAX_WORLD; r++)
          if (r < W && r != f.rank) pk[r] = ll_load(src + (size_t)r * f.ll_stride);
#pragma unroll
        for (int r = 0; r < CRL_MAX_WORLD; r++)
          if (r < W && r != f.rank && (pk[r].y != flag || pk[r].w != flag)) all = false;
        if (!all && clock64() - t0 > f.timeout_cycles) { bad = true; break; }
      }
      double tot = 0.0;
      float mn = INFINITY;
#pragma unroll
      for (int r = 0; r < CRL_MAX_WORLD; r++) {
        if (r >= W) continue;
        const double v = r == f.rank ? gs[k] : __longlong_as_double((long long)(((unsigned long long)pk[r].z << 32) | pk[r].x));
        tot += v;                       // rank order: bit-identical on every rank
        mn = fminf(mn, (float)v);
      }
      if (tail_owner && k == ngrad + 4) all_min_s = mn; else gs[k] = tot;
    }
    if (bad) atomicExch(f.p2p_err, 1);
    __syncthreads();
  }

  // ---- Float32 gradient (what Zygote returns), loss scalars, verification of the speculation
  for (int k = tid; k < ngrad; k += TC_THREADS) {
    const float gv = (float)gs[k];
    gfl[k] = gv;
    if (f.grads_out) f.grads_out[lo + k] = gv;
  }
  if (tail_owner && tid == 0) {
    const double* tl = gs + ngrad;
    if (f.stats_out) finalize_stats(tl, f.M_global, f.A, f.ent_coeff, f.v_coef, f.stats_out, f.algo);
    if (f.verify) {
      const float m = all_min_s;
      const float s_f = (float)(tl[3] / f.M_global);
      f.fin->s_unclipped = s_f; f.fin->min_vlc = m; f.fin->M_global = f.M_global; f.fin->cnt = 0ull;
      f.fin->need_fixup = (s_f > m) ? 1 : 0;
      if (s_f > m) f.ds_rw->spec_failed = 1;   // the host replays this update exactly
    }
  }
  // partial sums of squares of this slab per parameter array it touches -> normpart[array][cta] (ClipNorm is per array)
  __syncthreads();
  for (int ai = warp_id; ai < L.n_arrays; ai += TC_WARPS) {
    const int o = L.off[ai], n = L.size[ai];
    if (ngrad == 0 || !(o < lo + ngrad && o + n > lo)) continue;
    const int k0 = max(o, lo) - lo, k1 = min(o + n, lo + ngrad) - lo;
    double ss = 0.0;
    for (int k = k0 + lane_id; k < k1; k += 32) ss += (double)gfl[k] * (double)gfl[k];
    ss = warp_sum(ss);
    if (lane_id == 0) f.normpart[ai * G + (int)blockIdx.x] = ss;
  }
  // this thread's Adam operands are requested before the barrier (their values cannot change behind it)
  const bool pre = ngrad <= TC_THREADS;
  float pre_m = 0.0f, pre_v = 0.0f, pre_p = 0.0f;
  if (pre && tid < ngrad) { pre_m = f.m[lo + tid]; pre_v = f.v[lo + tid]; pre_p = f.params[lo + tid]; }
  FTR(3);
  grid_barrier(f.grid_bar);
  FTR(4);
  // a peer that never delivered: nobody applies this (or any later) minibatch; the host reports CRL_ERR_NCCL
  if (multi && (*reinterpret_cast<volatile int*>(f.p2p_err) != 0)) return;

  // ---- per-array norms of the arrays this slab touches (ClipNorm is per array, ppo.jl:93): one warp per array adds the
  //      partials of the CTAs that cover it, in an order that depends on nothing but the grid size
  for (int ai = warp_id; ai < L.n_arrays; ai += TC_WARPS) {
    const int o = L.off[ai], n = L.size[ai];
    if (ngrad == 0 || !(o < lo + ngrad && o + n > lo)) continue;
    const int c_first = o / slab, c_last = (o + n - 1) / slab;
    double ss = 0.0;
    for (int c = c_first + lane_id; c <= c_last; c += 32) ss += __ldcg(f.normpart + ai * G + c);
    ss = warp_sum(ss);
    if (lane_id == 0) {
      const float nrm = (float)sqrt(ss);   // norm(Δ::Array{Float32})::Float32
      const bool clip = (double)nrm > (double)f.clip_norm;
      clip_s[ai] = clip ? 1 : 0;
      scale_s[ai] = clip ? (double)f.clip_norm / (double)nrm : 1.0;
    }
  }
  __syncthreads();

  FTR(5);
  // ---- Adam on the slab (same arithmetic as clip_adam_kernel: Float64 scalars, _rn intrinsics)
  const double b1 = 0.9, b2 = 0.999, eps = 1e-8;
  for (int k = tid; k < ngrad; k += TC_THREADS) {
    const int e = lo + k;
    int ai = 0;
    while (ai + 1 < L.n_arrays && e >= L.off[ai + 1]) ai++;
    const double bp1 = bp_s[2 * ai], bp2 = bp_s[2 * ai + 1];
    float d = gfl[k];
    if (clip_s[ai]) d = (float)__dmul_rn((double)d, scale_s[ai]);  // rmul!(Δ, thresh/nrm)
    const float m_old = pre ? pre_m : f.m[e], v_old = pre ? pre_v : f.v[e], p_old = pre ? pre_p : f.params[e];
    const float mt = (float)__dadd_rn(__dmul_rn(b1, (double)m_old), __dmul_rn(1.0 - b1, (double)d));
    const float vt = (float)__dadd_rn(__dmul_rn(b2, (double)v_old), __dmul_rn(__dmul_rn(1.0 - b2, (double)d), (double)d));
    f.m[e] = mt;
    f.v[e] = vt;
    const double den = __dadd_rn(sqrt(__ddiv_rn((double)vt, 1.0 - bp2)), eps);
    const float step = (float)__dmul_rn(__ddiv_rn(__ddiv_rn((double)mt, 1.0 - bp1), den), lr);
    const float pnew = __fsub_rn(p_old, step);
    f.params[e] = pnew;
    if (f.image) image_scatter<ENV>(f.image, e, pnew);
    if (e == L.off[ai]) {   // the CTA that owns an array's first element advances its beta powers
      f.beta_pow[2 * ai] = bp1 * b1;
      f.beta_pow[2 * ai + 1] = bp2 * b2;
    }
  }
#ifdef FT_TRACE
  FTR(6);
  if (ft_on)
    printf("FT %d %lld %lld %lld %lld %lld %lld %lld\n", (int)blockIdx.x, ftr[0], ftr[1], ftr[2], ftr[3], ftr[4], ftr[5], ftr[6]);
#endif
}

template <int ENV>
__global__ void __launch_bounds__(TC_THREADS, 1) loss_grad_tc_kernel(const __grid_constant__ UpdateArgs a) {
  using E = EnvTraits<ENV>;
  using SM = TcSmem<ENV>;
  using NO = NetOff<E::D, 1>;
  using NA = NetOff<E::D, E::A>;
  extern __shared__ __align__(128) float smem[];
  __shared__ TcBars bars;
  __shared__ uint32_t tmem_base_s;
  const int tid = threadIdx.x, warp = tid >> 5;
#ifdef TC_TRACE
  const long long k_t0 = clock64();
#endif
  // exchange sequence number of this minibatch. Unfused chain: CTA 0 advances it here for grad_reduce / clip_adam. Fused
  // tail: every CTA needs it, so all read the old value now and CTA 0 stores the new one behind the first grid barrier.
  const unsigned long long seq_next = a.p2p_seq ? *a.p2p_seq + 1ull : 0ull;
  if (!a.fuse_tail && a.p2p_seq && blockIdx.x == 0 && tid == 0) *a.p2p_seq = seq_next;
  const int net = (int)blockIdx.x < a.tc_actor_ctas ? 0 : 1;
  uint32_t* keys = reinterpret_cast<uint32_t*>(smem + SM::KEYS);
  if (tid == 0 && !a.idx.arr) perm_keys(a.idx.seed, a.idx.ds->update_index, a.idx.epoch, a.idx.rank, keys);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)), "r"(TMEM_COLS));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  if (tid == 32) {
    const uint32_t b[5] = {smem_u32(&bars.pbar), smem_u32(&bars.g1), smem_u32(&bars.g2), smem_u32(&bars.g3), smem_u32(&bars.g4)};
#pragma unroll
    for (int i = 0; i < 5; i++) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(b[i]));
    asm volatile("fence.mbarrier_init.release.cluster;");
  }
  // small parameters of this net, x~^T constant rows
  {
    const float* np = a.params + (net == 0 ? 0 : E::NET_A);
    const int nout = net == 0 ? E::A : 1;
    float* w1p = smem + SM::W1P;
    for (int i = tid; i < 4 * CRL_H; i += TC_THREADS) {
      const int f = 2 * (i >> 3) + (i & 1), d = (i >> 1) & 3;
      w1p[i] = d < E::D ? np[NO::W1 + f + CRL_H * d] : 0.0f;
    }
    for (int i = tid; i < CRL_H; i += TC_THREADS) { smem[SM::B1 + i] = np[NO::B1 + i]; smem[SM::B2 + i] = np[NO::B2 + i]; }
    for (int i = tid; i < 2 * CRL_H; i += TC_THREADS) {
      const int o = i / CRL_H, f = i % CRL_H;
      smem[SM::W3P + i] = o < nout ? np[NO::W3 + o + nout * f] : 0.0f;   // W3 offset is the same for both head widths
    }
    if (tid < 2) smem[SM::B3 + tid] = tid < nout ? np[(net == 0 ? NA::B3 : NO::B3) + tid] : 0.0f;
    if (tid >= 2 && tid < 4) smem[SM::B3 + tid] = (E::CONT && tid - 2 < E::A) ? a.params[E::NET_A + E::NET_C + (tid - 2)] : 0.0f;
    float* xt = smem + SM::XT;
    for (int i = tid; i < 2 * XT_GROUP; i += TC_THREADS) {
      const int half = i / XT_GROUP, r = (i % XT_GROUP) % (F_LBO / 4);  // xt_off: d*4 + chunk*36 + (s&3); floats 32..35 are padding
      const int d = r >> 2;
      xt[i] = (half == 0 && d == E::D) ? 1.0f : 0.0f;
    }
  }
  proxy_fence();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_base_s;
  // this net's four weight images: one elected thread, bulk asynchronous copies completed on an mbarrier
  const uint32_t pbar = smem_u32(&bars.pbar);
  // (a CTA without tiles -- full grid for the fused tail, small minibatch -- only zero-fills its partials: no images)
  const bool cta_has_tiles = (net == 0 ? (int)blockIdx.x : (int)blockIdx.x - a.tc_actor_ctas) < (a.M + TC_S - 1) / TC_S;
  if (tid == 0 && cta_has_tiles) {
    constexpr uint32_t BYTES = 4 * TC_W_FLOATS * 4, CHUNK = 16384;
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(pbar), "r"(BYTES) : "memory");
    const char* src = reinterpret_cast<const char*>(a.image + TcImage<ENV>::BASE + net * TcImage<ENV>::NET_FLOATS);
    const uint32_t dst = smem_u32(smem + SM::WB);
    for (uint32_t off = 0; off < BYTES; off += CHUNK)
      asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                   ::"r"(dst + off), "l"(src + off), "r"(CHUNK), "r"(pbar) : "memory");
  }
  if (cta_has_tiles) mbar_wait(pbar, 0);
#ifdef TC_TRACE
  const long long k_t1 = clock64();
#endif
  if (net == 0) tc_body<ENV, 0>(a, smem, &bars, tmem);
  else tc_body<ENV, 1>(a, smem, &bars, tmem);
#ifdef TC_TRACE
  if (tid == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1))
    printf("kernel net %d: prologue %lld  body+epilogue %lld\n", net, k_t1 - k_t0, clock64() - k_t1);
#endif
  tc_fence_before();
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS));
  if (a.fuse_tail) fused_tail<ENV>(a, smem + SM::FZ, seq_next);
}

}  // namespace

cudaError_t kernels_init_update_tc() {
  cudaError_t e = cudaFuncSetAttribute(loss_grad_tc_kernel<CRL_ENV_CARTPOLE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)TcSmem<CRL_ENV_CARTPOLE>::BYTES);
  if (e != cudaSuccess) return e;
  return cudaFuncSetAttribute(loss_grad_tc_kernel<CRL_ENV_PENDULUM>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              (int)TcSmem<CRL_ENV_PENDULUM>::BYTES);
}

// Chooses the tensor-core kernel for this minibatch when it applies (parameter image present) and fills
// in the launch geometry; CRL_NO_TC=1 keeps the FFMA kernel.
int loss_grad_tc_plan(UpdateArgs* a, int sm_count, bool full_grid) {
  static int disabled = -1;
  if (disabled < 0) {
    const char* e = getenv("CRL_NO_TC");
    disabled = (e && atoi(e) != 0) ? 1 : 0;
  }
  a->tc_actor_ctas = 0;
  // A2C: the actor's advantage needs the critic's output, which lives in other CTAs; only when the recorded values
  // are that output (values_fresh) can the one-net-per-CTA kernel be used
  if (disabled || !a->image || (a->algo == 1 && !a->values_fresh)) return 0;
  const int n_tiles = (a->M + TC_S - 1) / TC_S;
  int grid = (2 * n_tiles < sm_count && !full_grid) ? 2 * n_tiles : sm_count;
  grid &= ~1;
  if (grid < 2) grid = 2;
  // An actor tile (two heads, softmax, entropy) costs 1.15 x a critic tile: the clock stamps of the -DTC_TRACE build
  // are perturbed by the stamps and show them equal, while the timed splits of DESIGN.md §9 are fastest at 79 of 148
  // CTAs on the actor, which this cost picks for the benchmark's 1024 tiles. Every CTA runs a whole number of tiles:
  // pick the split that minimises the slower side.
  constexpr double actor_cost = 1.15;
  int na = grid / 2;
  {
    double best = 1e30;
    for (int cand = 1; cand < grid; cand++) {
      const double ta = actor_cost * ((n_tiles + cand - 1) / cand), tc = (double)((n_tiles + (grid - cand) - 1) / (grid - cand));
      const double cost = ta > tc ? ta : tc;
      if (cost < best - 1e-9) { best = cost; na = cand; }
    }
  }
  a->grid_loss = grid;
  a->tc_actor_ctas = na;
  return 1;
}

template <int ENV> static cudaError_t launch_fused_t(const UpdateArgs& a, cudaStream_t s) {
  // the grid barriers of the fused tail need every CTA resident: cooperative launch (grid <= SM count, 1 CTA per SM)
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)a.grid_loss);
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = TcSmem<ENV>::BYTES;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeCooperative;
  at[0].val.cooperative = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, loss_grad_tc_kernel<ENV>, a);
}

cudaError_t launch_loss_grad_tc(const UpdateArgs& a, cudaStream_t s) {
  if (a.fuse_tail)
    return a.env_kind == CRL_ENV_CARTPOLE ? launch_fused_t<CRL_ENV_CARTPOLE>(a, s) : launch_fused_t<CRL_ENV_PENDULUM>(a, s);
  if (a.env_kind == CRL_ENV_CARTPOLE)
    loss_grad_tc_kernel<CRL_ENV_CARTPOLE><<<a.grid_loss, TC_THREADS, TcSmem<CRL_ENV_CARTPOLE>::BYTES, s>>>(a);
  else
    loss_grad_tc_kernel<CRL_ENV_PENDULUM><<<a.grid_loss, TC_THREADS, TcSmem<CRL_ENV_PENDULUM>::BYTES, s>>>(a);
  return cudaGetLastError();
}
