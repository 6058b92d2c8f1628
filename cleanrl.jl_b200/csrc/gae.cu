// gae.cu — GAE reverse-time scan (gae(), ppo.jl:48-73) + returns (ppo.jl:181).
//
// Purely bandwidth-bound: per (env, step) it reads value 4 B + reward 4 B + done 1 B and writes
// advantage 4 B + return 4 B = 17 B. One thread owns VEC consecutive envs and walks t from the
// end; every row access is a coalesced, streaming (evict-first) 128-bit load/store across the
// warp. The recurrence is serial in t but the loads are not: each thread prefetches U rows into
// registers before it touches the dependent Float64 chain, so U x 36 B per thread are in flight (U = 4 measured best).
// values[t+1] is carried in a register, never re-read.
//
// The recurrence runs in Float64 exactly as the reference's promotion rules dictate
// (nonterm = 1.0 .- terminals and gae = 0.0 are Float64, ppo.jl:63,65) and uses _rn intrinsics
// so that no mul+add is contracted: results are bit-identical to the oracle.
#include <type_traits>

#include "kernels.h"

namespace {

template <int VEC> struct Vec;
template <> struct Vec<1> {
  using F = float;
  using B = unsigned char;
};
template <> struct Vec<4> {
  using F = float4;
  using B = uchar4;
};

__device__ __forceinline__ void unpack(float v, float o[1]) { o[0] = v; }
__device__ __forceinline__ void unpack(float4 v, float o[4]) { o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }
__device__ __forceinline__ void unpack(unsigned char v, unsigned char o[1]) { o[0] = v; }
__device__ __forceinline__ void unpack(uchar4 v, unsigned char o[4]) { o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }
__device__ __forceinline__ void pack(const float i[1], float& v) { v = i[0]; }
__device__ __forceinline__ void pack(const float i[4], float4& v) { v = make_float4(i[0], i[1], i[2], i[3]); }

template <int MODE, int VEC, int U>
__global__ void __launch_bounds__(128, VEC == 4 ? 5 : 1) gae_kernel(const float* __restrict__ values, const float* __restrict__ rewards,
                                                  const unsigned char* __restrict__ dones,
                                                  const float* __restrict__ next_value,
                                                  const unsigned char* __restrict__ next_done,
                                                  float* __restrict__ adv, float* __restrict__ ret, int T,
                                                  long long N, float gamma, float gl) {
  using VF = typename Vec<VEC>::F;
  using VB = typename Vec<VEC>::B;
  const long long nv = N / VEC;  // vectors per row
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nv) return;
  const VF* vv = reinterpret_cast<const VF*>(values);
  const VF* rr = reinterpret_cast<const VF*>(rewards);
  const VB* dd = reinterpret_cast<const VB*>(dones);
  VF* av = reinterpret_cast<VF*>(adv);
  VF* rv = reinterpret_cast<VF*>(ret);
  const double g = (double)gamma, gld = (double)gl;

  double gae[VEC];
  float vnext[VEC];
  unsigned char dnext[VEC];
#pragma unroll
  for (int k = 0; k < VEC; k++) gae[k] = 0.0;
  int t_hi;
  if (MODE == CRL_GAE_REF_COMPAT) {
    // Q1: the loop at ppo.jl:66 starts at T-1 (1-based); adv[T] is never written: define it as 0.
    const VF vl = __ldcs(vv + (long long)(T - 1) * nv + i);
    unpack(vl, vnext);
    unpack(T > 1 ? __ldcs(dd + (long long)(T - 1) * nv + i) : VB(), dnext);
    float z[VEC], rl[VEC];
#pragma unroll
    for (int k = 0; k < VEC; k++) { z[k] = 0.0f; rl[k] = 0.0f + vnext[k]; }
    VF o;
    pack(z, o);
    __stcs(av + (long long)(T - 1) * nv + i, o);
    pack(rl, o);
    __stcs(rv + (long long)(T - 1) * nv + i, o);
    t_hi = T - 2;
  } else {
    unpack(reinterpret_cast<const VF*>(next_value)[i], vnext);
    unpack(reinterpret_cast<const VB*>(next_done)[i], dnext);
    t_hi = T - 1;
    if (MODE == CRL_GAE_A2C_RETURNS) {
      // discounted_future_rewards (a2c.jl:13-24): the carried quantity is the return itself, seeded with final_value
#pragma unroll
      for (int k = 0; k < VEC; k++) gae[k] = (double)vnext[k];
    }
  }

  // One batch of U rows, newest first. FULL = all U rows exist: no per-row guards, so the compiler sees one basic block
  // and the three phases below really are three phases (with the guards every row was its own block and each row paid
  // its whole conversion -> delta -> recurrence -> conversion latency in turn: 25 us for 4096 envs x 128 steps). Only
  // the recurrence itself (one multiply and one add per row, Float64) is serial.
  auto batch = [&](int t0, auto full_c) {
    constexpr bool FULL = decltype(full_c)::value;
    VF v[U], r[U];
    VB d[U];
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int t = t0 - u;
      if (FULL || t >= 0) {
        v[u] = __ldcs(vv + (long long)t * nv + i);
        r[u] = __ldcs(rr + (long long)t * nv + i);
        if (t > 0) d[u] = __ldcs(dd + (long long)t * nv + i);  // dones[0] is never used
        else d[u] = VB();
      }
    }
    // phase 1 (independent per row): everything of the recurrence that does not depend on the carried value
    float vf[U][VEC];
    double dl[U][VEC], cf[U][VEC];   // REF/FIXED: delta and gamma*lambda*nonterm; A2C: reward and terminal flag
#pragma unroll
    for (int u = 0; u < U; u++) {
      if (FULL || t0 - u >= 0) {
        float rf[VEC];
        unsigned char df[VEC];
        unpack(v[u], vf[u]);
        unpack(r[u], rf);
        unpack(d[u], df);
#pragma unroll
        for (int k = 0; k < VEC; k++) {
          // the row above (newer) supplies values[t+1] and terminals[t+1]
          const float vn = u == 0 ? vnext[k] : vf[u - 1][k];
          unsigned char dn;
          if (u == 0) dn = dnext[k];
          else { unsigned char dp[VEC]; unpack(d[u - 1], dp); dn = dp[k]; }
          if (MODE == CRL_GAE_A2C_RETURNS) {
            dl[u][k] = (double)rf[k];
            cf[u][k] = dn ? 1.0 : 0.0;
          } else {
            const double nonterm = dn ? 0.0 : 1.0;  // 1.0 - terminals[t+1]
            dl[u][k] = __dsub_rn(__dadd_rn((double)rf[k], __dmul_rn(__dmul_rn(g, nonterm), (double)vn)), (double)vf[u][k]);
            cf[u][k] = __dmul_rn(gld, nonterm);
          }
        }
      }
    }
    // phase 2: the serial recurrence; phase 3 (outputs) is issued behind it row by row but depends on nothing later
#pragma unroll
    for (int u = 0; u < U; u++) {
      const int t = t0 - u;
      if (FULL || t >= 0) {
        float af[VEC], rt[VEC];
#pragma unroll
        for (int k = 0; k < VEC; k++) {
          if (MODE == CRL_GAE_A2C_RETURNS) {
            // future[t] = terminals[t] ? 0 : r[t] + γ future[t+1]; advantage = future - value (a2c.jl:20,83)
            gae[k] = cf[u][k] != 0.0 ? 0.0 : __dadd_rn(dl[u][k], __dmul_rn(g, gae[k]));
            rt[k] = (float)gae[k];
            af[k] = (float)__dsub_rn(gae[k], (double)vf[u][k]);
          } else {
            gae[k] = __dadd_rn(dl[u][k], __dmul_rn(cf[u][k], gae[k]));
            af[k] = (float)gae[k];
            rt[k] = __fadd_rn(af[k], vf[u][k]);
          }
        }
        VF o;
        pack(af, o);
        __stcs(av + (long long)t * nv + i, o);
        pack(rt, o);
        __stcs(rv + (long long)t * nv + i, o);
      }
    }
    // carried into the next (older) batch
    const int last = (FULL ? U : t0 + 1) - 1;
#pragma unroll
    for (int u = 0; u < U; u++) {
      if (u == last) {
        unsigned char dp[VEC];
        unpack(d[u], dp);
#pragma unroll
        for (int k = 0; k < VEC; k++) { vnext[k] = vf[u][k]; dnext[k] = dp[k]; }
      }
    }
  };
  for (int t0 = t_hi; t0 >= 0; t0 -= U) {
    if (t0 + 1 >= U) batch(t0, std::true_type());
    else batch(t0, std::false_type());
  }
}

template <int MODE>
cudaError_t launch_mode(const float* values, const float* rewards, const uint8_t* dones, const float* next_value,
                        const uint8_t* next_done, float* adv, float* ret, int T, long long N, float gamma, float gl,
                        cudaStream_t s) {
  auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
  auto al4 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3) == 0; };
  const bool vec_ok = (N % 4 == 0) && al16(values) && al16(rewards) && al16(adv) && al16(ret) && al4(dones) &&
                      (MODE == CRL_GAE_REF_COMPAT || (al16(next_value) && al4(next_done)));
  // vectorise only when there are enough threads to fill the machine several times over
  if (vec_ok && N / 4 >= 148LL * 128) {
    const long long nv = N / 4;
    const unsigned grid = (unsigned)((nv + 127) / 128);
    // prefetch depth U=4: measured on B200 at T=128, N=2^20 (profiles/r1_gae_sweep.txt): U=2 5.9 TB/s, U=4 6.1 TB/s,
    // U=8 4.8 TB/s, U=16 3.2 TB/s -- deeper prefetch costs occupancy and opens too many DRAM rows at once
    gae_kernel<MODE, 4, 4><<<grid, 128, 0, s>>>(values, rewards, dones, next_value, next_done, adv, ret, T, N, gamma, gl);
  } else {
    gae_kernel<MODE, 1, 16><<<(unsigned)((N + 127) / 128), 128, 0, s>>>(values, rewards, dones, next_value, next_done,
                                                                       adv, ret, T, N, gamma, gl);
  }
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_gae(const float* values, const float* rewards, const uint8_t* dones, const float* next_value,
                       const uint8_t* next_done, float* adv, float* ret, int T, long long N, float gamma,
                       float lambda, int mode, cudaStream_t s) {
  if (N == 0) return cudaSuccess;
  const float gl = gamma * lambda;  // Float32 product first (γ * λ * ..., ppo.jl:68)
  if (mode == CRL_GAE_REF_COMPAT)
    return launch_mode<CRL_GAE_REF_COMPAT>(values, rewards, dones, next_value, next_done, adv, ret, T, N, gamma, gl, s);
  if (mode == CRL_GAE_A2C_RETURNS)
    return launch_mode<CRL_GAE_A2C_RETURNS>(values, rewards, dones, next_value, next_done, adv, ret, T, N, gamma, gl, s);
  return launch_mode<CRL_GAE_FIXED>(values, rewards, dones, next_value, next_done, adv, ret, T, N, gamma, gl, s);
}
