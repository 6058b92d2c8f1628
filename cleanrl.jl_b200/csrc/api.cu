// api.cu — the C ABI of libcleanrl_cuda.so (include/cleanrl_cuda.h): handle, device memory,
// stream / CUDA-graph orchestration of one PPO update, NCCL plumbing, instrumentation.
// No CPU fallback anywhere: without a usable CUDA device every compute call fails loudly.
#include <dlfcn.h>
#include <nccl.h>  // declarations only; the library is resolved with dlopen at crl_comm_* time

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstring>
#include <string>
#include <vector>

#include "device_math.cuh"
#include "kernels.h"

// ------------------------------------------------------------------ errors
static thread_local std::string g_err;
static int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return code;
}
// for the other translation units of the library (dqn.cu): same thread-local message crl_last_error returns
int crl_internal_fail(int code, const char* msg) { g_err = msg; return code; }
#define CK(call)                                                                                        \
  do {                                                                                                  \
    cudaError_t e__ = (call);                                                                           \
    if (e__ != cudaSuccess)                                                                             \
      return fail(CRL_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)
#define CKRC(call)           \
  do {                       \
    int rc__ = (call);       \
    if (rc__ != CRL_OK) return rc__; \
  } while (0)

// ------------------------------------------------------------------ NCCL (dlopen)
struct NcclApi {
  void* handle = nullptr;
  decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&ncclCommInitRank) CommInitRank = nullptr;
  decltype(&ncclCommDestroy) CommDestroy = nullptr;
  decltype(&ncclAllReduce) AllReduce = nullptr;
  decltype(&ncclAllGather) AllGather = nullptr;
  decltype(&ncclGetErrorString) GetErrorString = nullptr;
};
static NcclApi g_nccl;
static int nccl_load() {
  if (g_nccl.handle) return CRL_OK;
  void* h = nullptr;
  const char* env = getenv("CRL_NCCL_LIB");
  if (env) h = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);  // reuse a copy torch already loaded
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return fail(CRL_ERR_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
#define SYM(name)                                                          \
  g_nccl.name = reinterpret_cast<decltype(g_nccl.name)>(dlsym(h, "nccl" #name)); \
  if (!g_nccl.name) return fail(CRL_ERR_NCCL, "libnccl lacks nccl" #name);
  SYM(GetUniqueId) SYM(CommInitRank) SYM(CommDestroy) SYM(AllReduce) SYM(AllGather) SYM(GetErrorString)
#undef SYM
  g_nccl.handle = h;
  return CRL_OK;
}
#define CKN(call)                                                                                     \
  do {                                                                                                \
    ncclResult_t r__ = (call);                                                                        \
    if (r__ != ncclSuccess) return fail(CRL_ERR_NCCL, "%s failed: %s", #call, g_nccl.GetErrorString(r__)); \
  } while (0)

// NCCL for the other translation units of the library (dqn.cu): communicator as an opaque pointer
int crl_internal_nccl_comm_init(void** comm, int world, int rank, const void* id128) {
  CKRC(nccl_load());
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  ncclComm_t cm = nullptr;
  CKN(g_nccl.CommInitRank(&cm, world, id, rank));
  *comm = cm;
  return CRL_OK;
}
int crl_internal_nccl_allreduce_sum(void* comm, void* buf, size_t count, int is_double, cudaStream_t s) {
  CKN(g_nccl.AllReduce(buf, buf, count, is_double ? ncclFloat64 : ncclFloat32, ncclSum, static_cast<ncclComm_t>(comm), s));
  return CRL_OK;
}
int crl_internal_nccl_allgather(void* comm, const void* send, void* recv, size_t bytes, cudaStream_t s) {
  CKN(g_nccl.AllGather(send, recv, bytes, ncclChar, static_cast<ncclComm_t>(comm), s));
  return CRL_OK;
}
void crl_internal_nccl_comm_destroy(void* comm) {
  if (comm && g_nccl.CommDestroy) g_nccl.CommDestroy(static_cast<ncclComm_t>(comm));
}

// ------------------------------------------------------------------ context
struct ProfEvent {
  int k;
  cudaEvent_t a, b;
};

struct crl_ctx {
  crl_config cfg;
  Layout L;
  int N, T, B, M;
  int sm_count;
  cudaStream_t stream;
  // parameters / optimiser
  float *params, *grads, *adam_m, *adam_v, *image;
  double* beta_pow;
  DevState* ds;
  // envs
  float* env_state;
  int* env_t;
  double* ep_return;
  int* ep_length;
  uint32_t* reset_count;
  float* next_obs;
  uint8_t* next_done;
  float* next_value;
  // rollout buffer
  float* state;
  void* action;
  float *logprob, *reward, *value, *advantage, *ret;
  uint8_t* terminal;
  // episodes
  EpisodeBuf* eb;
  crl_episode* records;
  int ep_capacity;
  // update scratch
  float* vnew;
  MbScalars *parts, *parts_send, *parts_recv;
  MbFinal* fin;
  float *gpart, *mpart;
  double *spart, *gsum, *stats_dev, *advparts;
  int32_t *idx_dev, *perm_dev;
  int grid_stats, grid_loss;
  // injected noise (lazy)
  double* action_noise_dev;
  float* reset_noise_dev;
  // pinned host mirrors
  crl_loss_stats* stats_host[2];  // double-buffered so the host can log update u-1 while update u runs
  EpisodeBuf* eb_host[2];
  cudaEvent_t fetch_ev[2];
  uint64_t update_seq;            // number of crl_train_update calls so far
  double* lr_host;
  // multi-GPU speculative updates: state snapshots for the (rare) exact replay
  unsigned char* snap[2];
  size_t snap_bytes;
  int* flag_host[2];              // pinned copy of DevState.spec_failed per result slot
  double lr_hist[2];
  uint64_t validated_seq;         // updates [0, validated_seq) are known to be exact
  uint64_t replays;               // speculative updates that had to be replayed exactly
  // graph
  cudaGraphExec_t graph_exec;
  uint64_t graph_kernels;
  // nccl
  ncclComm_t comm;
  // peer-memory (NVLink) exchange for the per-minibatch gradient allreduce
  unsigned char* p2p_buf;          // own exchange buffer (cudaMalloc, exported with cudaIpc)
  unsigned char* p2p_peer[CRL_MAX_WORLD];
  unsigned char** p2p_peers_dev;
  unsigned long long* p2p_seq;
  unsigned int* p2p_count;
  int* p2p_err;
  int p2p_stride;
  size_t p2p_flags_off;
  bool p2p_on;
  size_t ll_off;                   // flag-in-data region of the exchange buffer (fused tail), [2 slots][world][ll_stride] x 16 B
  int ll_stride;
  size_t adv_off;                  // same for the per-update advantage sums (adv_stats), [2 slots][world][adv_stride] x 16 B
  int adv_stride;
  long long p2p_timeout_cycles;
  // fused tail of the tcgen05 update kernel
  unsigned long long* grid_bar;
  double* normpart;
  int fused_grid;                  // grid size the barrier counter is used with (constant per handle)
  // instrumentation
  uint64_t launches;
  bool profiling;
  std::vector<ProfEvent> prof_pending;
  std::vector<cudaEvent_t> ev_pool;
  crl_kernel_times times;
  bool rolled, gae_done, have_update;
};

static int use_device(const crl_ctx* c) {
  CK(cudaSetDevice(c->cfg.device));
  return CRL_OK;
}

// Speculative updates (crl_train_update) are repaired lazily by validate_updates(). Every entry point that reads or
// mutates handle state settles them first, so that no caller can observe -- or build on -- the output of a failed
// speculation (a failed one is rare: it costs a stream synchronisation only when updates are pending).
static int validate_updates(crl_ctx* c, uint64_t upto);
static int settle(crl_ctx* c);
#define SETTLE(c) CKRC(settle(c))

template <typename T> static int dalloc(T** p, size_t n) {
  CK(cudaMalloc(reinterpret_cast<void**>(p), std::max<size_t>(n, 1) * sizeof(T)));
  CK(cudaMemset(*p, 0, std::max<size_t>(n, 1) * sizeof(T)));
  return CRL_OK;
}

// profiling wrapper: CUDA events on the handle's stream around one kernel class
struct KernelScope {
  crl_ctx* c;
  int k;
  cudaEvent_t a = nullptr, b = nullptr;
  KernelScope(crl_ctx* c_, int k_, bool mine = true) : c(c_), k(k_) {
    if (mine) c->launches++;
    if (!c->profiling) return;
    auto get = [&]() {
      cudaEvent_t e;
      if (!c->ev_pool.empty()) { e = c->ev_pool.back(); c->ev_pool.pop_back(); }
      else cudaEventCreate(&e);
      return e;
    };
    a = get();
    b = get();
    cudaEventRecord(a, c->stream);
  }
  ~KernelScope() {
    if (!c->profiling) return;
    cudaEventRecord(b, c->stream);
    c->prof_pending.push_back({k, a, b});
  }
};

static void prof_collect(crl_ctx* c) {
  for (auto& p : c->prof_pending) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, p.a, p.b) == cudaSuccess) {
      c->times.ms[p.k] += ms;
      c->times.launches[p.k] += 1;
    }
    c->ev_pool.push_back(p.a);
    c->ev_pool.push_back(p.b);
  }
  c->prof_pending.clear();
}

// ------------------------------------------------------------------ library
extern "C" CRL_API int crl_version(void) { return CRL_VERSION; }
extern "C" CRL_API const char* crl_last_error(void) { return g_err.c_str(); }
extern "C" CRL_API int crl_device_count(int32_t* count) {
  if (!count) return fail(CRL_ERR_INVALID, "count is NULL");
  int n = 0;
  CK(cudaGetDeviceCount(&n));
  *count = n;
  return CRL_OK;
}

static int check_cfg(const crl_config* c) {
  if (!c) return fail(CRL_ERR_INVALID, "cfg is NULL");
  if (c->struct_size != (int32_t)sizeof(crl_config))
    return fail(CRL_ERR_INVALID, "crl_config.struct_size %d != %d (header mismatch)", c->struct_size, (int)sizeof(crl_config));
  if (c->env_kind != CRL_ENV_CARTPOLE && c->env_kind != CRL_ENV_PENDULUM) return fail(CRL_ERR_INVALID, "unknown env_kind %d", c->env_kind);
  if (c->num_envs < 1 || c->num_steps < 1 || c->num_minibatches < 1 || c->update_epochs < 0)
    return fail(CRL_ERR_INVALID, "num_envs/num_steps/num_minibatches must be >= 1");
  const long long B = (long long)c->num_envs * c->num_steps;
  if (B >= (1ll << 31)) return fail(CRL_ERR_INVALID, "batch of %lld samples exceeds int32 indexing", B);
  if (B % c->num_minibatches != 0)  // Q10: the reference indexes out of bounds otherwise (ppo.jl:197,203)
    return fail(CRL_ERR_INVALID, "num_envs*num_steps = %lld is not divisible by num_minibatches = %d", B, c->num_minibatches);
  if (B / c->num_minibatches < 2) return fail(CRL_ERR_INVALID, "minibatch size must be >= 2 (corrected std, ppo.jl:221)");
  if (c->world_size < 1 || c->rank < 0 || c->rank >= c->world_size) return fail(CRL_ERR_INVALID, "bad world_size/rank");
  if (c->world_size > CRL_MAX_WORLD) return fail(CRL_ERR_INVALID, "world_size > %d is not supported", CRL_MAX_WORLD);
  if (c->gae_mode != CRL_GAE_REF_COMPAT && c->gae_mode != CRL_GAE_FIXED && c->gae_mode != CRL_GAE_A2C_RETURNS)
    return fail(CRL_ERR_INVALID, "bad gae_mode");
  // A2C (a2c.jl:78-97) steps once per rollout on the whole batch: the actor's advantage is the return minus the critic
  // output recorded by that rollout, which is only the current critic for the first (and only) minibatch
  if ((c->flags & CRL_FLAG_A2C) &&
      (c->num_minibatches != 1 || c->update_epochs != 1 || c->gae_mode != CRL_GAE_A2C_RETURNS))
    return fail(CRL_ERR_INVALID, "CRL_FLAG_A2C needs num_minibatches = 1, update_epochs = 1 and gae_mode = CRL_GAE_A2C_RETURNS");
  return CRL_OK;
}

extern "C" CRL_API int crl_create(const crl_config* cfg, crl_ctx** out) {
  if (!out) return fail(CRL_ERR_INVALID, "out is NULL");
  *out = nullptr;
  CKRC(check_cfg(cfg));
  int ndev = 0;
  CK(cudaGetDeviceCount(&ndev));
  if (cfg->device < 0 || cfg->device >= ndev) return fail(CRL_ERR_CUDA, "device %d not present (%d CUDA devices)", cfg->device, ndev);
  CK(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10)
    return fail(CRL_ERR_CUDA, "device %d is sm_%d%d; this library contains sm_100a code only", cfg->device, prop.major, prop.minor);

  CK(kernels_init_rollout());
  CK(kernels_init_update());
  crl_ctx* c = new crl_ctx();
  memset(&c->times, 0, sizeof(c->times));
  c->cfg = *cfg;
  make_layout(cfg->env_kind, &c->L);
  c->N = cfg->num_envs; c->T = cfg->num_steps; c->B = c->N * c->T; c->M = c->B / cfg->num_minibatches;
  c->sm_count = prop.multiProcessorCount;
  c->graph_exec = nullptr; c->graph_kernels = 0; c->comm = nullptr; c->launches = 0; c->profiling = false;
  c->rolled = c->gae_done = c->have_update = false;
  c->action_noise_dev = nullptr; c->reset_noise_dev = nullptr;
  const Layout& L = c->L;
  const size_t N = c->N, B = c->B;
#define A_(x) do { int rc_ = (x); if (rc_ != CRL_OK) { crl_destroy(c); return rc_; } } while (0)
  cudaError_t se = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
  if (se != cudaSuccess) { delete c; return fail(CRL_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(se)); }
  A_(dalloc(&c->params, L.P)); A_(dalloc(&c->grads, L.P)); A_(dalloc(&c->adam_m, L.P)); A_(dalloc(&c->adam_v, L.P));
  A_(dalloc(&c->beta_pow, 2 * CRL_MAX_ARRAYS)); A_(dalloc(&c->ds, 1)); A_(dalloc(&c->grid_bar, 1)); A_(dalloc(&c->normpart, (size_t)CRL_MAX_ARRAYS * prop.multiProcessorCount));
  A_(dalloc(&c->image, param_image_floats(cfg->env_kind)));
  A_(dalloc(&c->env_state, N * L.S)); A_(dalloc(&c->env_t, N)); A_(dalloc(&c->ep_return, N)); A_(dalloc(&c->ep_length, N));
  A_(dalloc(&c->reset_count, N)); A_(dalloc(&c->next_obs, N * L.D)); A_(dalloc(&c->next_done, N)); A_(dalloc(&c->next_value, N));
  A_(dalloc(&c->state, B * L.D));
  { float* act; A_(dalloc(&act, B * (L.continuous ? L.A : 1))); c->action = act; }
  A_(dalloc(&c->logprob, B)); A_(dalloc(&c->reward, B)); A_(dalloc(&c->value, B)); A_(dalloc(&c->advantage, B));
  A_(dalloc(&c->ret, B)); A_(dalloc(&c->terminal, B));
  c->ep_capacity = cfg->episode_capacity > 0 ? cfg->episode_capacity : (int)std::min<size_t>(B, B / 4 + N);
  A_(dalloc(&c->eb, 1)); A_(dalloc(&c->records, c->ep_capacity));
  c->grid_stats = mb_stats_grid(c->M, c->sm_count);
  c->grid_loss = loss_grad_grid(c->M, c->sm_count);
  A_(dalloc(&c->vnew, c->M)); A_(dalloc(&c->parts, c->sm_count)); A_(dalloc(&c->parts_send, 1));
  A_(dalloc(&c->parts_recv, cfg->world_size)); A_(dalloc(&c->fin, 1));
  A_(dalloc(&c->gpart, (size_t)c->sm_count * L.P)); A_(dalloc(&c->spart, (size_t)c->sm_count * 4));
  A_(dalloc(&c->gsum, L.P + 4 + CRL_MAX_WORLD)); A_(dalloc(&c->mpart, c->sm_count));
  const size_t nmb = (size_t)std::max(1, cfg->update_epochs) * cfg->num_minibatches;
  A_(dalloc(&c->advparts, nmb * ADV_CHUNKS * 2));
  A_(dalloc(&c->stats_dev, nmb * 4)); A_(dalloc(&c->idx_dev, B)); A_(dalloc(&c->perm_dev, (size_t)std::max(1, cfg->update_epochs) * B));
  {
    cudaError_t e3 = cudaMallocHost(reinterpret_cast<void**>(&c->lr_host), 16 * sizeof(double));
    bool ok = e3 == cudaSuccess;
    for (int i = 0; i < 2 && ok; i++) {
      ok = ok && cudaMallocHost(reinterpret_cast<void**>(&c->stats_host[i]), nmb * sizeof(crl_loss_stats)) == cudaSuccess;
      ok = ok && cudaMallocHost(reinterpret_cast<void**>(&c->eb_host[i]), sizeof(EpisodeBuf)) == cudaSuccess;
      ok = ok && cudaEventCreateWithFlags(&c->fetch_ev[i], cudaEventDisableTiming) == cudaSuccess;
      if (ok) { memset(c->stats_host[i], 0, nmb * sizeof(crl_loss_stats)); memset(c->eb_host[i], 0, sizeof(EpisodeBuf)); }
    }
    for (int i = 0; i < 2 && ok; i++) {
      ok = ok && cudaMallocHost(reinterpret_cast<void**>(&c->flag_host[i]), 2 * sizeof(int)) == cudaSuccess;
      if (ok) { c->flag_host[i][0] = 0; c->flag_host[i][1] = 0; }
    }
    if (!ok) { crl_destroy(c); return fail(CRL_ERR_CUDA, "pinned host allocation failed"); }
    c->update_seq = 0;
    c->validated_seq = 0;
  }
#undef A_
  // Flux keeps (β1, β2) as the initial power state of every array
  std::vector<double> bp(2 * CRL_MAX_ARRAYS);
  for (int i = 0; i < CRL_MAX_ARRAYS; i++) { bp[2 * i] = 0.9; bp[2 * i + 1] = 0.999; }
  cudaMemcpy(c->beta_pow, bp.data(), bp.size() * sizeof(double), cudaMemcpyHostToDevice);
  *out = c;
  return CRL_OK;
}

extern "C" CRL_API int crl_destroy(crl_ctx* c) {
  if (!c) return CRL_OK;
  cudaSetDevice(c->cfg.device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  if (c->graph_exec) cudaGraphExecDestroy(c->graph_exec);
  if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
  for (int r = 0; r < CRL_MAX_WORLD; r++)
    if (c->p2p_peer[r] && c->p2p_peer[r] != c->p2p_buf) cudaIpcCloseMemHandle(c->p2p_peer[r]);
  { void* pp[] = {c->p2p_buf, c->p2p_peers_dev, c->p2p_seq, c->p2p_err, c->p2p_count}; for (void* q : pp) if (q) cudaFree(q); }
  for (auto& p : c->prof_pending) { cudaEventDestroy(p.a); cudaEventDestroy(p.b); }
  for (auto e : c->ev_pool) cudaEventDestroy(e);
  void* ptrs[] = {c->grid_bar, c->normpart, c->image, c->params, c->grads, c->adam_m, c->adam_v, c->beta_pow, c->ds, c->env_state, c->env_t, c->ep_return,
                  c->ep_length, c->reset_count, c->next_obs, c->next_done, c->next_value, c->state, c->action, c->logprob,
                  c->reward, c->value, c->advantage, c->ret, c->terminal, c->eb, c->records, c->vnew, c->parts,
                  c->parts_send, c->parts_recv, c->fin, c->gpart, c->mpart, c->advparts, c->spart, c->gsum, c->stats_dev, c->idx_dev,
                  c->perm_dev, c->action_noise_dev, c->reset_noise_dev};
  for (void* p : ptrs) if (p) cudaFree(p);
  for (int i = 0; i < 2; i++) {
    if (c->stats_host[i]) cudaFreeHost(c->stats_host[i]);
    if (c->eb_host[i]) cudaFreeHost(c->eb_host[i]);
    if (c->fetch_ev[i]) cudaEventDestroy(c->fetch_ev[i]);
    if (c->flag_host[i]) cudaFreeHost(c->flag_host[i]);
    if (c->snap[i]) cudaFree(c->snap[i]);
  }
  if (c->lr_host) cudaFreeHost(c->lr_host);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
  return CRL_OK;
}

extern "C" CRL_API int crl_sync(crl_ctx* c) {
  if (!c) return fail(CRL_ERR_INVALID, "ctx is NULL");
  CKRC(use_device(c));
  SETTLE(c);
  CK(cudaStreamSynchronize(c->stream));
  return CRL_OK;
}

extern "C" CRL_API int crl_dims(const crl_ctx* c, int32_t* D, int32_t* A, int32_t* S, int32_t* P, int32_t* n_arrays) {
  if (!c) return fail(CRL_ERR_INVALID, "ctx is NULL");
  if (D) *D = c->L.D;
  if (A) *A = c->L.A;
  if (S) *S = c->L.S;
  if (P) *P = c->L.P;
  if (n_arrays) *n_arrays = c->L.n_arrays;
  return CRL_OK;
}

extern "C" CRL_API int crl_param_layout(const crl_ctx* c, int32_t* offsets, int32_t* sizes, int32_t max_arrays) {
  if (!c || !offsets || !sizes) return fail(CRL_ERR_INVALID, "NULL argument");
  if (max_arrays < c->L.n_arrays) return fail(CRL_ERR_INVALID, "need room for %d arrays", c->L.n_arrays);
  for (int i = 0; i < c->L.n_arrays; i++) { offsets[i] = c->L.off[i]; sizes[i] = c->L.size[i]; }
  return CRL_OK;
}

// ------------------------------------------------------------------ params / optimiser state
static int copy_vec(crl_ctx* c, void* dst, const void* src, size_t bytes, cudaMemcpyKind kind) {
  CKRC(use_device(c));
  CK(cudaMemcpyAsync(dst, src, bytes, kind, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return CRL_OK;
}
extern "C" CRL_API int crl_set_params(crl_ctx* c, const float* host, int32_t n) {
  if (!c || !host || n != c->L.P) return fail(CRL_ERR_INVALID, "crl_set_params: expected %d floats", c ? c->L.P : -1);
  CKRC(use_device(c));
  SETTLE(c);
  CK(cudaMemcpyAsync(c->params, host, 4 * (size_t)n, cudaMemcpyHostToDevice, c->stream));
  {
    KernelScope ks(c, CRL_K_OTHER);
    CK(launch_param_image(c->cfg.env_kind, c->params, c->image, c->stream));  // keep the staging image in sync
  }
  CK(cudaStreamSynchronize(c->stream));
  return CRL_OK;
}
extern "C" CRL_API int crl_get_params(crl_ctx* c, float* host, int32_t n) {
  if (!c || !host || n != c->L.P) return fail(CRL_ERR_INVALID, "crl_get_params: expected %d floats", c ? c->L.P : -1);
  SETTLE(c);
  return copy_vec(c, host, c->params, 4 * (size_t)n, cudaMemcpyDeviceToHost);
}
extern "C" CRL_API int crl_get_grads(crl_ctx* c, float* host, int32_t n) {
  if (!c || !host || n != c->L.P) return fail(CRL_ERR_INVALID, "crl_get_grads: expected %d floats", c ? c->L.P : -1);
  SETTLE(c);
  return copy_vec(c, host, c->grads, 4 * (size_t)n, cudaMemcpyDeviceToHost);
}
extern "C" CRL_API int crl_get_adam_state(crl_ctx* c, float* m, float* v, double* beta_pow) {
  if (!c || !m || !v || !beta_pow) return fail(CRL_ERR_INVALID, "NULL argument");
  SETTLE(c);
  CKRC(copy_vec(c, m, c->adam_m, 4 * (size_t)c->L.P, cudaMemcpyDeviceToHost));
  CKRC(copy_vec(c, v, c->adam_v, 4 * (size_t)c->L.P, cudaMemcpyDeviceToHost));
  return copy_vec(c, beta_pow, c->beta_pow, 16 * (size_t)c->L.n_arrays, cudaMemcpyDeviceToHost);
}
extern "C" CRL_API int crl_set_adam_state(crl_ctx* c, const float* m, const float* v, const double* beta_pow) {
  if (!c || !m || !v || !beta_pow) return fail(CRL_ERR_INVALID, "NULL argument");
  SETTLE(c);
  CKRC(copy_vec(c, c->adam_m, m, 4 * (size_t)c->L.P, cudaMemcpyHostToDevice));
  CKRC(copy_vec(c, c->adam_v, v, 4 * (size_t)c->L.P, cudaMemcpyHostToDevice));
  return copy_vec(c, c->beta_pow, beta_pow, 16 * (size_t)c->L.n_arrays, cudaMemcpyHostToDevice);
}

// ------------------------------------------------------------------ envs
extern "C" CRL_API int crl_env_reset(crl_ctx* c) {
  if (!c) return fail(CRL_ERR_INVALID, "ctx is NULL");
  CKRC(use_device(c));
  SETTLE(c);
  {
    KernelScope ks(c, CRL_K_OTHER);
    CK(launch_env_reset(c->cfg.env_kind, c->N, c->cfg.seed, c->cfg.env_id_base, c->env_state, c->env_t, c->ep_return,
                        c->ep_length, c->reset_count, c->next_obs, c->next_done, c->stream));
  }
  return CRL_OK;
}
extern "C" CRL_API int crl_env_set_state(crl_ctx* c, const float* state, const int32_t* t) {
  if (!c || !state) return fail(CRL_ERR_INVALID, "NULL argument");
  CKRC(use_device(c));
  SETTLE(c);
  CK(cudaMemcpyAsync(c->env_state, state, 4 * (size_t)c->N * c->L.S, cudaMemcpyHostToDevice, c->stream));
  if (t) CK(cudaMemcpyAsync(c->env_t, t, 4 * (size_t)c->N, cudaMemcpyHostToDevice, c->stream));
  else CK(cudaMemsetAsync(c->env_t, 0, 4 * (size_t)c->N, c->stream));
  {
    KernelScope ks(c, CRL_K_OTHER);
    CK(launch_env_refresh(c->cfg.env_kind, c->N, c->env_state, c->next_obs, c->next_done, c->stream));
  }
  CK(cudaStreamSynchronize(c->stream));
  return CRL_OK;
}

// ------------------------------------------------------------------ rollout / GAE
static RolloutArgs rollout_args(crl_ctx* c, const double* an, const float* rn) {
  RolloutArgs a;
  a.params = c->params; a.ds = c->ds; a.seed = c->cfg.seed; a.env_id_base = c->cfg.env_id_base;
  a.N = c->N; a.T = c->T; a.max_steps = c->cfg.max_episode_steps;
  a.env_state = c->env_state; a.env_t = c->env_t; a.ep_return = c->ep_return; a.ep_length = c->ep_length;
  a.reset_count = c->reset_count; a.next_obs = c->next_obs; a.next_done = c->next_done; a.next_value = c->next_value;
  a.state = c->state; a.action = c->action; a.logprob = c->logprob; a.reward = c->reward; a.value = c->value;
  a.terminal = c->terminal; a.action_noise = an; a.reset_noise = rn; a.eb = c->eb; a.records = c->records;
  a.ep_capacity = c->ep_capacity;
  a.fresh_obs_after_reset = (c->cfg.flags & CRL_FLAG_A2C) ? 1 : 0;
  return a;
}

static int enqueue_rollout(crl_ctx* c, const double* an_dev, const float* rn_dev) {
  {
    KernelScope ks(c, CRL_K_OTHER);
    CK(launch_episode_buf_init(c->eb, c->stream));
  }
  KernelScope ks(c, CRL_K_ROLLOUT);
  CK(launch_rollout(c->cfg.env_kind, rollout_args(c, an_dev, rn_dev), c->stream));
  return CRL_OK;
}

extern "C" CRL_API int crl_rollout(crl_ctx* c, const double* action_noise, const float* reset_noise) {
  if (!c) return fail(CRL_ERR_INVALID, "ctx is NULL");
  CKRC(use_device(c));
  SETTLE(c);
  const size_t B = c->B;
  const double* an = nullptr;
  const float* rn = nullptr;
  if (action_noise) {
    const size_t n = B * (c->L.continuous ? c->L.A : 1);
    if (!c->action_noise_dev) CK(cudaMalloc(reinterpret_cast<void**>(&c->action_noise_dev), n * sizeof(double)));
    CK(cudaMemcpyAsync(c->action_noise_dev, action_noise, n * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    an = c->action_noise_dev;
  }
  if (reset_noise) {
    if (!c->reset_noise_dev) CK(cudaMalloc(reinterpret_cast<void**>(&c->reset_noise_dev), B * 4 * sizeof(float)));
    CK(cudaMemcpyAsync(c->reset_noise_dev, reset_noise, B * 4 * sizeof(float), cudaMemcpyHostToDevice, c->stream));
    rn = c->reset_noise_dev;
  }
  CKRC(enqueue_rollout(c, an, rn));
  {
    KernelScope ks(c, CRL_K_OTHER);
    CK(launch_advance(c->ds, (unsigned long long)c->T, 0ull, c->stream));
  }
  CK(cudaStreamSynchronize(c->stream));  // host noise buffers are borrowed for this call only
  c->rolled = true;
  c->gae_done = false;
  return CRL_OK;
}

static int enqueue_gae(crl_ctx* c) {
  KernelScope ks(c, CRL_K_GAE);
  CK(launch_gae(c->value, c->reward, c->terminal, c->next_value, c->next_done, c->advantage, c->ret, c->T, c->N,
                c->cfg.gamma, c->cfg.gae_lambda, c->cfg.gae_mode, c->stream));
  return CRL_OK;
}

extern "C" CRL_API int crl_gae(crl_ctx* c) {
  if (!c) return fail(CRL_ERR_INVALID, "ctx is NULL");
  if (!c->rolled) return fail(CRL_ERR_STATE, "crl_gae called before crl_rollout");
  CKRC(use_device(c));
  SETTLE(c);
  CKRC(enqueue_gae(c));
  c->gae_done = true;
  return CRL_OK;
}

// ------------------------------------------------------------------ update
static IdxSrc idx_perm(crl_ctx* c, int epoch, int start) {
  IdxSrc ix;
  ix.arr = nullptr; ix.start = (uint32_t)start; ix.B = (uint32_t)c->B; ix.half_bits = perm_half_bits((uint32_t)c->B);
  ix.epoch = (uint32_t)epoch; ix.rank = (uint32_t)c->cfg.rank; ix.seed = c->cfg.seed; ix.ds = c->ds;
  return ix;
}
static IdxSrc idx_array(crl_ctx* c, const int32_t* arr) {
  IdxSrc ix = idx_perm(c, 0, 0);
  ix.arr = arr;
  return ix;
}

// one minibatch: mb_stats -> [all-gather] -> mb_count -> [allreduce cnt] -> loss_grad -> grad_reduce
// -> [allreduce grads] -> clip_adam. lr_host < 0 reads lr from DevState.
// ---- snapshots (multi-GPU speculative path) ---------------------------------------------------------------
struct SnapItem { void* ptr; size_t bytes; };
static std::vector<SnapItem> snap_items(crl_ctx* c) {
  const size_t P = c->L.P, N = c->N;
  return {{c->params, 4 * P}, {c->image, 4 * (size_t)param_image_floats(c->cfg.env_kind)}, {c->adam_m, 4 * P},
          {c->adam_v, 4 * P}, {c->beta_pow, 16 * (size_t)CRL_MAX_ARRAYS}, {c->env_state, 4 * N * c->L.S}, {c->env_t, 4 * N},
          {c->ep_return, 8 * N}, {c->ep_length, 4 * N}, {c->reset_count, 4 * N}, {c->ds, sizeof(DevState)}};
}
// The snapshot taken before every speculative update: one launch instead of eleven device-to-device copies (the items
// are all multiples of 4 bytes; 330 KB at BASELINE configs[1]).
constexpr int SNAP_MAX = 12;
struct SnapCopy { const uint32_t* src[SNAP_MAX]; uint32_t* dst[SNAP_MAX]; unsigned words[SNAP_MAX]; int n; };
__global__ void snapshot_kernel(SnapCopy sc) {
  const unsigned stride = gridDim.x * blockDim.x, t0 = blockIdx.x * blockDim.x + threadIdx.x;
  for (int i = 0; i < sc.n; i++) {
    const uint32_t* __restrict__ s = sc.src[i];
    uint32_t* __restrict__ d = sc.dst[i];
    const unsigned w = sc.words[i], w4 = w / 4;   // sources and destinations are 16-byte aligned
    for (unsigned k = t0; k < w4; k += stride) reinterpret_cast<uint4*>(d)[k] = reinterpret_cast<const uint4*>(s)[k];
    for (unsigned k = 4 * w4 + t0; k < w; k += stride) d[k] = s[k];
  }
}
static int snapshot_copy(crl_ctx* c, int slot, bool restore) {
  size_t off = 0;
  if (!restore) {
    SnapCopy sc;
    sc.n = 0;
    bool ok = true;
    for (auto& it : snap_items(c)) {
      if (sc.n >= SNAP_MAX || (it.bytes & 3) || (reinterpret_cast<uintptr_t>(it.ptr) & 15)) { ok = false; break; }
      sc.src[sc.n] = reinterpret_cast<const uint32_t*>(it.ptr);
      sc.dst[sc.n] = reinterpret_cast<uint32_t*>(c->snap[slot] + off);
      sc.words[sc.n] = (unsigned)(it.bytes / 4);
      sc.n++;
      off += (it.bytes + 15) & ~size_t(15);
    }
    if (ok) {
      KernelScope ks(c, CRL_K_OTHER);
      snapshot_kernel<<<64, 256, 0, c->stream>>>(sc);
      CK(cudaGetLastError());
      return CRL_OK;
    }
    off = 0;
  }
  for (auto& it : snap_items(c)) {
    const size_t b = (it.bytes + 15) & ~size_t(15);
    if (restore) CK(cudaMemcpyAsync(it.ptr, c->snap[slot] + off, it.bytes, cudaMemcpyDeviceToDevice, c->stream));
    else CK(cudaMemcpyAsync(c->snap[slot] + off, it.ptr, it.bytes, cudaMemcpyDeviceToDevice, c->stream));
    off += b;
  }
  return CRL_OK;
}
static int snapshot_alloc(crl_ctx* c) {
  if (c->snap[0]) return CRL_OK;
  size_t tot = 0;
  for (auto& it : snap_items(c)) tot += (it.bytes + 15) & ~size_t(15);
  c->snap_bytes = tot;
  for (int i = 0; i < 2; i++) CK(cudaMalloc(reinterpret_cast<void**>(&c->snap[i]), tot));
  return CRL_OK;
}

static int enqueue_adv_stats(crl_ctx* c, const int32_t* arr_base, int M, int nmb, int n_sets) {
  AdvStatsArgs aa;
  aa.idx.arr = nullptr; aa.idx.start = 0; aa.idx.B = (uint32_t)c->B; aa.idx.half_bits = perm_half_bits((uint32_t)c->B);
  aa.idx.epoch = 0; aa.idx.rank = (uint32_t)c->cfg.rank; aa.idx.seed = c->cfg.seed; aa.idx.ds = c->ds;
  aa.arr_base = arr_base; aa.B = c->B; aa.M = M; aa.nmb = nmb; aa.n_sets = n_sets;
  aa.advantages = c->advantage; aa.advparts = c->advparts;
  aa.x_peers = nullptr; aa.x_local = nullptr; aa.x_off = 0; aa.x_world = 1; aa.x_rank = 0; aa.x_stride = 0; aa.x_err = nullptr; aa.x_timeout = 0;
  if (c->cfg.world_size > 1 && c->p2p_on && n_sets * ADV_CHUNKS * 2 <= c->adv_stride) {
    aa.x_peers = c->p2p_peers_dev; aa.x_local = c->p2p_buf; aa.x_off = c->adv_off; aa.x_world = c->cfg.world_size;
    aa.x_rank = c->cfg.rank; aa.x_stride = c->adv_stride; aa.x_err = c->p2p_err; aa.x_timeout = c->p2p_timeout_cycles;
  }
  KernelScope ks(c, CRL_K_MB_STATS);
  CK(launch_adv_stats(aa, c->stream));
  return CRL_OK;
}

static AdamArgs adam_args(crl_ctx* c, int M, double lr_host, double* stats_slot) {
  AdamArgs aa;
  memset(&aa, 0, sizeof(aa));
  aa.env_kind = c->cfg.env_kind; aa.params = c->params; aa.image = c->image; aa.gsum = c->gsum; aa.gf = nullptr;
  aa.grad_scale = 1.0; aa.stat_ranks = 1.0; aa.grads_out = c->grads; aa.m = c->adam_m; aa.v = c->adam_v;
  aa.beta_pow = c->beta_pow; aa.ds = c->ds; aa.lr_host = lr_host; aa.clip_norm = c->cfg.clip_norm;
  aa.ent_coeff = c->cfg.ent_coeff; aa.v_coef = c->cfg.v_coef; aa.M_global = (double)M; aa.A = c->L.A;
  aa.stats_out = stats_slot; aa.world = 1; aa.rank = c->cfg.rank; aa.M = M; aa.P = c->L.P; aa.ds_rw = c->ds; aa.fin = c->fin;
  aa.algo = (c->cfg.flags & CRL_FLAG_A2C) ? 1 : 0;
  return aa;
}

// One minibatch (ppo.jl:197-251).
//  spec = true (throughput path, any number of GPUs): loss_grad speculates that the scalar s of the value loss never
//    wins the max (Q5) and uses advantage statistics precomputed for the whole update; grad_reduce packs
//    gradient + loss sums + sum s + this rank's min behind each other; the finishing kernel exchanges them with the
//    peers (NVLink peer memory, or one NCCL allreduce), verifies the speculation and applies clip + Adam.
//    3 launches per minibatch, 1 exchange. A failed verification is repaired by validate_updates().
//  spec = false (stage-by-stage API, replay): exact statistics first: mb_stats -> [all-gather] -> mb_count ->
//    [allreduce count] -> loss_grad(EXACT) -> grad_reduce -> [allreduce] -> clip_adam.
// lr_host < 0 reads lr from DevState. `set` indexes the advantage sums written by enqueue_adv_stats.
static int enqueue_minibatch(crl_ctx* c, const IdxSrc& ix, int M, double lr_host, double* stats_slot, int set,
                             bool spec = false) {
  const int W = c->cfg.world_size;
  const bool multi = W > 1;
  const bool local_stats = (c->cfg.flags & CRL_FLAG_LOCAL_STATS) != 0;
  if (multi && !c->comm) return fail(CRL_ERR_STATE, "world_size > 1 but crl_comm_init was not called");
  UpdateArgs ua;
  memset(&ua, 0, sizeof(ua));
  ua.env_kind = c->cfg.env_kind; ua.params = c->params; ua.image = c->image; ua.idx = ix; ua.M = M;
  ua.states = c->state; ua.actions = c->action; ua.logprobs = c->logprob; ua.advantages = c->advantage;
  ua.returns = c->ret; ua.values = c->value;
  ua.clip_coef = c->cfg.clip_coef; ua.ent_coeff = c->cfg.ent_coeff; ua.v_coef = c->cfg.v_coef;
  ua.vnew = c->vnew; ua.parts = c->parts; ua.n_parts_cap = c->sm_count;
  const int gs = mb_stats_grid(M, c->sm_count);
  ua.grid_loss = loss_grad_grid(M, c->sm_count);
  ua.parts_in = c->parts; ua.n_parts_in = gs; ua.fin = c->fin; ua.world = 1;
  ua.gpart = c->gpart; ua.spart = c->spart; ua.gsum = c->gsum;
  ua.mode = LG_EXACT; ua.advparts = c->advparts + (size_t)set * ADV_CHUNKS * 2; ua.mpart = c->mpart;
  ua.rank = c->cfg.rank;
  ua.algo = (c->cfg.flags & CRL_FLAG_A2C) ? 1 : 0;
  ua.no_vclip = (c->cfg.flags & CRL_FLAG_NO_VCLIP) ? 1 : 0;
  ua.tc_net_a = c->L.critic - c->L.actor; ua.tc_net_c = (c->L.continuous ? c->L.logstd : c->L.P) - c->L.critic;
  ua.values_fresh = spec ? 1 : 0;       // throughput path: the rollout that filled `value` used the current parameters
  // Fused tail: the tcgen05 kernel reduces, exchanges and applies clip + Adam itself (one cooperative launch per
  // minibatch). Needs the peer-memory exchange when there are several ranks; the FFMA kernel (CRL_NO_TC=1) and the
  // NCCL fallback keep the 3-kernel chain.
  const bool want_fuse = (spec || ua.algo == 1) && (!multi || c->p2p_on);
  loss_grad_tc_plan(&ua, c->sm_count, want_fuse);  // tensor-core kernel when it applies: sets grid_loss / tc_actor_ctas
  AdamArgs aa = adam_args(c, M, lr_host, stats_slot);
  if (spec || ua.algo == 1) {  // the A2C losses have no minibatch-global scalars: the 3-kernel chain is already exact
    const bool p2p = multi && c->p2p_on;
    ua.mode = LG_SPEC; ua.world = W;
    if (p2p) {
      ua.p2p_data = reinterpret_cast<double*>(c->p2p_buf); ua.p2p_stride = c->p2p_stride; ua.p2p_seq = c->p2p_seq;
      ua.p2p_peers = c->p2p_peers_dev; ua.p2p_flags_off = c->p2p_flags_off; ua.p2p_count = c->p2p_count;
    }
    aa.M_global = (double)M * W; aa.world = W; aa.verify = 1;
    if (ua.tc_actor_ctas > 0 && want_fuse && ua.grid_loss <= c->sm_count &&
        (c->fused_grid == 0 || c->fused_grid == ua.grid_loss)) {
      c->fused_grid = ua.grid_loss;
      ua.fuse_tail = 1;
      aa.grid_bar = c->grid_bar;
      aa.normpart = c->normpart;
      aa.p2p_err = c->p2p_err;
      if (p2p) {
        aa.ll_peers = c->p2p_peers_dev; aa.ll_local = c->p2p_buf; aa.ll_off = c->ll_off; aa.ll_stride = c->ll_stride;
        aa.timeout_cycles = c->p2p_timeout_cycles;
      }
      ua.adam = aa;
      KernelScope ks(c, CRL_K_LOSS_GRAD);
      CK(launch_loss_grad(ua, c->stream));
      return CRL_OK;
    }
    { KernelScope ks(c, CRL_K_LOSS_GRAD); CK(launch_loss_grad(ua, c->stream)); }
    { KernelScope ks(c, CRL_K_GRAD_REDUCE); CK(launch_grad_reduce(ua, c->L.P, c->stream)); }
    if (multi && !p2p) {
      KernelScope ks(c, CRL_K_ALLREDUCE, false);
      CKN(g_nccl.AllReduce(c->gsum, c->gsum, (size_t)c->L.P + 4 + W, ncclFloat64, ncclSum, c->comm, c->stream));
    }
    if (p2p) {
      aa.p2p_local = reinterpret_cast<const double*>(c->p2p_buf); aa.p2p_seq = c->p2p_seq; aa.p2p_err = c->p2p_err; aa.p2p_stride = c->p2p_stride;
      aa.p2p_flags_off = c->p2p_flags_off; aa.timeout_cycles = c->p2p_timeout_cycles;
    }
    KernelScope ks(c, CRL_K_CLIP_ADAM);
    CK(launch_clip_adam(aa, c->stream));
    return CRL_OK;
  }
  const bool exchange = multi && !local_stats;
  if (exchange) { ua.parts_in = c->parts_recv; ua.n_parts_in = W; ua.world = W; }
  { KernelScope ks(c, CRL_K_MB_STATS); CK(launch_mb_stats(ua, gs, c->stream)); }
  if (exchange) {
    { KernelScope ks(c, CRL_K_OTHER); CK(launch_stats_pack(c->parts, gs, c->parts_send, c->stream)); }
    KernelScope ks(c, CRL_K_ALLREDUCE, false);
    CKN(g_nccl.AllGather(c->parts_send, c->parts_recv, sizeof(MbScalars), ncclChar, c->comm, c->stream));
  }
  { KernelScope ks(c, CRL_K_MB_COUNT); CK(launch_mb_count(ua, c->stream)); }
  if (exchange) {
    KernelScope ks(c, CRL_K_ALLREDUCE, false);
    CKN(g_nccl.AllReduce(&c->fin->cnt, &c->fin->cnt, 1, ncclUint64, ncclSum, c->comm, c->stream));
  }
  { KernelScope ks(c, CRL_K_LOSS_GRAD); CK(launch_loss_grad(ua, c->stream)); }
  { KernelScope ks(c, CRL_K_GRAD_REDUCE); CK(launch_grad_reduce(ua, c->L.P, c->stream)); }
  if (multi) {
    KernelScope ks(c, CRL_K_ALLREDUCE, false);
    CKN(g_nccl.AllReduce(c->gsum, c->gsum, (size_t)c->L.P + 4, ncclFloat64, ncclSum, c->comm, c->stream));
  }
  aa.grad_scale = (multi && local_stats) ? 1.0 / W : 1.0;
  aa.stat_ranks = (multi && local_stats) ? (double)W : 1.0;
  aa.M_global = (double)M * (exchange ? W : 1);
  { KernelScope ks(c, CRL_K_CLIP_ADAM); CK(launch_clip_adam(aa, c->stream)); }
  return CRL_OK;
}

static void stats_to_host(const double* s4, crl_loss_stats* out) {
  out->loss = s4[0]; out->pg_loss = s4[1]; out->v_loss = s4[2]; out->entropy_loss = s4[3];
}

extern "C" CRL_API int crl_update_minibatch(crl_ctx* c, const int32_t* idx, int32_t M, double lr, crl_loss_stats* stats) {
  if (!c || !idx) return fail(CRL_ERR_INVALID, "NULL argument");
  if (!c->gae_done) return fail(CRL_ERR_STATE, "crl_update_minibatch called before crl_gae");
  if (M < 2 || M > c->B) return fail(CRL_ERR_INVALID, "M = %d out of range [2, %d]", M, c->B);
  if (M > c->M) return fail(CRL_ERR_INVALID, "M = %d exceeds the configured minibatch size %d", M, c->M);
  if (!(lr >= 0.0)) return fail(CRL_ERR_INVALID, "lr must be >= 0");
  CKRC(use_device(c));
  SETTLE(c);
  CK(cudaMemcpyAsync(c->idx_dev, idx, 4 * (size_t)M, cudaMemcpyHostToDevice, c->stream));
  CKRC(enqueue_minibatch(c, idx_array(c, c->idx_dev), M, lr, c->stats_dev, 0));
  double s4[4];
  CK(cudaMemcpyAsync(s4, c->stats_dev, sizeof(s4), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (stats) stats_to_host(s4, stats);
  return CRL_OK;
}

static int enqueue_epochs(crl_ctx* c, const int32_t* perm_dev, double lr_host, bool spec = false) {
  int k = 0;
  const int n_sets = c->cfg.update_epochs * c->cfg.num_minibatches;
  const bool a2c = (c->cfg.flags & CRL_FLAG_A2C) != 0;  // the A2C losses use no advantage normalisation
  if (spec && !perm_dev) {
    // throughput path: materialise this update's epoch permutations once (8 MB, L2-resident) instead of
    // re-evaluating the Feistel network per sample in adv_stats and in every loss_grad tile
    KernelScope ks(c, CRL_K_OTHER);
    CK(launch_fill_perms_dev(c->perm_dev, (uint32_t)c->B, c->cfg.seed, c->ds, c->cfg.update_epochs, (uint32_t)c->cfg.rank, c->stream));
    perm_dev = c->perm_dev;
  }
  if (spec && !a2c) CKRC(enqueue_adv_stats(c, perm_dev, c->M, c->cfg.num_minibatches, n_sets));
  if (spec && !a2c && c->cfg.world_size > 1 && !c->p2p_on) {  // global advantage sums for all minibatches of the update: one
                                                               // collective per update (peer memory: adv_stats exchanged them itself)
    KernelScope ks(c, CRL_K_ALLREDUCE, false);
    CKN(g_nccl.AllReduce(c->advparts, c->advparts, (size_t)n_sets * ADV_CHUNKS * 2, ncclFloat64, ncclSum, c->comm, c->stream));
  }
  for (int e = 0; e < c->cfg.update_epochs; e++) {  // ppo.jl:193
    for (int start = 0; start < c->B; start += c->M) {  // ppo.jl:197
      IdxSrc ix = perm_dev ? idx_array(c, perm_dev + (size_t)e * c->B + start) : idx_perm(c, e, start);
      CKRC(enqueue_minibatch(c, ix, c->M, lr_host, c->stats_dev + 4 * (size_t)k, k, spec));
      k++;
    }
  }
  return CRL_OK;
}

extern "C" CRL_API int crl_update_epochs(crl_ctx* c, const int32_t* perms, double lr, crl_loss_stats* stats) {
  if (!c) return fail(CRL_ERR_INVALID, "ctx is NULL");
  if (!c->gae_done) return fail(CRL_ERR_STATE, "crl_update_epochs called before crl_gae");
  if (!(lr >= 0.0)) return fail(CRL_ERR_INVALID, "lr must be >= 0");
  CKRC(use_device(c));
  SETTLE(c);
  const size_t nmb = (size_t)c->cfg.update_epochs * c->cfg.num_minibatches;
  if (perms) CK(cudaMemcpyAsync(c->perm_dev, perms, 4 * (size_t)c->cfg.update_epochs * c->B, cudaMemcpyHostToDevice, c->stream));
  CKRC(enqueue_epochs(c, perms ? c->perm_dev : nullptr, lr));
  {
    KernelScope ks(c, CRL_K_OTHER);
    CK(launch_advance(c->ds, 0ull, 1ull, c->stream));
  }
  std::vector<double> s4(4 * std::max<size_t>(nmb, 1));
  if (nmb) CK(cudaMemcpyAsync(s4.data(), c->stats_dev, nmb * 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (stats) for (size_t i = 0; i < nmb; i++) stats_to_host(&s4[4 * i], stats + i);
  return CRL_OK;
}

extern "C" CRL_API int crl_device_permutation(crl_ctx* c, int64_t update_index, int32_t epoch, int32_t* out) {
  if (!c || !out) return fail(CRL_ERR_INVALID, "NULL argument");
  CKRC(use_device(c));
  {
    KernelScope ks(c, CRL_K_OTHER);
    CK(launch_fill_perm(c->idx_dev, (uint32_t)c->B, c->cfg.seed, (unsigned long long)update_index, (uint32_t)epoch,
                        (uint32_t)c->cfg.rank, c->stream));
  }
  CK(cudaMemcpyAsync(out, c->idx_dev, 4 * (size_t)c->B, cudaMemcpyDeviceToHost, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  return CRL_OK;
}

// the body of one PPO update with device RNG (what the CUDA graph captures)
static int enqueue_train_update(crl_ctx* c, bool spec) {
  CKRC(enqueue_rollout(c, nullptr, nullptr));
  CKRC(enqueue_gae(c));
  CKRC(enqueue_epochs(c, nullptr, -1.0, spec));
  {
    KernelScope ks(c, CRL_K_OTHER);
    CK(launch_advance(c->ds, (unsigned long long)c->T, 1ull, c->stream));
  }
  return CRL_OK;
}

// crl_train_update speculates (see enqueue_minibatch) unless per-shard statistics were requested or CRL_EXACT is set
static bool speculative(const crl_ctx* c) {
  return !(c->cfg.flags & CRL_FLAG_LOCAL_STATS) && getenv("CRL_EXACT") == nullptr && getenv("CRL_MULTI_EXACT") == nullptr;
}

// enqueue one update into result slot `slot`. exact = true forces the non-speculative multi-GPU sequence (replay).
static int run_update(crl_ctx* c, double lr, int slot, bool exact) {
  const bool spec_multi = speculative(c) && !exact;
  if (spec_multi) {
    CKRC(snapshot_alloc(c));
    CKRC(snapshot_copy(c, slot, false));  // state BEFORE the update, for the (rare) exact replay
  }
  c->lr_hist[slot] = lr;
  c->lr_host[slot] = lr;
  CK(cudaMemcpyAsync(&c->ds->lr, c->lr_host + slot, sizeof(double), cudaMemcpyHostToDevice, c->stream));
  const bool use_graph = !exact && !c->profiling && getenv("CRL_NO_GRAPH") == nullptr;
  if (!use_graph) {
    CKRC(enqueue_train_update(c, spec_multi));
  } else {
    if (!c->graph_exec) {
      const uint64_t before = c->launches;
      cudaGraph_t graph = nullptr;
      CK(cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
      int rc = enqueue_train_update(c, spec_multi);
      cudaError_t ee = cudaStreamEndCapture(c->stream, &graph);
      if (rc != CRL_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
      if (ee != cudaSuccess) return fail(CRL_ERR_CUDA, "cudaStreamEndCapture: %s", cudaGetErrorString(ee));
      c->graph_kernels = c->launches - before;
      c->launches = before;
      cudaError_t ie = cudaGraphInstantiate(&c->graph_exec, graph, 0);
      cudaGraphDestroy(graph);
      if (ie != cudaSuccess) { c->graph_exec = nullptr; return fail(CRL_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ie)); }
    }
    CK(cudaGraphLaunch(c->graph_exec, c->stream));
    c->launches += c->graph_kernels;
  }
  // results of this update -> pinned slot; the event lets the host fetch update u-1 while update u is still
  // running (crl_fetch_update_at with lag = 1)
  const size_t nmb = (size_t)c->cfg.update_epochs * c->cfg.num_minibatches;
  static_assert(sizeof(crl_loss_stats) == 4 * sizeof(double), "crl_loss_stats must be 4 doubles");
  if (nmb) CK(cudaMemcpyAsync(c->stats_host[slot], c->stats_dev, nmb * sizeof(crl_loss_stats), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(c->eb_host[slot], c->eb, sizeof(EpisodeBuf), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemcpyAsync(c->flag_host[slot], &c->ds->spec_failed, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  if (c->p2p_on) CK(cudaMemcpyAsync(c->flag_host[slot] + 1, c->p2p_err, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CK(cudaMemsetAsync(&c->ds->spec_failed, 0, sizeof(int), c->stream));
  CK(cudaEventRecord(c->fetch_ev[slot], c->stream));
  return CRL_OK;
}

// Make sure every update with index <= upto is exact. A speculative multi-GPU update whose verification failed
// (identically on every rank) is repaired here: wait for the stream, restore the snapshot taken before that update
// and replay it -- and anything enqueued after it -- with the exact statistics-exchange sequence.
static int validate_updates(crl_ctx* c, uint64_t upto) {
  while (c->validated_seq <= upto && c->validated_seq < c->update_seq) {
    const uint64_t u = c->validated_seq;
    const int slot = (int)(u & 1);
    CK(cudaEventSynchronize(c->fetch_ev[slot]));
    if (speculative(c) && c->flag_host[slot][0]) {
      CK(cudaStreamSynchronize(c->stream));
      c->replays += 1;
      CKRC(snapshot_copy(c, slot, true));
      for (uint64_t r = u; r < c->update_seq; r++) CKRC(run_update(c, c->lr_hist[r & 1], (int)(r & 1), true));
      CK(cudaStreamSynchronize(c->stream));
      c->validated_seq = c->update_seq;
      return CRL_OK;
    }
    c->validated_seq = u + 1;
  }
  return CRL_OK;
}

static int settle(crl_ctx* c) {
  if (c->validated_seq < c->update_seq) return validate_updates(c, c->update_seq - 1);
  return CRL_OK;
}

extern "C" CRL_API int crl_train_update(crl_ctx* c, double lr) {
  if (!c) return fail(CRL_ERR_INVALID, "ctx is NULL");
  if (!(lr >= 0.0)) return fail(CRL_ERR_INVALID, "lr must be >= 0");
  CKRC(use_device(c));
  // the result slot (and snapshot) about to be reused belongs to update seq-2: it must be validated first
  if (c->update_seq >= 2) CKRC(validate_updates(c, c->update_seq - 2));
  CKRC(run_update(c, lr, (int)(c->update_seq & 1), false));
  c->update_seq += 1;
  c->rolled = true;
  c->gae_done = true;
  c->have_update = true;
  return CRL_OK;
}

extern "C" CRL_API int crl_fetch_update_at(crl_ctx* c, int32_t lag, crl_loss_stats* stats, crl_episode_agg* agg) {
  if (!c) return fail(CRL_ERR_INVALID, "ctx is NULL");
  if (lag < 0 || lag > 1) return fail(CRL_ERR_INVALID, "lag must be 0 (latest update) or 1 (the one before)");
  if (!c->have_update || c->update_seq < (uint64_t)lag + 1) return fail(CRL_ERR_STATE, "no such update has been enqueued yet");
  CKRC(use_device(c));
  const uint64_t target = c->update_seq - 1 - (uint64_t)lag;
  CKRC(validate_updates(c, target));
  if (c->p2p_on && (c->flag_host[0][1] || c->flag_host[1][1]))
    return fail(CRL_ERR_NCCL, "peer-memory allreduce timed out waiting for another rank");
  const int slot = (int)(target & 1);
  CK(cudaEventSynchronize(c->fetch_ev[slot]));
  const size_t nmb = (size_t)c->cfg.update_epochs * c->cfg.num_minibatches;
  if (stats && nmb) memcpy(stats, c->stats_host[slot], nmb * sizeof(crl_loss_stats));
  if (agg) {
    const EpisodeBuf& e = *c->eb_host[slot];
    agg->count = (int64_t)e.n_episodes; agg->sum_return = e.sum_return; agg->sum_length = e.sum_length;
    agg->max_return = e.max_return;
    agg->dropped = e.count > (unsigned)c->ep_capacity ? (int64_t)(e.count - c->ep_capacity) : 0;
  }
  return CRL_OK;
}

extern "C" CRL_API int crl_fetch_update(crl_ctx* c, crl_loss_stats* stats, crl_episode_agg* agg) {
  return crl_fetch_update_at(c, 0, stats, agg);
}

// ------------------------------------------------------------------ data access
static int field_info(crl_ctx* c, int f, void** p, size_t* bytes) {
  const Layout& L = c->L;
  const size_t N = c->N, B = c->B;
  switch (f) {
    case CRL_F_STATE: *p = c->state; *bytes = B * L.D * 4; break;
    case CRL_F_ACTION: *p = c->action; *bytes = B * (L.continuous ? L.A : 1) * 4; break;
    case CRL_F_LOGPROB: *p = c->logprob; *bytes = B * 4; break;
    case CRL_F_REWARD: *p = c->reward; *bytes = B * 4; break;
    case CRL_F_TERMINAL: *p = c->terminal; *bytes = B; break;
    case CRL_F_VALUE: *p = c->value; *bytes = B * 4; break;
    case CRL_F_ADVANTAGE: *p = c->advantage; *bytes = B * 4; break;
    case CRL_F_RETURN: *p = c->ret; *bytes = B * 4; break;
    case CRL_F_NEXT_OBS: *p = c->next_obs; *bytes = N * L.D * 4; break;
    case CRL_F_NEXT_DONE: *p = c->next_done; *bytes = N; break;
    case CRL_F_NEXT_VALUE: *p = c->next_value; *bytes = N * 4; break;
    case CRL_F_ENV_STATE: *p = c->env_state; *bytes = N * L.S * 4; break;
    case CRL_F_ENV_T: *p = c->env_t; *bytes = N * 4; break;
    case CRL_F_EP_RETURN: *p = c->ep_return; *bytes = N * 8; break;
    case CRL_F_EP_LENGTH: *p = c->ep_length; *bytes = N * 4; break;
    case CRL_F_RESET_COUNT: *p = c->reset_count; *bytes = N * 4; break;
    case CRL_F_VNEW: *p = c->vnew; *bytes = (size_t)c->M * 4; break;
    default: return fail(CRL_ERR_INVALID, "unknown field %d", f);
  }
  return CRL_OK;
}
extern "C" CRL_API int crl_read_field(crl_ctx* c, int32_t field, void* host, size_t bytes) {
  if (!c || !host) return fail(CRL_ERR_INVALID, "NULL argument");
  void* p; size_t nb;
  CKRC(field_info(c, field, &p, &nb));
  if (bytes != nb) return fail(CRL_ERR_INVALID, "field %d holds %zu bytes, caller passed %zu", field, nb, bytes);
  CKRC(use_device(c));
  SETTLE(c);
  return copy_vec(c, host, p, nb, cudaMemcpyDeviceToHost);
}
extern "C" CRL_API int crl_write_field(crl_ctx* c, int32_t field, const void* host, size_t bytes) {
  if (!c || !host) return fail(CRL_ERR_INVALID, "NULL argument");
  void* p; size_t nb;
  CKRC(field_info(c, field, &p, &nb));
  if (bytes != nb) return fail(CRL_ERR_INVALID, "field %d holds %zu bytes, caller passed %zu", field, nb, bytes);
  CKRC(use_device(c));
  SETTLE(c);
  CKRC(copy_vec(c, p, host, nb, cudaMemcpyHostToDevice));
  if (field <= CRL_F_VALUE) c->rolled = true;
  if (field == CRL_F_ADVANTAGE || field == CRL_F_RETURN) c->gae_done = true;
  return CRL_OK;
}

extern "C" CRL_API int crl_pop_episodes(crl_ctx* c, crl_episode* out, int32_t max_records, int32_t* n_out, crl_episode_agg* agg) {
  if (!c) return fail(CRL_ERR_INVALID, "ctx is NULL");
  CKRC(use_device(c));
  SETTLE(c);
  EpisodeBuf e;
  CKRC(copy_vec(c, &e, c->eb, sizeof(e), cudaMemcpyDeviceToHost));
  const int have = (int)std::min<unsigned>(e.count, (unsigned)c->ep_capacity);
  std::vector<crl_episode> recs(std::max(have, 1));
  if (have) CKRC(copy_vec(c, recs.data(), c->records, (size_t)have * sizeof(crl_episode), cudaMemcpyDeviceToHost));
  recs.resize(have);
  // the reference logs in (step, env) order, ppo.jl:149 (Q11)
  std::sort(recs.begin(), recs.end(), [](const crl_episode& x, const crl_episode& y) {
    return x.step != y.step ? x.step < y.step : x.env < y.env;
  });
  int n = 0;
  if (out) { n = std::min(have, (int)std::max(0, max_records)); memcpy(out, recs.data(), (size_t)n * sizeof(crl_episode)); }
  if (n_out) *n_out = n;
  if (agg) {
    agg->count = (int64_t)e.n_episodes; agg->sum_return = e.sum_return; agg->sum_length = e.sum_length;
    agg->max_return = e.max_return;
    agg->dropped = (int64_t)e.count - (int64_t)n;
  }
  return CRL_OK;
}

// ------------------------------------------------------------------ multi-GPU
extern "C" CRL_API int crl_comm_unique_id(void* out128) {
  if (!out128) return fail(CRL_ERR_INVALID, "out128 is NULL");
  CKRC(nccl_load());
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is expected to be 128 bytes");
  ncclUniqueId id;
  CKN(g_nccl.GetUniqueId(&id));
  memcpy(out128, &id, sizeof(id));
  return CRL_OK;
}
extern "C" CRL_API int crl_comm_init(crl_ctx* c, const void* id128) {
  if (!c || !id128) return fail(CRL_ERR_INVALID, "NULL argument");
  if (c->cfg.world_size < 2) return fail(CRL_ERR_INVALID, "crl_comm_init needs world_size >= 2");
  CKRC(nccl_load());
  CKRC(use_device(c));
  ncclUniqueId id;
  memcpy(&id, id128, sizeof(id));
  CKN(g_nccl.CommInitRank(&c->comm, c->cfg.world_size, id, c->cfg.rank));
  // NCCL connects its channels lazily on the first collective: do that here (set-up time), not inside the first update
  CK(cudaMemsetAsync(c->gsum, 0, sizeof(double) * 8, c->stream));
  CKN(g_nccl.AllReduce(c->gsum, c->gsum, 8, ncclFloat64, ncclSum, c->comm, c->stream));
  CKN(g_nccl.AllGather(c->parts_send, c->parts_recv, sizeof(MbScalars), ncclChar, c->comm, c->stream));
  CK(cudaStreamSynchronize(c->stream));
  if (getenv("CRL_NO_P2P") == nullptr) {
    // peer-memory exchange buffers: every rank exports its buffer with cudaIpc, the handles travel through one
    // NCCL all-gather, and each rank maps all peers (NVLink P2P). Any failure leaves the NCCL path in place.
    const int W = c->cfg.world_size;
    c->p2p_stride = (c->L.P + 4 + CRL_MAX_WORLD + 1) & ~1;
    c->p2p_flags_off = (size_t)2 * W * c->p2p_stride * sizeof(double);   // [2 slots][W ranks][stride] doubles, then the flags
    // behind them: the flag-in-data region of the fused tail, 16-byte packets {lo, seq, hi, seq} (gradient, 4 loss sums, min)
    c->ll_stride = (c->L.P + 4 + 1 + 7) & ~7;
    c->ll_off = (c->p2p_flags_off + CRL_MAX_WORLD * sizeof(unsigned long long) + 255) & ~size_t(255);
    c->adv_stride = std::max(1, c->cfg.update_epochs) * c->cfg.num_minibatches * ADV_CHUNKS * 2;
    c->adv_off = c->ll_off + (size_t)2 * W * c->ll_stride * 16;
    const size_t bytes = c->adv_off + (size_t)2 * W * c->adv_stride * 16;
    {
      // how long a kernel waits for a peer's data before it gives up (error, no update applied): a peer may legitimately
      // be seconds late (first CUDA-graph instantiation, a host stall on the rank that logs). CRL_P2P_TIMEOUT_MS overrides.
      const char* e = getenv("CRL_P2P_TIMEOUT_MS");
      const double ms = e ? atof(e) : 30000.0;
      int khz = 1965000;
      cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, c->cfg.device);
      c->p2p_timeout_cycles = (long long)(ms * (double)khz);
    }
    bool ok = cudaMalloc(reinterpret_cast<void**>(&c->p2p_buf), bytes) == cudaSuccess &&
              cudaMemset(c->p2p_buf, 0, bytes) == cudaSuccess;
    cudaIpcMemHandle_t mine;
    ok = ok && cudaIpcGetMemHandle(&mine, c->p2p_buf) == cudaSuccess;
    unsigned char* stage = nullptr;
    ok = ok && cudaMalloc(reinterpret_cast<void**>(&stage), (size_t)(W + 1) * sizeof(mine)) == cudaSuccess;
    std::vector<cudaIpcMemHandle_t> all(W);
    if (ok) {
      ok = cudaMemcpy(stage, &mine, sizeof(mine), cudaMemcpyHostToDevice) == cudaSuccess;
      ok = ok && g_nccl.AllGather(stage, stage + sizeof(mine), sizeof(mine), ncclChar, c->comm, c->stream) == ncclSuccess;
      ok = ok && cudaStreamSynchronize(c->stream) == cudaSuccess;
      ok = ok && cudaMemcpy(all.data(), stage + sizeof(mine), (size_t)W * sizeof(mine), cudaMemcpyDeviceToHost) == cudaSuccess;
    }
    if (stage) cudaFree(stage);
    for (int r = 0; r < W && ok; r++) {
      if (r == c->cfg.rank) { c->p2p_peer[r] = c->p2p_buf; continue; }
      void* ptr = nullptr;
      ok = cudaIpcOpenMemHandle(&ptr, all[r], cudaIpcMemLazyEnablePeerAccess) == cudaSuccess;
      c->p2p_peer[r] = static_cast<unsigned char*>(ptr);
    }
    ok = ok && cudaMalloc(reinterpret_cast<void**>(&c->p2p_peers_dev), CRL_MAX_WORLD * sizeof(void*)) == cudaSuccess;
    ok = ok && cudaMemcpy(c->p2p_peers_dev, c->p2p_peer, CRL_MAX_WORLD * sizeof(void*), cudaMemcpyHostToDevice) == cudaSuccess;
    ok = ok && dalloc(&c->p2p_seq, 1) == CRL_OK && dalloc(&c->p2p_err, 1) == CRL_OK && dalloc(&c->p2p_count, 1) == CRL_OK;
    // all ranks must agree on using the peer path: one more collective carries the verdict
    double verdict = ok ? 1.0 : 0.0;
    CK(cudaMemcpy(c->gsum, &verdict, sizeof(double), cudaMemcpyHostToDevice));
    CKN(g_nccl.AllReduce(c->gsum, c->gsum, 1, ncclFloat64, ncclSum, c->comm, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaMemcpy(&verdict, c->gsum, sizeof(double), cudaMemcpyDeviceToHost));
    cudaGetLastError();  // clear any sticky-free error from a failed IPC attempt
    c->p2p_on = verdict > W - 0.5;
  }
  return CRL_OK;
}

// ------------------------------------------------------------------ instrumentation
extern "C" CRL_API int crl_kernel_launches(const crl_ctx* c, uint64_t* count) {
  if (!c || !count) return fail(CRL_ERR_INVALID, "NULL argument");
  *count = c->launches;
  return CRL_OK;
}
extern "C" CRL_API int crl_spec_replays(const crl_ctx* c, uint64_t* count) {
  if (!c || !count) return fail(CRL_ERR_INVALID, "NULL argument");
  *count = c->replays;
  return CRL_OK;
}
extern "C" CRL_API int crl_profile(crl_ctx* c, int32_t enable) {
  if (!c) return fail(CRL_ERR_INVALID, "ctx is NULL");
  CKRC(use_device(c));
  CK(cudaStreamSynchronize(c->stream));
  prof_collect(c);
  c->profiling = enable != 0;
  return CRL_OK;
}
extern "C" CRL_API int crl_profile_read(crl_ctx* c, crl_kernel_times* out, int32_t reset) {
  if (!c || !out) return fail(CRL_ERR_INVALID, "NULL argument");
  CKRC(use_device(c));
  CK(cudaStreamSynchronize(c->stream));
  prof_collect(c);
  *out = c->times;
  if (reset) memset(&c->times, 0, sizeof(c->times));
  return CRL_OK;
}
extern "C" CRL_API int crl_stream(const crl_ctx* c, void** cuda_stream) {
  if (!c || !cuda_stream) return fail(CRL_ERR_INVALID, "NULL argument");
  *cuda_stream = c->stream;
  return CRL_OK;
}

// ------------------------------------------------------------------ raw entry points
static int need_sm100() {
  static int inited_dev = -1;
  int dev = 0;
  CK(cudaGetDevice(&dev));
  if (inited_dev == dev) return CRL_OK;
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, dev));
  if (prop.major != 10) return fail(CRL_ERR_CUDA, "current device is sm_%d%d; sm_100 required", prop.major, prop.minor);
  CK(kernels_init_rollout());
  CK(kernels_init_update());
  inited_dev = dev;
  return CRL_OK;
}

extern "C" CRL_API int crl_gae_raw(const float* values, const float* rewards, const uint8_t* dones, const float* next_value,
                           const uint8_t* next_done, float* adv, float* ret, int32_t T, int64_t N, float gamma,
                           float lambda, int32_t mode, void* stream) {
  if (!values || !rewards || !dones || !adv || !ret) return fail(CRL_ERR_INVALID, "NULL argument");
  if (T < 1 || N < 0) return fail(CRL_ERR_INVALID, "T must be >= 1 and N >= 0");
  if (mode != CRL_GAE_REF_COMPAT && mode != CRL_GAE_FIXED && mode != CRL_GAE_A2C_RETURNS) return fail(CRL_ERR_INVALID, "bad gae mode");
  if (mode != CRL_GAE_REF_COMPAT && (!next_value || !next_done)) return fail(CRL_ERR_INVALID, "FIXED / A2C modes need the bootstrap arrays");
  CK(launch_gae(values, rewards, dones, next_value, next_done, adv, ret, T, N, gamma, lambda, mode, (cudaStream_t)stream));
  return CRL_OK;
}

extern "C" CRL_API int crl_env_step_raw(int32_t env_kind, float* state, int32_t* t, const void* action, float* reward,
                                uint8_t* done, int64_t n, int32_t max_episode_steps, void* stream) {
  if (env_kind != CRL_ENV_CARTPOLE && env_kind != CRL_ENV_PENDULUM) return fail(CRL_ERR_INVALID, "unknown env_kind");
  if (n < 0 || (n > 0 && (!state || !t || !action || !reward || !done))) return fail(CRL_ERR_INVALID, "NULL argument");
  CK(launch_env_step_raw(env_kind, state, t, action, reward, done, n, max_episode_steps, (cudaStream_t)stream));
  return CRL_OK;
}

extern "C" CRL_API int crl_policy_forward_raw(int32_t env_kind, const float* params, const float* obs, float* out_policy,
                                      float* logp, float* value, int64_t n, void* stream) {
  if (env_kind != CRL_ENV_CARTPOLE && env_kind != CRL_ENV_PENDULUM) return fail(CRL_ERR_INVALID, "unknown env_kind");
  if (n < 0 || (n > 0 && (!params || !obs || !out_policy || !value))) return fail(CRL_ERR_INVALID, "NULL argument");
  if (env_kind == CRL_ENV_CARTPOLE && n > 0 && !logp) return fail(CRL_ERR_INVALID, "logp is NULL");
  CKRC(need_sm100());
  CK(launch_policy_forward_raw(env_kind, params, obs, out_policy, logp, value, n, (cudaStream_t)stream));
  return CRL_OK;
}

// scratch for the raw loss entry point (per process, grown on demand)
struct RawScratch {
  int device = -1, M = 0, sm = 0;
  float* vnew = nullptr;
  MbScalars* parts = nullptr;
  MbFinal* fin = nullptr;
  float *gpart = nullptr, *mpart = nullptr;
  double *spart = nullptr, *gsum = nullptr, *advparts = nullptr;
  DevState* ds = nullptr;
};
static RawScratch g_raw;

extern "C" CRL_API int crl_ppo_loss_raw(int32_t env_kind, const float* params, const int32_t* idx, int32_t M,
                                const float* states, const void* actions, const float* logprobs,
                                const float* advantages, const float* returns, const float* values, float clip_coef,
                                float ent_coeff, float v_coef, float* grads_out, double* stats_out, void* stream) {
  Layout L;
  if (!make_layout(env_kind, &L)) return fail(CRL_ERR_INVALID, "unknown env_kind");
  if (!params || !idx || !states || !actions || !logprobs || !advantages || !returns || !values || !grads_out)
    return fail(CRL_ERR_INVALID, "NULL argument");
  if (M < 2) return fail(CRL_ERR_INVALID, "M must be >= 2");
  CKRC(need_sm100());
  int dev = 0;
  CK(cudaGetDevice(&dev));
  cudaStream_t s = (cudaStream_t)stream;
  if (g_raw.device != dev || g_raw.M < M) {
    CK(cudaDeviceSynchronize());
    void* old[] = {g_raw.vnew, g_raw.parts, g_raw.fin, g_raw.gpart, g_raw.spart, g_raw.gsum, g_raw.ds, g_raw.mpart, g_raw.advparts};
    for (void* p : old) if (p) cudaFree(p);
    g_raw = RawScratch();
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, dev));
    g_raw.sm = prop.multiProcessorCount;
    CKRC(dalloc(&g_raw.vnew, M)); CKRC(dalloc(&g_raw.parts, g_raw.sm)); CKRC(dalloc(&g_raw.fin, 1));
    CKRC(dalloc(&g_raw.gpart, (size_t)g_raw.sm * CRL_H * (CRL_H + 16) * 2)); CKRC(dalloc(&g_raw.spart, (size_t)g_raw.sm * 4));
    CKRC(dalloc(&g_raw.gsum, (size_t)CRL_H * (CRL_H + 16) * 2)); CKRC(dalloc(&g_raw.ds, 1));
    CKRC(dalloc(&g_raw.mpart, g_raw.sm)); CKRC(dalloc(&g_raw.advparts, ADV_CHUNKS * 2));
    g_raw.device = dev; g_raw.M = M;
  }
  UpdateArgs ua;
  memset(&ua, 0, sizeof(ua));  // every optional path (peer exchange, tcgen05 split) off unless set below
  ua.env_kind = env_kind; ua.algo = 0; ua.params = params; ua.image = nullptr; ua.M = M;
  ua.idx.arr = idx; ua.idx.start = 0; ua.idx.B = (uint32_t)M; ua.idx.half_bits = 1; ua.idx.epoch = 0; ua.idx.rank = 0;
  ua.idx.seed = 0; ua.idx.ds = g_raw.ds;
  ua.states = states; ua.actions = actions; ua.logprobs = logprobs; ua.advantages = advantages; ua.returns = returns;
  ua.values = values; ua.clip_coef = clip_coef; ua.ent_coeff = ent_coeff; ua.v_coef = v_coef;
  ua.vnew = g_raw.vnew; ua.parts = g_raw.parts; ua.n_parts_cap = g_raw.sm;
  const int gs = mb_stats_grid(M, g_raw.sm);
  ua.parts_in = g_raw.parts; ua.n_parts_in = gs; ua.fin = g_raw.fin; ua.world = 1;
  ua.gpart = g_raw.gpart; ua.spart = g_raw.spart; ua.grid_loss = loss_grad_grid(M, g_raw.sm); ua.gsum = g_raw.gsum;
  ua.advparts = g_raw.advparts; ua.mpart = g_raw.mpart;
  ua.mode = LG_EXACT;
  CK(launch_mb_stats(ua, gs, s));
  CK(launch_mb_count(ua, s));
  CK(launch_loss_grad(ua, s));
  CK(launch_grad_reduce(ua, L.P, s));
  CK(launch_loss_finalize(g_raw.gsum, L.P, grads_out, (double)M, L.A, ent_coeff, v_coef, stats_out, s));
  return CRL_OK;
}

extern "C" CRL_API int crl_clip_adam_raw(int32_t env_kind, float* params, const float* grads, float* m, float* v,
                                 double* beta_pow, double lr, float clip_norm, void* stream) {
  Layout L;
  if (!make_layout(env_kind, &L)) return fail(CRL_ERR_INVALID, "unknown env_kind");
  if (!params || !grads || !m || !v || !beta_pow) return fail(CRL_ERR_INVALID, "NULL argument");
  if (!(lr >= 0.0)) return fail(CRL_ERR_INVALID, "lr must be >= 0");
  CKRC(need_sm100());
  AdamArgs aa;
  memset(&aa, 0, sizeof(aa));
  aa.world = 1;
  aa.env_kind = env_kind; aa.params = params; aa.image = nullptr; aa.gsum = nullptr; aa.gf = grads; aa.grad_scale = 1.0; aa.stat_ranks = 1.0;
  aa.grads_out = nullptr; aa.m = m; aa.v = v; aa.beta_pow = beta_pow; aa.ds = nullptr; aa.lr_host = lr;
  aa.clip_norm = clip_norm; aa.ent_coeff = 0.f; aa.v_coef = 0.f; aa.M_global = 1.0; aa.A = L.A; aa.stats_out = nullptr;
  CK(launch_clip_adam(aa, (cudaStream_t)stream));
  return CRL_OK;
}
