// C ABI (include/mrl_b200.h): host-side orchestration of the kernels.
#include "common.cuh"
#include "kernels.h"
#include "../../include/mrl_b200.h"
#include "comm.h"

#include <atomic>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>

static thread_local std::string g_err;
static std::atomic<long long> g_launches{0};
// Batch contents are identified by a process-wide version number: a freed batch whose address is reused can never
// match a net's activation cache (the cache key is (batch pointer, version, parameter version)).
static std::atomic<unsigned long long> g_batch_version{1};

static int fail(const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_err = buf;
  return 1;
}
#define CK(call)                                                                            \
  do {                                                                                      \
    cudaError_t _e = (call);                                                                \
    if (_e != cudaSuccess) return fail("%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e)); \
  } while (0)
#define CKL(call, nk) \
  do {                \
    CK(call);         \
    g_launches += nk; \
  } while (0)
#define RET(call)          \
  do {                     \
    int _r = (call);       \
    if (_r) return _r;     \
  } while (0)

// ---- optional per-kernel-class timing with CUDA events on the launching stream (bench.py's roofline)
enum { PK_L1F = 0, PK_MIDF, PK_MIDB_GRAD, PK_MIDB_FVP, PK_L1G, PK_REDUCE, PK_CG, PK_GAE, PK_PACK, PK_ROLLOUT,
       PK_CEM_SEARCH, PK_COUNT };
static const char* kPkNames[PK_COUNT] = {"l1_forward", "mid_forward", "mid_backward_grad", "mid_backward_fvp",
                                         "l1_grad",    "reduce",      "cg_vector",         "gae",
                                         "pack_params", "rollout",    "cem_search"};
struct Prof {
  bool on = false;
  std::vector<cudaEvent_t> pool;
  size_t used = 0;
  std::vector<int> kinds;
  double ms[PK_COUNT] = {0};
  long long cnt[PK_COUNT] = {0};
};
static Prof g_prof;
static void prof_mark(int kind, cudaStream_t st, bool begin) {
  if (!g_prof.on) return;
  if (g_prof.used == g_prof.pool.size()) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    g_prof.pool.push_back(e);
  }
  cudaEventRecord(g_prof.pool[g_prof.used++], st);
  if (begin) g_prof.kinds.push_back(kind);
}
#define CKP(kind, call, nk)          \
  do {                               \
    prof_mark(kind, st, true);       \
    CKL(call, nk);                   \
    prof_mark(kind, st, false);      \
  } while (0)

extern "C" int mrl_profile_enable(int on) {
  g_prof.on = on != 0;
  g_prof.used = 0;
  g_prof.kinds.clear();
  for (int k = 0; k < PK_COUNT; ++k) { g_prof.ms[k] = 0; g_prof.cnt[k] = 0; }
  return 0;
}
extern "C" int mrl_profile_kinds(void) { return PK_COUNT; }
extern "C" const char* mrl_profile_kind_name(int k) { return (k >= 0 && k < PK_COUNT) ? kPkNames[k] : ""; }
// Synchronises the device, folds all recorded intervals into the per-kind totals and returns them.
extern "C" int mrl_profile_read(double* ms_out, long long* count_out) {
  cudaError_t e = cudaDeviceSynchronize();
  if (e != cudaSuccess) { g_err = cudaGetErrorString(e); return 1; }
  for (size_t i = 0; i < g_prof.kinds.size(); ++i) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, g_prof.pool[2 * i], g_prof.pool[2 * i + 1]);
    g_prof.ms[g_prof.kinds[i]] += ms;
    g_prof.cnt[g_prof.kinds[i]] += 1;
  }
  g_prof.used = 0;
  g_prof.kinds.clear();
  for (int k = 0; k < PK_COUNT; ++k) { ms_out[k] = g_prof.ms[k]; count_out[k] = g_prof.cnt[k]; }
  return 0;
}

extern "C" const char* mrl_last_error(void) { return g_err.c_str(); }
int mrl_set_error(const char* msg) { g_err = msg; return 1; }   // used by comm.cu
extern "C" int mrl_version(void) { return 100; }
extern "C" long long mrl_launch_count(void) { return g_launches.load(); }

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = bytes + bytes / 8 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <typename T>
  T* as() const { return reinterpret_cast<T*>(p); }
};

static size_t dtype_size(int dt) { return (dt == MRL_F32 || dt == MRL_I32) ? 4 : 8; }

// ======================================================================== batch
struct mrl_batch {
  int device = 0, ob_dim = 0, with_time = 0, xdim = 0, d0p = 0;
  long long N = 0, Nglobal = 0;
  int n_tiles = 0, n_paths = 0;
  double timestep_limit = 1.0;
  unsigned long long version = 0;
  int pol_head = -1, pol_dout = 0, naux_pol = 0;
  bool has_baseline = false, has_adv32 = false, has_ret = false;
  DevBuf XG, XA, aux_pol, aux_vf, offsets, terminated, tindex, stage, stage2, baseline, ret, adv, adv32, stats,
      gather;
};

static int stage_in(DevBuf& stage, const void* src, size_t bytes, int loc, cudaStream_t st, const void** out) {
  if (loc == MRL_DEVICE) {
    *out = src;
    return 0;
  }
  CK(stage.reserve(bytes));
  CK(cudaMemcpyAsync(stage.p, src, bytes, cudaMemcpyHostToDevice, st));
  *out = stage.p;
  return 0;
}

extern "C" int mrl_batch_create(mrl_batch** out, int device, int ob_dim, int with_time_feature) {
  if (!out || ob_dim <= 0) return fail("mrl_batch_create: bad arguments");
  CK(cudaSetDevice(device));
  mrl_batch* b = new mrl_batch();
  b->device = device;
  b->ob_dim = ob_dim;
  b->with_time = with_time_feature ? 1 : 0;
  b->xdim = ob_dim + b->with_time;
  b->d0p = round_up(b->xdim, 8);
  b->version = g_batch_version.fetch_add(1);
  *out = b;
  return 0;
}
extern "C" int mrl_batch_destroy(mrl_batch* b) {
  if (!b) return 0;
  cudaSetDevice(b->device);
  DevBuf* bufs[] = {&b->XG, &b->XA, &b->aux_pol, &b->aux_vf, &b->offsets, &b->terminated, &b->tindex, &b->stage,
                    &b->stage2, &b->baseline, &b->ret, &b->adv, &b->adv32, &b->stats, &b->gather};
  for (DevBuf* d : bufs) d->release();
  delete b;
  return 0;
}
extern "C" long long mrl_batch_size(const mrl_batch* b) { return b ? b->N : -1; }
extern "C" int mrl_batch_set_global_n(mrl_batch* b, long long n) {
  if (!b || n < b->N) return fail("mrl_batch_set_global_n: n_global < local N");
  b->Nglobal = n;
  return 0;
}

extern "C" int mrl_batch_set_obs(mrl_batch* b, const void* ob, int dtype, long long ld, long long N, int loc,
                                 void* stream) {
  if (!b || !ob || N <= 0) return fail("mrl_batch_set_obs: bad arguments");
  if (dtype != MRL_F32 && dtype != MRL_F64) return fail("mrl_batch_set_obs: observations must be f32 or f64");
  if (ld < b->ob_dim) return fail("mrl_batch_set_obs: ld < ob_dim");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(b->device));
  b->N = N;
  b->Nglobal = N;
  b->n_tiles = (int)((N + MRL_TILE - 1) / MRL_TILE);
  b->version = g_batch_version.fetch_add(1);
  b->has_baseline = b->has_adv32 = b->has_ret = false;
  b->pol_head = -1;
  const void* src;
  RET(stage_in(b->stage, ob, (size_t)N * ld * dtype_size(dtype), loc, st, &src));
  const long long n_mtiles = (b->n_tiles + 1) / 2;
  CK(b->XA.reserve(l1tc_xa_floats(b->d0p / 8, n_mtiles) * 4));
  CKL(launch_pack_xa(src, dtype, ld, b->ob_dim, N, b->XA.as<float>(), b->d0p / 8, n_mtiles, st), 1);
  const int xg_ftiles = (b->xdim + 127) / 128;
  CK(b->XG.reserve(l1tc_xg_floats(xg_ftiles, b->n_tiles) * 4));
  CKL(launch_pack_xg(src, dtype, ld, b->ob_dim, N, b->XG.as<float>(), xg_ftiles, b->n_tiles, st), 1);
  return 0;
}

extern "C" int mrl_batch_set_paths(mrl_batch* b, const long long* offsets, const unsigned char* terminated,
                                   int n_paths, double timestep_limit, int loc, void* stream) {
  if (!b || !offsets || !terminated || n_paths <= 0) return fail("mrl_batch_set_paths: bad arguments");
  if (b->N <= 0) return fail("mrl_batch_set_paths: set observations first");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(b->device));
  CK(b->offsets.reserve((size_t)(n_paths + 1) * 8));
  CK(b->terminated.reserve((size_t)n_paths));
  cudaMemcpyKind kind = loc == MRL_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
  if (loc == MRL_HOST) {
    if (offsets[0] != 0 || offsets[n_paths] != b->N)
      return fail("mrl_batch_set_paths: offsets must start at 0 and end at N=%lld", b->N);
    for (int p = 0; p < n_paths; ++p)
      if (offsets[p + 1] < offsets[p]) return fail("mrl_batch_set_paths: offsets not monotone at path %d", p);
  }
  CK(cudaMemcpyAsync(b->offsets.p, offsets, (size_t)(n_paths + 1) * 8, kind, st));
  CK(cudaMemcpyAsync(b->terminated.p, terminated, (size_t)n_paths, kind, st));
  b->n_paths = n_paths;
  b->timestep_limit = timestep_limit;
  CK(b->tindex.reserve((size_t)b->N * 4));
  if (b->with_time) {
    if (!(timestep_limit > 0)) return fail("mrl_batch_set_paths: timestep_limit must be > 0");
    CKL(launch_time_feature(b->offsets.as<long long>(), n_paths, b->N, timestep_limit, b->ob_dim, b->tindex.as<int>(),
                            b->XA.as<float>(), b->d0p / 8, b->XG.as<float>(), (b->xdim + 127) / 128, st), 1);
  }
  return 0;
}

extern "C" int mrl_batch_get_time_index(mrl_batch* b, int* out, int loc, void* stream) {
  if (!b || !out || !b->with_time || b->n_paths <= 0) return fail("mrl_batch_get_time_index: no paths bound");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaMemcpyAsync(out, b->tindex.p, (size_t)b->N * 4, loc == MRL_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
  if (loc == MRL_HOST) CK(cudaStreamSynchronize(st));
  return 0;
}

extern "C" int mrl_batch_set_policy_inputs(mrl_batch* b, int head, int dout, const void* act, int act_dtype,
                                           const void* adv, int adv_dtype, const void* oldprob, int oldprob_dtype,
                                           int loc, void* stream) {
  if (!b || !act || !oldprob || b->N <= 0) return fail("mrl_batch_set_policy_inputs: bad arguments");
  if (head != MRL_GAUSS && head != MRL_CATEGORICAL) return fail("mrl_batch_set_policy_inputs: bad head");
  if (oldprob_dtype != MRL_F32 && oldprob_dtype != MRL_F64) return fail("oldprob must be f32/f64");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(b->device));
  const long long N = b->N;
  const int naux = head == MRL_GAUSS ? 1 + 3 * dout : 2 + dout;
  CK(b->aux_pol.reserve((size_t)b->n_tiles * naux * MRL_LDT * 4));
  float* aux = b->aux_pol.as<float>();
  const void* src;
  if (adv) {
    RET(stage_in(b->stage2, adv, (size_t)N * dtype_size(adv_dtype), loc, st, &src));
    CKL(launch_pack_tiles(src, adv_dtype, 1, 1, 1, N, aux, naux, 0, b->n_tiles, st), 1);
  } else {
    if (!b->has_adv32) return fail("mrl_batch_set_policy_inputs: adv == NULL but no advantages on the device");
    CKL(launch_pack_tiles(b->adv32.p, MRL_F32, 1, 1, 1, N, aux, naux, 0, b->n_tiles, st), 1);
  }
  const int acols = head == MRL_GAUSS ? dout : 1;
  if (head == MRL_GAUSS && act_dtype != MRL_F32 && act_dtype != MRL_F64) return fail("DiagGauss actions must be float");
  RET(stage_in(b->stage2, act, (size_t)N * acols * dtype_size(act_dtype), loc, st, &src));
  CKL(launch_pack_tiles(src, act_dtype, acols, acols, acols, N, aux, naux, 1, b->n_tiles, st), 1);
  const int pcols = head == MRL_GAUSS ? 2 * dout : dout;
  RET(stage_in(b->stage2, oldprob, (size_t)N * pcols * dtype_size(oldprob_dtype), loc, st, &src));
  CKL(launch_pack_tiles(src, oldprob_dtype, pcols, pcols, pcols, N, aux, naux, 1 + acols, b->n_tiles, st), 1);
  b->pol_head = head;
  b->pol_dout = dout;
  b->naux_pol = naux;
  return 0;
}

// dst <- rows idx[0..n) of src (observations in both tensor-core layouts + the policy side inputs), on the device
extern "C" int mrl_batch_gather(mrl_batch* dst, const mrl_batch* src, const int* idx, int n, int loc, void* stream) {
  if (!dst || !src || !idx || n <= 0) return fail("mrl_batch_gather: bad arguments");
  if (dst == src) return fail("mrl_batch_gather: dst and src must differ");
  if (src->N <= 0 || src->pol_head < 0) return fail("mrl_batch_gather: bind observations and policy inputs of the source first");
  if (dst->device != src->device || dst->ob_dim != src->ob_dim || dst->with_time != src->with_time)
    return fail("mrl_batch_gather: batches differ in device / shape");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(dst->device));
  const int* idx_dev = idx;
  if (loc == MRL_HOST) {
    CK(dst->stage2.reserve((size_t)n * 4));
    CK(cudaMemcpyAsync(dst->stage2.p, idx, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    idx_dev = dst->stage2.as<int>();
  }
  dst->N = n;
  dst->Nglobal = n;
  dst->n_tiles = (n + MRL_TILE - 1) / MRL_TILE;
  dst->version = g_batch_version.fetch_add(1);
  dst->has_baseline = dst->has_adv32 = dst->has_ret = false;
  dst->n_paths = 0;
  dst->pol_head = src->pol_head;
  dst->pol_dout = src->pol_dout;
  dst->naux_pol = src->naux_pol;
  const long long n_mtiles = (dst->n_tiles + 1) / 2;
  const int xg_ftiles = (dst->xdim + 127) / 128;
  CK(dst->XA.reserve(l1tc_xa_floats(dst->d0p / 8, n_mtiles) * 4));
  CK(dst->XG.reserve(l1tc_xg_floats(xg_ftiles, dst->n_tiles) * 4));
  CK(dst->aux_pol.reserve((size_t)dst->n_tiles * src->naux_pol * MRL_LDT * 4));
  CKL(launch_gather_rows(idx_dev, n, src->N, src->XA.as<float>(), dst->XA.as<float>(), dst->d0p / 8, src->XG.as<float>(),
                         dst->XG.as<float>(), xg_ftiles, src->aux_pol.as<float>(), dst->aux_pol.as<float>(), src->naux_pol, st), 1);
  return 0;
}

// advantage row of the policy side inputs <- the float32 advantages mrl_batch_gae left on the device
extern "C" int mrl_batch_refresh_advantages(mrl_batch* b, void* stream) {
  if (!b || !b->has_adv32 || b->pol_head < 0) return fail("mrl_batch_refresh_advantages: needs mrl_batch_gae and bound policy inputs");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(b->device));
  CKL(launch_pack_tiles(b->adv32.p, MRL_F32, 1, 1, 1, b->N, b->aux_pol.as<float>(), b->naux_pol, 0, b->n_tiles, st), 1);
  return 0;
}

// FP32 FMA throughput of this GPU (the pipe the SIMT GEMMs are bound by), for the roofline report.
__global__ void fma_peak_kernel(float* out, int iters) {
  float a0 = threadIdx.x * 1e-6f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f, a4 = a0 + 4.f, a5 = a0 + 5.f,
        a6 = a0 + 6.f, a7 = a0 + 7.f;
  const float m = 0.999999f, c = 1e-7f;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
      a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
    }
  }
  out[blockIdx.x * blockDim.x + threadIdx.x] = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
}
extern "C" int mrl_measure_fp32_tflops(int device, double* tflops_out) {
  if (!tflops_out) return fail("mrl_measure_fp32_tflops: null out");
  CK(cudaSetDevice(device));
  int sms = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  const int blocks = sms * 8, threads = 256, iters = 4096;
  float* out = nullptr;
  CK(cudaMalloc(&out, (size_t)blocks * threads * 4));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 5; ++rep) {
    cudaEventRecord(e0, 0);
    fma_peak_kernel<<<blocks, threads>>>(out, iters);
    cudaEventRecord(e1, 0);
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double flops = 2.0 * 64.0 * iters * (double)blocks * threads;
    best = fmax(best, flops / (ms * 1e-3) / 1e12);
  }
  g_launches += 5;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(out);
  *tflops_out = best;
  return 0;
}

// mma.sync m16n8k8 TF32 throughput of this GPU (the pipe the register-chain kernels are bound by): 8 independent
// accumulators per warp, 16 warps per SM, for the roofline report.
__global__ void mma_peak_kernel(float* out, int iters) {
  float c[8][4];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) c[i][j] = 0.f;
  const unsigned a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, b0 = a0 * 3, b1 = a0 * 5;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 8; ++i)
      asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                   : "+f"(c[i][0]), "+f"(c[i][1]), "+f"(c[i][2]), "+f"(c[i][3])
                   : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
  }
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) s += c[i][j];
  out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}
extern "C" int mrl_measure_mma_tf32_tflops(int device, double* tflops_out) {
  if (!tflops_out) return fail("mrl_measure_mma_tf32_tflops: null out");
  CK(cudaSetDevice(device));
  int sms = 0;
  CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  const int blocks = sms, threads = 512, iters = 8192;
  float* out = nullptr;
  CK(cudaMalloc(&out, (size_t)blocks * threads * 4));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    cudaEventRecord(e0, 0);
    mma_peak_kernel<<<blocks, threads>>>(out, iters);
    cudaEventRecord(e1, 0);
    CK(cudaEventSynchronize(e1));
    float ms = 0.f;
    cudaEventElapsedTime(&ms, e0, e1);
    const double flops = (double)blocks * (threads / 32) * iters * 8.0 * (16.0 * 8.0 * 8.0 * 2.0);
    best = fmax(best, flops / (ms * 1e-3) / 1e12);
  }
  g_launches += 4;
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  cudaFree(out);
  *tflops_out = best;
  return 0;
}

__global__ void mix_target_kernel(const double* __restrict__ ret, const double* __restrict__ base, double mix,
                                  long long N, float* __restrict__ aux) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (N + MRL_TILE - 1) / MRL_TILE * MRL_TILE) return;
  const float v = t < N ? (float)(ret[t] * mix + base[t] * (1.0 - mix)) : 0.f;
  aux[(t / MRL_TILE) * MRL_LDT + (t % MRL_TILE)] = v;
}

extern "C" int mrl_batch_set_vf_target(mrl_batch* b, const void* y, int dtype, int loc, void* stream) {
  if (!b || !y || b->N <= 0) return fail("mrl_batch_set_vf_target: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(b->device));
  CK(b->aux_vf.reserve((size_t)b->n_tiles * MRL_LDT * 4));
  const void* src;
  RET(stage_in(b->stage2, y, (size_t)b->N * dtype_size(dtype), loc, st, &src));
  CKL(launch_pack_tiles(src, dtype, 1, 1, 1, b->N, b->aux_vf.as<float>(), 1, 0, b->n_tiles, st), 1);
  return 0;
}
// target = mixfrac * return + (1 - mixfrac) * ypred_old (core.py:622-624) from device-resident data
extern "C" int mrl_batch_mix_vf_target(mrl_batch* b, double mixfrac, void* stream) {
  if (!b || !b->has_ret || !b->has_baseline) return fail("mrl_batch_mix_vf_target: needs mrl_batch_gae first");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(b->device));
  CK(b->aux_vf.reserve((size_t)b->n_tiles * MRL_LDT * 4));
  const long long n = (long long)b->n_tiles * MRL_TILE;
  mix_target_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(b->ret.as<double>(), b->baseline.as<double>(),
                                                                 mixfrac, b->N, b->aux_vf.as<float>());
  CKL(cudaGetLastError(), 1);
  return 0;
}

// ------------------------------------------------------------------------ GAE
__global__ void merge_moments_kernel(const double* __restrict__ gathered, int world, double* __restrict__ stats) {
  double n = 0.0, mean = 0.0, m2 = 0.0;
  for (int r = 0; r < world; ++r) {
    const double bn = gathered[3 * r], bm = gathered[3 * r + 1], b2 = gathered[3 * r + 2];
    if (bn == 0.0) continue;
    if (n == 0.0) { n = bn; mean = bm; m2 = b2; continue; }
    const double tot = n + bn, d = bm - mean;
    mean += d * (bn / tot);
    m2 += b2 + d * d * (n * bn / tot);
    n = tot;
  }
  stats[0] = n; stats[1] = mean; stats[2] = m2;
}
__global__ void place_moments_kernel(const double* __restrict__ stats, double* __restrict__ gathered, int world, int rank) {
  const int i = threadIdx.x;
  if (i < 3 * world) gathered[i] = (i / 3 == rank) ? stats[i % 3] : 0.0;
}
__global__ void f32_to_f64_kernel(const float* __restrict__ x, double* __restrict__ y, long long N) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) y[i] = (double)x[i];
}

static int gae_impl(const void* reward_dev, int rdt, const void* base_dev, int bdt, const long long* off_dev,
                    const unsigned char* term_dev, int n_paths, long long N, double gamma, double lam, double* ret,
                    double* adv, cudaStream_t st) {
  if (rdt != MRL_F32 && rdt != MRL_F64) return fail("reward must be f32/f64");
  if (bdt != MRL_F32 && bdt != MRL_F64) return fail("baseline must be f32/f64");
  CKP(PK_GAE, launch_gae(reward_dev, rdt == MRL_F64, base_dev, bdt == MRL_F64, off_dev, term_dev, n_paths, N, gamma, lam,
                 ret, adv, st), 1);
  return 0;
}

extern "C" int mrl_batch_gae(mrl_batch* b, const void* reward, int reward_dtype, const void* baseline,
                             int baseline_dtype, double gamma, double lam, int standardize, mrl_comm* comm,
                             double* ret_out, double* adv_out, int loc, void* stream) {
  if (!b || !reward || b->N <= 0 || b->n_paths <= 0) return fail("mrl_batch_gae: bind observations and paths first");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(b->device));
  const long long N = b->N;
  const void* r_dev;
  RET(stage_in(b->stage2, reward, (size_t)N * dtype_size(reward_dtype), loc, st, &r_dev));
  const void* v_dev;
  int vdt = baseline_dtype;
  if (baseline) {
    if (loc == MRL_DEVICE) {
      v_dev = baseline;
    } else {
      CK(b->gather.reserve((size_t)N * dtype_size(baseline_dtype)));
      CK(cudaMemcpyAsync(b->gather.p, baseline, (size_t)N * dtype_size(baseline_dtype), cudaMemcpyHostToDevice, st));
      v_dev = b->gather.p;
    }
    CK(b->baseline.reserve((size_t)N * 8));
    if (vdt == MRL_F64) CK(cudaMemcpyAsync(b->baseline.p, v_dev, (size_t)N * 8, cudaMemcpyDeviceToDevice, st));
    else {
      f32_to_f64_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>((const float*)v_dev, b->baseline.as<double>(), N);
      CKL(cudaGetLastError(), 1);
    }
    b->has_baseline = true;
  } else if (!b->has_baseline) {
    return fail("mrl_batch_gae: baseline == NULL but mrl_net_predict_into_baseline was not called");
  }
  CK(b->ret.reserve((size_t)N * 8));
  CK(b->adv.reserve((size_t)N * 8));
  CK(b->adv32.reserve((size_t)N * 4));
  CK(b->stats.reserve(64 + MRL_MOMENTS_SCRATCH_DOUBLES * 8));
  RET(gae_impl(r_dev, reward_dtype, b->baseline.p, MRL_F64, b->offsets.as<long long>(),
               b->terminated.as<unsigned char>(), b->n_paths, N, gamma, lam, b->ret.as<double>(),
               b->adv.as<double>(), st));
  b->has_ret = true;
  if (standardize) {
    CKL(launch_moments(b->adv.as<double>(), N, b->stats.as<double>(), b->stats.as<double>() + 8, st), 2);
    if (comm && mrl_comm_world(comm) > 1) {
      const int world = mrl_comm_world(comm), rank = mrl_comm_rank(comm);
      CK(b->gather.reserve((size_t)3 * world * 8 + 64));
      place_moments_kernel<<<1, 3 * world, 0, st>>>(b->stats.as<double>(), b->gather.as<double>(), world, rank);
      CKL(cudaGetLastError(), 1);
      RET(mrl_comm_allreduce_f64(comm, b->gather.as<double>(), 3 * world, st));
      merge_moments_kernel<<<1, 1, 0, st>>>(b->gather.as<double>(), world, b->stats.as<double>());
      CKL(cudaGetLastError(), 1);
    }
    CKL(launch_normalize(b->adv.as<double>(), N, b->stats.as<double>(), b->adv32.as<float>(), st), 1);
  } else {
    cast_f64_f32(b->adv.as<double>(), b->adv32.as<float>(), N, st);
    CKL(cudaGetLastError(), 1);
  }
  b->has_adv32 = true;
  cudaMemcpyKind kind = loc == MRL_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  if (ret_out) CK(cudaMemcpyAsync(ret_out, b->ret.p, (size_t)N * 8, kind, st));
  if (adv_out) CK(cudaMemcpyAsync(adv_out, b->adv.p, (size_t)N * 8, kind, st));
  if (loc == MRL_HOST && (ret_out || adv_out)) CK(cudaStreamSynchronize(st));
  return 0;
}

extern "C" int mrl_gae(const void* reward, int reward_dtype, const void* baseline, int baseline_dtype,
                       const long long* offsets, const unsigned char* terminated, int n_paths, long long N,
                       double gamma, double lam, double* ret_out, double* adv_out, int loc, void* stream) {
  if (!reward || !baseline || !offsets || !terminated || !ret_out || !adv_out || N <= 0 || n_paths <= 0)
    return fail("mrl_gae: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  if (loc == MRL_DEVICE)
    return gae_impl(reward, reward_dtype, baseline, baseline_dtype, offsets, terminated, n_paths, N, gamma, lam,
                    ret_out, adv_out, st);
  DevBuf r, v, o, t, ro, ao;
  const size_t rb = (size_t)N * dtype_size(reward_dtype), vb = (size_t)N * dtype_size(baseline_dtype);
  int rc = 0;
  do {
    if (r.reserve(rb) || v.reserve(vb) || o.reserve((size_t)(n_paths + 1) * 8) || t.reserve(n_paths) ||
        ro.reserve((size_t)N * 8) || ao.reserve((size_t)N * 8)) { rc = fail("mrl_gae: out of device memory"); break; }
    cudaMemcpyAsync(r.p, reward, rb, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(v.p, baseline, vb, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(o.p, offsets, (size_t)(n_paths + 1) * 8, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(t.p, terminated, n_paths, cudaMemcpyHostToDevice, st);
    rc = gae_impl(r.p, reward_dtype, v.p, baseline_dtype, o.as<long long>(), t.as<unsigned char>(), n_paths, N,
                  gamma, lam, ro.as<double>(), ao.as<double>(), st);
    if (rc) break;
    cudaMemcpyAsync(ret_out, ro.p, (size_t)N * 8, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(adv_out, ao.p, (size_t)N * 8, cudaMemcpyDeviceToHost, st);
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) rc = fail("mrl_gae: %s", cudaGetErrorString(e));
  } while (0);
  r.release(); v.release(); o.release(); t.release(); ro.release(); ao.release();
  return rc;
}

extern "C" int mrl_standardize(double* x, long long N, double* stats_out, int loc, void* stream) {
  if (!x || N <= 0) return fail("mrl_standardize: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  DevBuf xd, sd;
  double* xp = x;
  if (loc == MRL_HOST) {
    CK(xd.reserve((size_t)N * 8));
    CK(cudaMemcpyAsync(xd.p, x, (size_t)N * 8, cudaMemcpyHostToDevice, st));
    xp = xd.as<double>();
  }
  CK(sd.reserve(64 + MRL_MOMENTS_SCRATCH_DOUBLES * 8));
  CKL(launch_standardize(xp, N, sd.as<double>(), sd.as<double>() + 8, nullptr, st), 3);
  if (loc == MRL_HOST) CK(cudaMemcpyAsync(x, xp, (size_t)N * 8, cudaMemcpyDeviceToHost, st));
  if (stats_out) CK(cudaMemcpyAsync(stats_out, sd.p, 24, loc == MRL_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, st));
  CK(cudaStreamSynchronize(st));
  xd.release(); sd.release();
  return 0;
}

extern "C" int mrl_zfilter_scan(const void* x, int x_dtype, long long N, int d, double* state_n, double* state_M,
                                double* state_S, int demean, int destd, double clip, void* y, int y_dtype, int loc,
                                void* stream) {
  if (!x || !y || !state_n || !state_M || !state_S || N <= 0 || d <= 0) return fail("mrl_zfilter_scan: bad arguments");
  if ((x_dtype != MRL_F32 && x_dtype != MRL_F64) || (y_dtype != MRL_F32 && y_dtype != MRL_F64))
    return fail("mrl_zfilter_scan: x and y must be f32/f64");
  cudaStream_t st = (cudaStream_t)stream;
  DevBuf xd, yd, sd, scr;
  int rc = 0;
  do {
    const size_t xb = (size_t)N * d * dtype_size(x_dtype), yb = (size_t)N * d * dtype_size(y_dtype);
    const void* xp = x;
    void* yp = y;
    cudaError_t e = cudaSuccess;
    if (loc == MRL_HOST) {
      if ((e = xd.reserve(xb)) || (e = yd.reserve(yb))) { rc = fail("mrl_zfilter_scan: %s", cudaGetErrorString(e)); break; }
      cudaMemcpyAsync(xd.p, x, xb, cudaMemcpyHostToDevice, st);
      xp = xd.p; yp = yd.p;
    }
    if ((e = sd.reserve((size_t)(4 * d + 8) * 8)) || (e = scr.reserve((size_t)zfilter_scratch_doubles(N, d) * 8))) {
      rc = fail("mrl_zfilter_scan: %s", cudaGetErrorString(e)); break;
    }
    cudaMemcpyAsync(sd.p, state_M, (size_t)d * 8, cudaMemcpyHostToDevice, st);
    cudaMemcpyAsync(sd.as<double>() + d, state_S, (size_t)d * 8, cudaMemcpyHostToDevice, st);
    e = launch_zfilter_scan(xp, x_dtype == MRL_F64, N, d, *state_n, sd.as<double>(), demean, destd, clip, yp,
                            y_dtype == MRL_F64, scr.as<double>(), st);
    if (e != cudaSuccess) { rc = fail("mrl_zfilter_scan: %s", cudaGetErrorString(e)); break; }
    g_launches += 4;
    if (loc == MRL_HOST) cudaMemcpyAsync(y, yd.p, yb, cudaMemcpyDeviceToHost, st);
    std::vector<double> out(2 * d + 1);
    cudaMemcpyAsync(out.data(), sd.as<double>() + 2 * d, (size_t)(2 * d + 1) * 8, cudaMemcpyDeviceToHost, st);
    e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) { rc = fail("mrl_zfilter_scan: %s", cudaGetErrorString(e)); break; }
    memcpy(state_M, out.data(), (size_t)d * 8);
    memcpy(state_S, out.data() + d, (size_t)d * 8);
    *state_n = out[2 * d];
  } while (0);
  xd.release(); yd.release(); sd.release(); scr.release();
  return rc;
}

// ======================================================================== network
struct mrl_net {
  int device = 0;
  NetGeom g;
  DevBuf adam_m, adam_v, sgd_acc;   // PpoSgd: Adam moments (float32) and the running sum of the minibatch losses
  long long adam_t = 0;
  DevBuf WC, VC;           // tcgen05 Fisher-vector chain: weight images of theta / of the tangent
  bool tc_fvp = false;
  bool layers = false;     // layers >= 2 run layer by layer (mlp_layers.cu): the fused mid_* kernels cannot hold the net
  DevBuf R0, R1;           // its ping-pong buffers (deltas, R-activations)
  DevBuf DG, WBt, WBv, theta, theta_prev, theta_trial, img, imgv, vflat, Z1, cache, part1, partm, loss_part, out32,
      out64, g32, cg_b, cg_x, cg_r, cg_p, p32, x32, fullstep, cgstate, cgscratch, scal, headout, stage;
  unsigned long long params_version = 1, cache_params_version = 0, cache_batch_version = 0;
  const mrl_batch* cache_batch = nullptr;
  mrl_comm* comm = nullptr;
  double* h_scal = nullptr;   // pinned
  CgState* h_cg = nullptr;    // pinned
  bool last_valid = false;
};

static int world_of(const mrl_net* n) { return n->comm ? mrl_comm_world(n->comm) : 1; }

extern "C" int mrl_net_create(mrl_net** out, int device, int n_layers, const int* dims, int head, int activation) {
  if (!out || !dims || n_layers < 1 || n_layers > MRL_MAX_LAYERS) return fail("mrl_net_create: 1..%d layers", MRL_MAX_LAYERS);
  if (head < 0 || head > 2 || activation < 0 || activation > 2) return fail("mrl_net_create: bad head/activation");
  for (int l = 0; l <= n_layers; ++l)
    if (dims[l] <= 0) return fail("mrl_net_create: dims must be positive");
  for (int l = 1; l <= n_layers; ++l)
    if (dims[l] > 256) return fail("mrl_net_create: layer width %d > 256 not supported by the fused kernels", dims[l]);
  if (dims[n_layers] > 64) return fail("mrl_net_create: output dim %d > 64 not supported", dims[n_layers]);
  if (head == MRL_VALUE && dims[n_layers] != 1) return fail("mrl_net_create: value head needs output dim 1");
  CK(cudaSetDevice(device));
  mrl_net* n = new mrl_net();
  n->device = device;
  const int d = dims[n_layers];
  const int naux = head == MRL_GAUSS ? 1 + 3 * d : (head == MRL_CATEGORICAL ? 2 + d : 1);
  mrl_build_geom(&n->g, n_layers, dims, head, activation, naux);
  if (!l1tc_supported(n->g)) {
    delete n;
    return fail("mrl_net_create: input dim %d x first hidden width %d exceeds the TMEM budget of the layer-1 tensor-core kernels", dims[0], dims[1]);
  }
  int dev_smem = 0;
  CK(cudaDeviceGetAttribute(&dev_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  // a net whose fused reverse-sweep kernel does not fit in shared memory runs layers >= 2 one launch at a time
  n->layers = mid_backward_smem(n->g, head == MRL_VALUE ? MRL_MODE_GRAD : MRL_MODE_FVP) + 2048 > (size_t)dev_smem;
  const size_t P = n->g.P;
  cudaError_t e = cudaSuccess;
  auto R = [&](DevBuf& b, size_t bytes) { if (e == cudaSuccess) e = b.reserve(bytes); };
  R(n->theta, P * 4); R(n->theta_prev, P * 4); R(n->theta_trial, P * 4); R(n->vflat, P * 4);
  R(n->img, (size_t)n->g.img_floats * 4); R(n->imgv, (size_t)n->g.img_floats * 4);
  R(n->WBt, l1tc_wb_floats(n->g) * 4); R(n->WBv, l1tc_wb_floats(n->g) * 4);
  R(n->out32, P * 4); R(n->out64, P * 8); R(n->g32, P * 4);
  R(n->cg_b, P * 8); R(n->cg_x, P * 8); R(n->cg_r, P * 8); R(n->cg_p, P * 8);
  R(n->p32, P * 4); R(n->x32, P * 4); R(n->fullstep, P * 8);
  R(n->cgstate, sizeof(CgState)); R(n->scal, 32 * 8); R(n->cgscratch, CG_SCRATCH_DOUBLES * 8);
  {
    n->tc_fvp = !n->layers && fvp_tc_supported(n->g);
    if (n->tc_fvp) {
      R(n->WC, fvp_tc_image_floats(n->g, 0) * 4);
      R(n->VC, fvp_tc_image_floats(n->g, 1) * 4);
    }
  }
  if (e == cudaSuccess) e = cudaMallocHost(&n->h_scal, 32 * 8);
  if (e == cudaSuccess) e = cudaMallocHost(&n->h_cg, sizeof(CgState));
  if (e == cudaSuccess) e = cudaMemset(n->theta.p, 0, P * 4);
  if (e == cudaSuccess) e = cudaMemset(n->cgscratch.p, 0, CG_SCRATCH_DOUBLES * 8);
  if (e != cudaSuccess) {
    mrl_net_destroy(n);
    return fail("mrl_net_create: %s", cudaGetErrorString(e));
  }
  *out = n;
  return 0;
}

extern "C" int mrl_net_destroy(mrl_net* n) {
  if (!n) return 0;
  cudaSetDevice(n->device);
  DevBuf* bufs[] = {&n->adam_m, &n->adam_v, &n->sgd_acc, &n->WC, &n->VC, &n->DG, &n->WBt, &n->WBv, &n->theta, &n->theta_prev, &n->theta_trial, &n->img, &n->imgv, &n->vflat,
                    &n->Z1, &n->cache, &n->part1, &n->partm, &n->loss_part, &n->out32, &n->out64, &n->g32,
                    &n->cg_b, &n->cg_x, &n->cg_r, &n->cg_p, &n->p32, &n->x32, &n->fullstep, &n->cgstate, &n->cgscratch, &n->scal,
                    &n->headout, &n->stage, &n->R0, &n->R1};
  for (DevBuf* d : bufs) d->release();
  if (n->h_scal) cudaFreeHost(n->h_scal);
  if (n->h_cg) cudaFreeHost(n->h_cg);
  delete n;
  return 0;
}
extern "C" long long mrl_net_num_params(const mrl_net* n) { return n ? n->g.P : -1; }
extern "C" int mrl_net_set_comm(mrl_net* n, mrl_comm* c) {
  if (!n) return fail("mrl_net_set_comm: null net");
  n->comm = c;
  return 0;
}

__global__ void negate_first(double* s) { s[0] = -s[0]; }
__global__ void f64_to_f32_kernel(const double* __restrict__ x, float* __restrict__ y, long long N) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < N) y[i] = (float)x[i];
}
void cast_f64_f32(const double* x, float* y, long long N, cudaStream_t st) {
  if (N > 0) f64_to_f32_kernel<<<(unsigned)((N + 255) / 256), 256, 0, st>>>(x, y, N);
}

static int repack(mrl_net* n, cudaStream_t st) {
  CKP(PK_PACK, launch_pack_params(n->g, n->theta.as<float>(), n->img.as<float>(), n->WBt.as<float>(), st), 1);
  if (n->tc_fvp) CKP(PK_PACK, launch_fvp_tc_pack(n->g, n->theta.as<float>(), n->WC.as<float>(), 0, st), 1);
  n->params_version++;
  return 0;
}

extern "C" int mrl_net_set_params(mrl_net* n, const void* theta, int dtype, int loc, void* stream) {
  if (!n || !theta) return fail("mrl_net_set_params: bad arguments");
  if (dtype != MRL_F32 && dtype != MRL_F64) return fail("mrl_net_set_params: theta must be f32/f64");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  const size_t P = n->g.P;
  const void* src;
  RET(stage_in(n->stage, theta, P * dtype_size(dtype), loc, st, &src));
  if (dtype == MRL_F32) {
    if (src != n->theta.p) CK(cudaMemcpyAsync(n->theta.p, src, P * 4, cudaMemcpyDeviceToDevice, st));
  } else {
    cast_f64_f32((const double*)src, n->theta.as<float>(), (long long)P, st);   // theta.astype(floatX), core.py:540
    CKL(cudaGetLastError(), 1);
  }
  return repack(n, st);
}
extern "C" int mrl_net_get_params(mrl_net* n, float* theta, int loc, void* stream) {
  if (!n || !theta) return fail("mrl_net_get_params: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  CK(cudaMemcpyAsync(theta, n->theta.p, (size_t)n->g.P * 4, loc == MRL_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
  if (loc == MRL_HOST) CK(cudaStreamSynchronize(st));
  return 0;
}

// ------------------------------------------------------------------------ passes
struct Plan { int slab_tiles, n_slabs; };
static Plan plan_for(const mrl_batch* b, bool pairs = false) {
  // One CTA per slab; a slab is <= MRL_MAX_SLAB_TILES tiles (fp32 accumulation span).  Small batches get
  // one wave of CTAs; large ones the slab size with the fewest tile-rounds on this GPU's SM count.
  const int sms = mrl_sm_count();   // callers have made b->device current
  Plan p;
  if (pairs) {
    // kernels that walk two tiles per pass: the forward chain, and the tcgen05 Fisher-vector chain whose
    // 128-timestep MMA tiles are pairs of cache tiles (slabs of 1..8 of them)
    if (b->n_tiles <= sms * 2) {
      p.slab_tiles = 2;
    } else {
      long long best = -1;
      p.slab_tiles = MRL_MAX_SLAB_TILES;
      const int smin = b->n_tiles <= sms * MRL_MAX_SLAB_TILES ? 2 : 8;
      for (int s = MRL_MAX_SLAB_TILES; s >= smin; s -= 2) {
        const long long slabs = (b->n_tiles + s - 1) / s;
        const long long cost = (slabs + sms - 1) / sms * (s / 2);
        if (best < 0 || cost < best) { best = cost; p.slab_tiles = s; }
      }
    }
    p.n_slabs = (b->n_tiles + p.slab_tiles - 1) / p.slab_tiles;
    return p;
  }
  // The backward chain kernel walks 3 tiles per pass (the forward one 2) and clips the last pass of a slab, so
  // any slab size is legal; the cost of a plan is (waves of slabs) x (passes per slab).
  if (b->n_tiles <= sms * 3) {
    p.slab_tiles = 3;
  } else {
    long long best = -1;
    p.slab_tiles = 15;
    const int smin = b->n_tiles <= sms * MRL_MAX_SLAB_TILES ? 3 : 8;
    for (int s = MRL_MAX_SLAB_TILES; s >= smin; --s) {
      const long long slabs = (b->n_tiles + s - 1) / s;
      const long long cost = (slabs + sms - 1) / sms * ((s + 2) / 3);
      if (best < 0 || cost < best) { best = cost; p.slab_tiles = s; }
    }
  }
  if (p.slab_tiles < 1) p.slab_tiles = 1;
  p.n_slabs = (b->n_tiles + p.slab_tiles - 1) / p.slab_tiles;
  return p;
}

static int check_pair(const mrl_net* n, const mrl_batch* b, bool need_aux) {
  if (!n || !b) return fail("null net or batch");
  if (b->N <= 0) return fail("batch has no observations");
  if (n->device != b->device) return fail("net and batch live on different devices");
  if (n->g.d[0] > b->xdim) return fail("net input dim %d > batch feature dim %d", n->g.d[0], b->xdim);
  if (need_aux) {
    if (n->g.head == MRL_VALUE) {
      if (!b->aux_vf.p) return fail("value target not bound (mrl_batch_set_vf_target)");
    } else {
      if (b->pol_head != n->g.head || b->pol_dout != n->g.d[n->g.L])
        return fail("policy inputs not bound for this head (mrl_batch_set_policy_inputs)");
    }
  }
  return 0;
}
static const float* aux_of(const mrl_net* n, const mrl_batch* b) {
  return n->g.head == MRL_VALUE ? b->aux_vf.as<float>() : b->aux_pol.as<float>();
}

static int reserve_ws(mrl_net* n, const mrl_batch* b, const Plan& pl) {
  const NetGeom& g = n->g;
  // one tile of slack behind both: the tcgen05 chain reads up to 15 feature rows past a layer's width (see
  // mlp_fvp_tc.cu); fresh allocations are zeroed so that the slack never holds a NaN pattern
  for (DevBuf* d : {&n->Z1, &n->cache}) {
    const size_t rows = d == &n->Z1 ? (size_t)g.d[1] : (size_t)g.act_rows;
    const size_t bytes = (size_t)(b->n_tiles + 1) * rows * MRL_LDT * 4;
    if (bytes > d->cap) {
      CK(d->reserve(bytes));
      CK(cudaMemsetAsync(d->p, 0, d->cap, 0));
      CK(cudaStreamSynchronize(0));
    }
  }
  CK(n->DG.reserve(l1tc_dg_floats(g, b->n_tiles) * 4));
  if (n->layers) {
    CK(n->R0.reserve(layers_ws_floats(g, b->n_tiles) * 4));
    CK(n->R1.reserve(layers_ws_floats(g, b->n_tiles) * 4));
  }
  CK(n->part1.reserve((size_t)pl.n_slabs * g.d[0] * g.n1p * 4));
  CK(n->partm.reserve((size_t)pl.n_slabs * g.pmid * 4));
  CK(n->loss_part.reserve((size_t)pl.n_slabs * 4 * 8));
  return 0;
}

// L1F + mid forward.  losses -> n->scal[0..3] (device, already scaled by 1/N_global and all-reduced); clip_eps > 0:
// scal[0] is the mean clipped objective and scal[3] the fraction of clipped rows
static int pass_forward(mrl_net* n, mrl_batch* b, bool want_losses, bool want_cache, float* head_out,
                        cudaStream_t st, int reverse_kl = 0, float clip_eps = 0.f) {
  const NetGeom& g = n->g;
  const Plan pl = plan_for(b, true);
  RET(reserve_ws(n, b, pl));
  // the batch tile has b->d0p feature rows; the net consumes the first g.d0p of them
  NetGeom gl = g;
  CKP(PK_L1F, launch_l1_forward_tc(gl, b->XA.as<float>(), b->d0p / 8, n->WBt.as<float>(), n->Z1.as<float>(), b->n_tiles, st), 1);
  MidFwdArgs a;
  a.img = n->img.as<float>();
  a.Zt = n->Z1.as<float>();
  a.aux = want_losses ? aux_of(n, b) : nullptr;
  a.cache = want_cache ? n->cache.as<float>() : nullptr;
  a.head_out = head_out;
  a.loss_part = want_losses ? n->loss_part.as<double>() : nullptr;
  a.N = b->N;
  a.n_tiles = b->n_tiles;
  a.slab_tiles = pl.slab_tiles;
  a.reverse_kl = reverse_kl;
  if (n->layers) {
    // the layer-by-layer path keeps its activations in the cache even when the caller does not want them
    a.cache = n->cache.as<float>();
    if (!want_cache) n->cache_batch = nullptr;
    int nk = 0;
    CKP(PK_MIDF, launch_layers_forward(g, a, pl.n_slabs, st, &nk, clip_eps), nk);
  } else if (chain_fwd_shape(g) != 0) CKP(PK_MIDF, launch_chain_forward(g, a, pl.n_slabs, st, clip_eps), 1);
  else CKP(PK_MIDF, launch_mid_forward(g, a, pl.n_slabs, st, clip_eps), 1);
  if (want_losses) {
    CKL(launch_reduce_losses(n->loss_part.as<double>(), pl.n_slabs, 1.0 / (double)b->Nglobal, n->scal.as<double>(), st), 1);
    if (world_of(n) > 1) RET(mrl_comm_allreduce_f64(n->comm, n->scal.as<double>(), 4, st));
  }
  if (want_cache) {
    n->cache_params_version = n->params_version;
    n->cache_batch_version = b->version;
    n->cache_batch = b;
  }
  return 0;
}
static bool cache_ok(const mrl_net* n, const mrl_batch* b) {
  return n->cache_batch == b && n->cache_batch_version == b->version && n->cache_params_version == n->params_version;
}

// reverse sweep + layer-1 gradient + slab reduce -> out32 (float[P], device) and out64 (double[P]).
// MRL_MODE_GRAD_CLIP: the gradient of the PPO clipped objective with clip range clip_eps.
static int pass_backward(mrl_net* n, mrl_batch* b, int mode, const double* coef_dev, int reverse_kl,
                         const float* v_dev, double l2c2, float* out32, double* out64, cudaStream_t st,
                         float clip_eps = 0.f) {
  const NetGeom& g = n->g;
  const bool tc = mode == MRL_MODE_FVP && n->tc_fvp;
  const Plan pl = plan_for(b, tc);
  RET(reserve_ws(n, b, pl));
  if (!cache_ok(n, b)) RET(pass_forward(n, b, false, true, nullptr, st));
  MidBwdArgs a;
  a.img = n->img.as<float>();
  a.imgv = nullptr;
  a.Zt = nullptr;
  if (mode == MRL_MODE_FVP) {
    // tangent -> operand images: one launch packs the layer-1 operand and (tcgen05 chain) the chain images
    if (tc) CKP(PK_PACK, launch_fvp_tc_pack(g, v_dev, n->VC.as<float>(), 1, st, n->WBv.as<float>()), 1);
    else CKP(PK_PACK, launch_pack_params(g, v_dev, n->imgv.as<float>(), n->WBv.as<float>(), st), 1);
    CKP(PK_L1F, launch_l1_forward_tc(g, b->XA.as<float>(), b->d0p / 8, n->WBv.as<float>(), n->Z1.as<float>(), b->n_tiles, st), 1);
    a.imgv = n->imgv.as<float>();
    a.Zt = n->Z1.as<float>();
  }
  a.aux = mode != MRL_MODE_FVP ? aux_of(n, b) : nullptr;
  a.cache = n->cache.as<float>();
  a.coef = coef_dev;
  a.DG = n->DG.as<float>();
  a.nu = l1tc_nu(g);
  a.partm = n->partm.as<float>();
  a.N = b->N;
  a.n_tiles = b->n_tiles;
  a.slab_tiles = pl.slab_tiles;
  a.mode = mode;
  a.reverse_kl = reverse_kl;
  if (n->layers) {
    int nk = 0;
    CKP(mode == MRL_MODE_FVP ? PK_MIDB_FVP : PK_MIDB_GRAD,
        launch_layers_backward(g, a, n->R0.as<float>(), n->R1.as<float>(), pl.n_slabs, st, &nk, clip_eps), nk);
  } else if (tc) {
    FvpTcArgs x;
    x.WC = n->WC.as<float>(); x.VC = n->VC.as<float>(); x.vflat = v_dev; x.img = n->img.as<float>();
    x.Zt = n->Z1.as<float>(); x.cache = n->cache.as<float>(); x.DG = n->DG.as<float>(); x.partm = n->partm.as<float>();
    x.N = b->N; x.n_tiles = b->n_tiles; x.slab_tiles = pl.slab_tiles; x.n_slabs = pl.n_slabs;
    CKP(PK_MIDB_FVP, launch_fvp_tc(g, x, st), 1);
  } else if (mode != MRL_MODE_FVP && chain_bwd_shape(g) != 0) CKP(PK_MIDB_GRAD, launch_chain_backward(g, a, pl.n_slabs, st, clip_eps), 1);
  else CKP(mode == MRL_MODE_FVP ? PK_MIDB_FVP : PK_MIDB_GRAD, launch_mid_backward(g, a, pl.n_slabs, st, clip_eps), 1);
  CKP(PK_L1G, launch_l1_grad_tc(g, b->XG.as<float>(), (b->xdim + 127) / 128, n->DG.as<float>(), n->part1.as<float>(),
                                pl.slab_tiles, b->n_tiles, pl.n_slabs, st), 1);
  const int world = world_of(n);
  // terms that are not sums over timesteps are divided by `world` so that the sum over ranks restores them
  const double vls = (mode == MRL_MODE_FVP) ? 2.0 / world : 0.0;
  const bool p2p = world > 1 && mrl_comm_p2p_ready(n->comm, g.P);
  // peer-memory transport: the reduce kernel publishes this rank's vector, waits for the peers' and writes the sum
  // over ranks itself (comm.h); otherwise out64 holds this rank's share and NCCL sums it
  P2pPush push;
  P2pGather gather;
  if (p2p) {
    RET(mrl_comm_p2p_begin(n->comm, g.P, &push));
    RET(mrl_comm_p2p_pending(n->comm, &gather));
  }
  CKP(PK_REDUCE, launch_reduce_partials(g, n->part1.as<float>(), n->partm.as<float>(), pl.n_slabs, 1.0 / (double)b->Nglobal,
                             l2c2 != 0.0 ? n->theta.as<float>() : nullptr, l2c2 / world,
                             mode == MRL_MODE_FVP ? v_dev : nullptr, vls, (world > 1 && !p2p) ? nullptr : out32,
                             out64, p2p ? &push : nullptr, p2p ? &gather : nullptr, st), 1);
  if (world > 1 && !p2p) {
    RET(mrl_comm_allreduce_f64(n->comm, out64, g.P, st));
    if (out32) {
      cast_f64_f32(out64, out32, g.P, st);
      CKL(cudaGetLastError(), 1);
    }
  }
  return 0;
}

static int d2h_sync(void* dst, const void* src, size_t bytes, cudaStream_t st) {
  CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  return 0;
}
// after a stream synchronisation: did a peer-memory sum of this net time out?
static int comm_ok(const mrl_net* n) { return n->comm ? mrl_comm_p2p_error(n->comm) : 0; }

extern "C" int mrl_net_forward(mrl_net* n, mrl_batch* b, float* out, int loc, void* stream) {
  RET(check_pair(n, b, false));
  if (!out) return fail("mrl_net_forward: out is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  const size_t bytes = (size_t)b->N * n->g.d[n->g.L] * 4;
  float* dev = out;
  if (loc == MRL_HOST) {
    CK(n->headout.reserve(bytes));
    dev = n->headout.as<float>();
  }
  RET(pass_forward(n, b, false, false, dev, st));
  if (loc == MRL_HOST) RET(d2h_sync(out, dev, bytes, st));
  return 0;
}

extern "C" int mrl_net_predict_into_baseline(mrl_net* n, mrl_batch* b, void* stream) {
  RET(check_pair(n, b, false));
  if (n->g.head != MRL_VALUE) return fail("mrl_net_predict_into_baseline: not a value net");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  CK(n->headout.reserve((size_t)b->N * 4));
  CK(b->baseline.reserve((size_t)b->N * 8));
  RET(pass_forward(n, b, false, false, n->headout.as<float>(), st));
  f32_to_f64_kernel<<<(unsigned)((b->N + 255) / 256), 256, 0, st>>>(n->headout.as<float>(), b->baseline.as<double>(), b->N);
  CKL(cudaGetLastError(), 1);
  b->has_baseline = true;
  return 0;
}

extern "C" int mrl_net_losses(mrl_net* n, mrl_batch* b, double out[3], void* stream) {
  RET(check_pair(n, b, true));
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  RET(pass_forward(n, b, true, false, nullptr, st));
  RET(d2h_sync(n->h_scal, n->scal.p, 32, st));
  if (n->g.head != MRL_VALUE) out[0] = -n->h_scal[0];   // surr = -(1/N) sum rho*adv  (trpo.py:42)
  else out[0] = n->h_scal[0];
  out[1] = n->h_scal[1];
  out[2] = n->h_scal[2];
  return 0;
}

static int copy_out(void* dst, const void* src_dev, size_t bytes, int loc, cudaStream_t st) {
  CK(cudaMemcpyAsync(dst, src_dev, bytes, loc == MRL_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, st));
  if (loc == MRL_HOST) CK(cudaStreamSynchronize(st));
  return 0;
}

extern "C" int mrl_net_policy_gradient(mrl_net* n, mrl_batch* b, float* gout, int loc, double losses[3], void* stream) {
  RET(check_pair(n, b, true));
  if (n->g.head == MRL_VALUE) return fail("mrl_net_policy_gradient: value net");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  RET(pass_forward(n, b, true, true, nullptr, st));
  RET(pass_backward(n, b, MRL_MODE_GRAD, nullptr, 0, nullptr, 0.0, n->g32.as<float>(), n->out64.as<double>(), st));
  if (losses) {
    RET(d2h_sync(n->h_scal, n->scal.p, 32, st));
    losses[0] = -n->h_scal[0]; losses[1] = n->h_scal[1]; losses[2] = n->h_scal[2];
  }
  if (gout) RET(copy_out(gout, n->g32.p, (size_t)n->g.P * 4, loc, st));
  return 0;
}

extern "C" int mrl_net_fvp(mrl_net* n, mrl_batch* b, const float* v, float* out, int loc, void* stream) {
  RET(check_pair(n, b, false));
  if (!v || !out) return fail("mrl_net_fvp: null vector");
  if (n->g.head == MRL_VALUE) return fail("mrl_net_fvp: value net");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  const float* vdev = v;
  if (loc == MRL_HOST) {
    CK(cudaMemcpyAsync(n->vflat.p, v, (size_t)n->g.P * 4, cudaMemcpyHostToDevice, st));
    vdev = n->vflat.as<float>();
  }
  RET(pass_backward(n, b, MRL_MODE_FVP, nullptr, 0, vdev, 0.0, n->out32.as<float>(), n->out64.as<double>(), st));
  return copy_out(out, n->out32.p, (size_t)n->g.P * 4, loc, st);
}

extern "C" int mrl_net_ppo_lossgrad(mrl_net* n, mrl_batch* b, double kl_coeff, double kl_cutoff, int reverse_kl,
                                    double* pensurr, double* gout, double losses[3], void* stream) {
  RET(check_pair(n, b, true));
  if (n->g.head == MRL_VALUE) return fail("mrl_net_ppo_lossgrad: value net");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  // forward: surr/kl/ent; kl(new||old) needs its own sum when reverse_kl: handled inside the forward by aux order
  RET(pass_forward(n, b, true, gout != nullptr, nullptr, st, reverse_kl));
  double* scal = n->scal.as<double>();
  // scal[0] holds +mean(rho*adv): the coefficient kernel expects surr = -that
  negate_first<<<1, 1, 0, st>>>(scal);
  CKL(cudaGetLastError(), 1);
  CKL(launch_ppo_coef(scal, kl_coeff, kl_cutoff, scal + 8, scal + 10, st), 1);
  if (gout)   // gout == NULL: losses / pensurr only (compute_losses, ppo.py:57)
    RET(pass_backward(n, b, MRL_MODE_GRAD, scal + 8, reverse_kl, nullptr, 0.0, nullptr, n->out64.as<double>(), st));
  RET(d2h_sync(n->h_scal, n->scal.p, 16 * 8, st));
  RET(comm_ok(n));
  if (losses) { losses[0] = n->h_scal[0]; losses[1] = n->h_scal[1]; losses[2] = n->h_scal[2]; }
  if (pensurr) *pensurr = n->h_scal[10];
  if (gout) RET(d2h_sync(gout, n->out64.p, (size_t)n->g.P * 8, st));
  return 0;
}

__global__ void l2_sum_kernel(const float* __restrict__ theta, int P, double coef, double* __restrict__ out) {
  __shared__ double scratch[32];
  double s = 0.0;
  for (int i = threadIdx.x; i < P; i += blockDim.x) s += (double)theta[i] * (double)theta[i];
  s = block_sum(s, scratch);
  if (threadIdx.x == 0) *out = coef * s;
}

extern "C" int mrl_net_vf_lossgrad(mrl_net* n, mrl_batch* b, double l2coeff, double losses[3], double* gout, void* stream) {
  RET(check_pair(n, b, true));
  if (n->g.head != MRL_VALUE) return fail("mrl_net_vf_lossgrad: not a value net");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  RET(pass_forward(n, b, true, gout != nullptr, nullptr, st));
  l2_sum_kernel<<<1, 1024, 0, st>>>(n->theta.as<float>(), n->g.P, l2coeff, n->scal.as<double>() + 4);
  CKL(cudaGetLastError(), 1);
  if (gout) RET(pass_backward(n, b, MRL_MODE_GRAD, nullptr, 0, nullptr, 2.0 * l2coeff, nullptr, n->out64.as<double>(), st));
  RET(d2h_sync(n->h_scal, n->scal.p, 8 * 8, st));
  RET(comm_ok(n));
  const double mse = n->h_scal[0], l2 = n->h_scal[4];
  if (losses) { losses[0] = mse + l2; losses[1] = mse; losses[2] = l2; }
  if (gout) RET(d2h_sync(gout, n->out64.p, (size_t)n->g.P * 8, st));
  return 0;
}

// ------------------------------------------------------------------------ PpoSgd minibatch step
// the Adam moments and step counter of adam_updates (ppo.py:231-258), allocated at the first minibatch step
static int adam_init(mrl_net* n, cudaStream_t st) {
  if (n->adam_m.p) return 0;
  const size_t P = n->g.P;
  CK(n->adam_m.reserve(P * 4));
  CK(n->adam_v.reserve(P * 4));
  CK(n->sgd_acc.reserve(4 * 8));
  CK(cudaMemsetAsync(n->adam_m.p, 0, P * 4, st));
  CK(cudaMemsetAsync(n->adam_v.p, 0, P * 4, st));
  CK(cudaMemsetAsync(n->sgd_acc.p, 0, 4 * 8, st));
  n->adam_t = 0;
  return 0;
}
// one Adam step on theta with the float64 gradient in out64, then the repack of the parameter images
static int adam_apply(mrl_net* n, double stepsize, double beta1, double beta2, double epsilon, cudaStream_t st) {
  n->adam_t += 1;
  const float f1 = (float)beta1, f2 = (float)beta2;
  // a_t in float32, operation by operation as the numpy float32 expression of the host version
  const float a_t = (float)stepsize * sqrtf(1.f - powf(f2, (float)n->adam_t)) / (1.f - powf(f1, (float)n->adam_t));
  CKL(launch_adam_step((int)n->g.P, n->out64.as<double>(), n->theta.as<float>(), n->adam_m.as<float>(),
                       n->adam_v.as<float>(), a_t, f1, f2, (float)epsilon, st), 1);
  return repack(n, st);
}

// One `train` call of PpoSgdUpdater (ppo.py:162-167,199): penalised-surrogate loss and gradient on the minibatch, then
// the Adam update of adam_updates (ppo.py:231-258), everything on the device and without a host synchronisation; the
// losses (evaluated BEFORE the step, as Theano evaluates outputs before applying updates) are added to a running sum.
extern "C" int mrl_net_ppo_sgd_step(mrl_net* n, mrl_batch* b, double kl_coeff, double kl_cutoff, int reverse_kl,
                                    double stepsize, double beta1, double beta2, double epsilon, void* stream) {
  RET(check_pair(n, b, true));
  if (n->g.head == MRL_VALUE) return fail("mrl_net_ppo_sgd_step: value net");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  RET(adam_init(n, st));
  RET(pass_forward(n, b, true, true, nullptr, st, reverse_kl));
  double* scal = n->scal.as<double>();
  negate_first<<<1, 1, 0, st>>>(scal);
  CKL(cudaGetLastError(), 1);
  CKL(launch_ppo_coef(scal, kl_coeff, kl_cutoff, scal + 8, scal + 10, st), 1);
  CKL(launch_accum_losses(scal, n->sgd_acc.as<double>(), st), 1);
  RET(pass_backward(n, b, MRL_MODE_GRAD, scal + 8, reverse_kl, nullptr, 0.0, nullptr, n->out64.as<double>(), st));
  return adam_apply(n, stepsize, beta1, beta2, epsilon, st);
}
// mean of the minibatch losses accumulated since the last read (surr, kl, ent) and their count; resets the sum
extern "C" int mrl_net_ppo_sgd_read(mrl_net* n, double losses[3], long long* count, void* stream) {
  if (!n || !losses) return fail("mrl_net_ppo_sgd_read: bad arguments");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  if (!n->sgd_acc.p) return fail("mrl_net_ppo_sgd_read: no minibatch step has run");
  RET(d2h_sync(n->h_scal, n->sgd_acc.p, 32, st));
  RET(comm_ok(n));
  const double c = n->h_scal[3];
  for (int i = 0; i < 3; ++i) losses[i] = c > 0 ? n->h_scal[i] / c : 0.0;
  if (count) *count = (long long)c;
  CK(cudaMemsetAsync(n->sgd_acc.p, 0, 32, st));
  return 0;
}
// ------------------------------------------------------------------------ PPO with the clipped surrogate objective
// clip_eps must be > 0 also after the rounding to float32 in which the kernels compare; +inf is no clipping
static int check_clip(const char* fn, const mrl_net* n, const mrl_batch* b, double clip_eps) {
  if (!((float)clip_eps > 0.f)) return fail("%s: clip_eps must be > 0 (got %g)", fn, clip_eps);
  if (!n || !b) return fail("%s: null net or batch", fn);
  if (n->g.head == MRL_VALUE) return fail("%s: value net", fn);
  return check_pair(n, b, true);
}

extern "C" int mrl_net_ppo_clip_lossgrad(mrl_net* n, mrl_batch* b, double clip_eps, double* gout, double losses[4],
                                         void* stream) {
  RET(check_clip("mrl_net_ppo_clip_lossgrad", n, b, clip_eps));
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  const float eps = (float)clip_eps;
  RET(pass_forward(n, b, true, gout != nullptr, nullptr, st, 0, eps));
  if (gout) RET(pass_backward(n, b, MRL_MODE_GRAD_CLIP, nullptr, 0, nullptr, 0.0, nullptr, n->out64.as<double>(), st, eps));
  RET(d2h_sync(n->h_scal, n->scal.p, 4 * 8, st));
  RET(comm_ok(n));
  if (losses) {
    losses[0] = -n->h_scal[0]; losses[1] = n->h_scal[1]; losses[2] = n->h_scal[2]; losses[3] = n->h_scal[3];
  }
  if (gout) RET(d2h_sync(gout, n->out64.p, (size_t)n->g.P * 8, st));
  return 0;
}

// One minibatch step of PPO-clip: forward with the activation cache (no loss sums), the clipped gradient, the Adam
// step of mrl_net_ppo_sgd_step on the same moments, the repack; no host synchronisation.
extern "C" int mrl_net_ppo_clip_sgd_step(mrl_net* n, mrl_batch* b, double clip_eps, double stepsize, double beta1,
                                         double beta2, double epsilon, void* stream) {
  RET(check_clip("mrl_net_ppo_clip_sgd_step", n, b, clip_eps));
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  RET(adam_init(n, st));
  const float eps = (float)clip_eps;
  RET(pass_forward(n, b, false, true, nullptr, st));
  RET(pass_backward(n, b, MRL_MODE_GRAD_CLIP, nullptr, 0, nullptr, 0.0, nullptr, n->out64.as<double>(), st, eps));
  return adam_apply(n, stepsize, beta1, beta2, epsilon, st);
}

// restart Adam (moments and step counter to zero)
extern "C" int mrl_net_adam_reset(mrl_net* n, void* stream) {
  if (!n) return fail("mrl_net_adam_reset: null net");
  CK(cudaSetDevice(n->device));
  n->adam_t = 0;
  if (n->adam_m.p) {
    cudaStream_t st = (cudaStream_t)stream;
    CK(cudaMemsetAsync(n->adam_m.p, 0, (size_t)n->g.P * 4, st));
    CK(cudaMemsetAsync(n->adam_v.p, 0, (size_t)n->g.P * 4, st));
    CK(cudaMemsetAsync(n->sgd_acc.p, 0, 32, st));
  }
  return 0;
}

// ------------------------------------------------------------------------ TRPO step
extern "C" int mrl_net_trpo_step(mrl_net* n, mrl_batch* b, const mrl_trpo_cfg* cfg, double stats[6], int info[6],
                                 void* stream) {
  RET(check_pair(n, b, true));
  if (!cfg || !stats) return fail("mrl_net_trpo_step: null cfg/stats");
  if (n->g.head == MRL_VALUE) return fail("mrl_net_trpo_step: value net");
  cudaStream_t st = (cudaStream_t)stream;
  CK(cudaSetDevice(n->device));
  const NetGeom& g = n->g;
  const int P = g.P;
  int loss_passes = 0;
  n->last_valid = false;

  // gradient + losses at theta_old (trpo.py:94-95); the forward pass also fills the activation cache
  CK(cudaMemcpyAsync(n->theta_prev.p, n->theta.p, (size_t)P * 4, cudaMemcpyDeviceToDevice, st));
  RET(pass_forward(n, b, true, true, nullptr, st));
  loss_passes++;
  RET(pass_backward(n, b, MRL_MODE_GRAD, nullptr, 0, nullptr, 0.0, n->g32.as<float>(), n->out64.as<double>(), st));
  CKL(launch_cg_init(P, n->g32.as<float>(), n->cg_b.as<double>(), n->cg_x.as<double>(), n->cg_r.as<double>(),
                     n->cg_p.as<double>(), n->p32.as<float>(), n->cgstate.as<CgState>(), st), 1);
  CK(cudaMemcpyAsync(n->h_scal, n->scal.p, 32, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(n->h_cg, n->cgstate.p, sizeof(CgState), cudaMemcpyDeviceToHost, st));
  // CG does not depend on the host check below, so it is enqueued before the sync
  for (int it = 0; it < cfg->cg_iters; ++it) {
    RET(pass_backward(n, b, MRL_MODE_FVP, nullptr, 0, n->p32.as<float>(), 0.0, n->out32.as<float>(),
                      n->out64.as<double>(), st));
    CKP(PK_CG, launch_cg_step(P, n->out32.as<float>(), cfg->cg_damping, cfg->residual_tol, n->cg_x.as<double>(),
                       n->cg_r.as<double>(), n->cg_p.as<double>(), n->p32.as<float>(), n->cgstate.as<CgState>(),
                       n->cgscratch.as<double>(), st), 1);
  }
  CKL(launch_cg_prepare_shs(P, n->cg_x.as<double>(), n->x32.as<float>(), st), 1);
  RET(pass_backward(n, b, MRL_MODE_FVP, nullptr, 0, n->x32.as<float>(), 0.0, n->out32.as<float>(),
                    n->out64.as<double>(), st));
  CKL(launch_cg_finish(P, n->out32.as<float>(), cfg->cg_damping, cfg->max_kl, n->g32.as<float>(),
                       n->cg_x.as<double>(), n->fullstep.as<double>(), n->cgstate.as<CgState>(), st), 1);
  CK(cudaStreamSynchronize(st));   // h_scal / h_cg (first snapshot) are valid now
  RET(comm_ok(n));
  const double before[3] = {-n->h_scal[0], n->h_scal[1], n->h_scal[2]};
  const double gmax = n->h_cg->gmax;
  double after[3] = {before[0], before[1], before[2]};
  int skipped = 0, success = 0, accepted = -1, cg_run = 0;
  if (!(gmax > 1e-8)) {            // np.allclose(g, 0): |g_i| <= atol=1e-8  (trpo.py:102)
    skipped = 1;
  } else {
    RET(d2h_sync(n->h_cg, n->cgstate.p, sizeof(CgState), st));
    cg_run = n->h_cg->iters;
    const double rate = n->h_cg->expected_rate;
    const double fval = before[0];  // f(x) re-evaluates the same graph at the same theta (trpo.py:147)
    for (int k = 0; k < cfg->max_backtracks; ++k) {
      const double stepfrac = ldexp(1.0, -k);
      CKL(launch_ls_candidate(P, n->theta_prev.as<float>(), n->fullstep.as<double>(), stepfrac,
                              n->theta.as<float>(), st), 1);
      RET(repack(n, st));
      RET(pass_forward(n, b, true, false, nullptr, st));
      loss_passes++;
      RET(d2h_sync(n->h_scal, n->scal.p, 32, st));
      const double newf = -n->h_scal[0];
      const double actual = fval - newf, expected = rate * stepfrac, ratio = actual / expected;
      if (ratio > cfg->accept_ratio && actual > 0) {
        success = 1;
        accepted = k;
        after[0] = newf; after[1] = n->h_scal[1]; after[2] = n->h_scal[2];
        break;
      }
    }
    RET(comm_ok(n));
    if (!success) {                // rollback (trpo.py:133 with theta = x)
      CK(cudaMemcpyAsync(n->theta.p, n->theta_prev.p, (size_t)P * 4, cudaMemcpyDeviceToDevice, st));
      RET(repack(n, st));
    }
    n->last_valid = true;
  }
  stats[0] = before[0]; stats[1] = after[0];
  stats[2] = before[1]; stats[3] = after[1];
  stats[4] = before[2]; stats[5] = after[2];
  if (info) {
    info[0] = skipped; info[1] = success; info[2] = accepted; info[3] = cg_run;
    info[4] = skipped ? 0 : cg_run + 1;   // Fvp evaluations the reference would make; launches after an early break are no-ops
    info[5] = loss_passes;
  }
  return 0;
}

extern "C" int mrl_net_get_trpo_vectors(mrl_net* n, double* stepdir, double* fullstep, double* scalars) {
  if (!n || !n->last_valid) return fail("mrl_net_get_trpo_vectors: no completed step");
  CK(cudaSetDevice(n->device));
  const size_t bytes = (size_t)n->g.P * 8;
  if (stepdir) CK(cudaMemcpy(stepdir, n->cg_x.p, bytes, cudaMemcpyDeviceToHost));
  if (fullstep) CK(cudaMemcpy(fullstep, n->fullstep.p, bytes, cudaMemcpyDeviceToHost));
  if (scalars) {
    CK(cudaMemcpy(n->h_cg, n->cgstate.p, sizeof(CgState), cudaMemcpyDeviceToHost));
    scalars[0] = n->h_cg->shs; scalars[1] = n->h_cg->lm; scalars[2] = n->h_cg->expected_rate;
    scalars[3] = n->h_cg->rdotr;
  }
  return 0;
}

// ======================================================================== device-resident rollouts (rollout.cu)
struct mrl_rollout {
  int device = 0, env = 0, N = 0, T = 0, d0 = 0, sd = 0, dout = 0, pd = 0, head = 0;   // pd: prob row width
  DevBuf s_obs, s_state, s_prob, s_act, s_rew, lengths, term, headbuf, body, filt, returns, thetas;
  double* h_head = nullptr;      // pinned: header, then lengths int32[N], terminated int32[N]
  double* h_filt = nullptr;      // pinned: incoming filter states
  char* h_body = nullptr;        // pinned: compacted rows of the last round
  size_t h_body_cap = 0;
  long long total = 0;
  int n_round = 0;               // environments of the last round (a population round may run fewer than N)
  int with_states = 0, with_rows = 1;
};
static int ro_head_doubles(int d0) { return 9 + 4 * d0; }
static int ro_act_width(const mrl_rollout* r) { return r->head == MRL_HEAD_CAT ? 1 : r->dout; }
static const char* ro_env_names = "MRL_ENV_CARTPOLE, MRL_ENV_PENDULUM, MRL_ENV_ACROBOT, MRL_ENV_MOUNTAIN_CAR, "
                                  "MRL_ENV_MOUNTAIN_CAR_CONTINUOUS or an id from mrl_rollout_env_compile";

#define RO_USER_MAX_GAUSS 8    // DiagGauss entries of a user environment (per-thread registers of the action draw)
#define RO_USER_MAX_CLASSES 16
#define RO_USER_MAX_STATE 16
extern "C" int mrl_rollout_env_compile(const char* name, const char* source, int ob_dim, int state_dim, int head,
                                       int n_out, int* env_out) {
  const char* who = "mrl_rollout_env_compile";
  if (!name || !source || !env_out) return fail("%s: bad arguments", who);
  if (head != MRL_HEAD_CAT && head != MRL_HEAD_GAUSS)
    return fail("%s: head = %d; a user environment acts through a Categorical (%d) or DiagGauss (%d) head", who, head,
                MRL_HEAD_CAT, MRL_HEAD_GAUSS);
  if (ob_dim < 1 || ob_dim > RO_KMAX_OBS)
    return fail("%s: ob_dim = %d; device rollouts take observations of 1..%d entries (the per-step filter scan "
                "carries the observation entries and the reward)", who, ob_dim, RO_KMAX_OBS);
  if (state_dim < 1 || state_dim > RO_USER_MAX_STATE)
    return fail("%s: state_dim = %d; a user environment's state has 1..%d entries", who, state_dim, RO_USER_MAX_STATE);
  if (head == MRL_HEAD_CAT && (n_out < 1 || n_out > RO_USER_MAX_CLASSES))
    return fail("%s: n_out = %d; a Categorical head of a user environment has 1..%d classes", who, n_out,
                RO_USER_MAX_CLASSES);
  if (head == MRL_HEAD_GAUSS && (n_out < 1 || n_out > RO_USER_MAX_GAUSS))
    return fail("%s: n_out = %d; a DiagGauss head of a user environment has 1..%d entries", who, n_out,
                RO_USER_MAX_GAUSS);
  std::string err;
  if (rollout_user_compile(name, source, ob_dim, state_dim, head, n_out, env_out, &err)) {
    g_err = std::string(who) + ": " + err;
    return 1;
  }
  return 0;
}

extern "C" int mrl_rollout_env_log(int env, char* buf, int len) {
  const std::string* log = rollout_user_log(env);
  if (!log) return fail("mrl_rollout_env_log: %d is not the id of a compiled user environment", env);
  if (!buf || len < 1) return fail("mrl_rollout_env_log: bad arguments");
  const size_t n = log->size() < (size_t)len - 1 ? log->size() : (size_t)len - 1;
  memcpy(buf, log->data(), n);
  buf[n] = '\0';
  return 0;
}

extern "C" int mrl_rollout_max_envs(void) { return RO_MAX_ENVS; }

extern "C" int mrl_rollout_env_info(int env, int* ob_dim, int* state_dim, int* head, int* n_out) {
  int d0, sd, dout, pd;
  const int h = rollout_env_dims(env, &d0, &sd, &dout, &pd);
  if (h < 0) return fail("mrl_rollout_env_info: unknown env %d (%s)", env, ro_env_names);
  if (ob_dim) *ob_dim = d0;
  if (state_dim) *state_dim = sd;
  if (head) *head = h;
  if (n_out) *n_out = dout;
  return 0;
}

extern "C" int mrl_rollout_destroy(mrl_rollout* r) {
  if (!r) return 0;
  cudaSetDevice(r->device);
  DevBuf* bufs[] = {&r->s_obs, &r->s_state, &r->s_prob, &r->s_act, &r->s_rew, &r->lengths, &r->term, &r->headbuf,
                    &r->body, &r->filt, &r->returns, &r->thetas};
  for (DevBuf* d : bufs) d->release();
  if (r->h_head) cudaFreeHost(r->h_head);
  if (r->h_filt) cudaFreeHost(r->h_filt);
  if (r->h_body) cudaFreeHost(r->h_body);
  delete r;
  return 0;
}

extern "C" int mrl_rollout_create(mrl_rollout** out, int device, int env, int n_envs, int timestep_limit) {
  if (!out) return fail("mrl_rollout_create: null output");
  int d0, sd, dout, pd;
  const int head = rollout_env_dims(env, &d0, &sd, &dout, &pd);
  if (head < 0) return fail("mrl_rollout_create: unknown env %d (%s)", env, ro_env_names);
  if (n_envs < 1 || n_envs > RO_MAX_ENVS)
    return fail("mrl_rollout_create: n_envs = %d; the rollout kernel runs 1..%d environments per round", n_envs, RO_MAX_ENVS);
  if (timestep_limit < 1) return fail("mrl_rollout_create: timestep_limit must be >= 1");
  CK(cudaSetDevice(device));
  if (env >= RO_USER_ENV0) {
    std::string err;
    if (rollout_user_load(env, &err)) return fail("mrl_rollout_create: %s", err.c_str());
  }
  mrl_rollout* r = new mrl_rollout();
  r->device = device; r->env = env; r->N = n_envs; r->T = timestep_limit; r->n_round = n_envs;
  r->d0 = d0; r->sd = sd; r->dout = dout; r->pd = pd; r->head = head;
  const size_t rows = (size_t)n_envs * timestep_limit;
  const RolloutLayout lay = rollout_layout((long long)rows, d0, sd, pd, ro_act_width(r), 1);
  cudaError_t e = cudaSuccess;
  auto R = [&](DevBuf& b, size_t bytes) { if (e == cudaSuccess) e = b.reserve(bytes); };
  R(r->s_obs, rows * d0 * 8); R(r->s_state, rows * sd * 8); R(r->s_prob, rows * pd * 4);
  R(r->s_act, rows * ro_act_width(r) * 4); R(r->s_rew, rows * 8); R(r->lengths, (size_t)n_envs * 4); R(r->term, (size_t)n_envs * 4);
  R(r->headbuf, (size_t)ro_head_doubles(d0) * 8); R(r->body, lay.end); R(r->filt, (size_t)(4 + 2 * d0) * 8);
  R(r->returns, (size_t)n_envs * 8);
  const size_t hb = (size_t)ro_head_doubles(d0) * 8 + (size_t)n_envs * 8;
  if (e == cudaSuccess) e = cudaMallocHost(&r->h_head, hb);
  if (e == cudaSuccess) e = cudaMallocHost(&r->h_filt, (size_t)(4 + 2 * d0) * 8);
  if (e != cudaSuccess) {
    mrl_rollout_destroy(r);
    return fail("mrl_rollout_create: %s", cudaGetErrorString(e));
  }
  *out = r;
  return 0;
}

// The net's geometry in the round's arguments: layer widths and the activation rows of the forward in shared memory.
static void ro_net_args(RolloutArgs& a, int L, const int* d) {
  a.L = L;
  int wmax = 1;
  for (int l = 0; l <= L; ++l) {
    a.d[l] = d[l];
    if (l > 0 && l < L && d[l] > wmax) wmax = d[l];
  }
  a.ldh = wmax + 1;                               // odd stride: the rows of one warp fall into distinct banks
  a.rows_chunk = 8192 / a.ldh < 128 ? 8192 / a.ldh : 128;   // 64 KB of activations
}

// Filters in, one launch, and the copies back of a round (mrl_rollout_run, mrl_rollout_run_population).  `a` holds
// the round's shape, net and parameters; `returns` (population rounds) receives the scores on the host.
static int ro_round(mrl_rollout* r, RolloutArgs& a, int act, bool pop, const char* who,
                    const mrl_zfilter_cfg* ob_cfg, double* ob_state, double* ob_pushed,
                    const mrl_zfilter_cfg* rew_cfg, double* rew_state, double* rew_pushed,
                    double* returns, int want_rows, int want_states, long long* n_timesteps, cudaStream_t st) {
  const bool ob_on = ob_cfg && ob_cfg->enabled, rew_on = rew_cfg && rew_cfg->enabled;
  const int d0 = r->d0;
  int n_ctas, threads;
  rollout_shape(a.N, &n_ctas, &a.per_cta, &threads);
  a.ob_on = ob_on; a.rew_on = rew_on;
  a.ob_demean = ob_on && ob_cfg->demean; a.ob_destd = ob_on && ob_cfg->destd; a.ob_clip = ob_on ? ob_cfg->clip : 0.0;
  a.want_rows = want_rows != 0;
  a.filt_in = r->filt.as<double>();
  a.s_obs = r->s_obs.as<double>(); a.s_state = want_states ? r->s_state.as<double>() : nullptr;
  a.s_prob = r->s_prob.as<float>(); a.s_act = r->s_act.p; a.s_rew = r->s_rew.as<double>();
  a.lengths = r->lengths.as<int>(); a.term = r->term.as<int>();
  a.head = r->headbuf.as<double>(); a.body = r->body.as<char>();
  a.returns = r->returns.as<double>();
  const size_t smem = rollout_smem_bytes(a, d0, r->dout, pop);
  int dev_smem = 0;
  CK(cudaDeviceGetAttribute(&dev_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, r->device));
  if (smem + 16384 > (size_t)dev_smem)
    return fail("%s: the rollout kernel needs %zu B of shared memory per CTA, device offers %d", who, smem, dev_smem);
  double* hf = r->h_filt;
  for (int i = 0; i < 4 + 2 * d0; ++i) hf[i] = 0.0;
  if (ob_on) for (int i = 0; i < 1 + 2 * d0; ++i) hf[i] = ob_state[i];
  if (rew_on) for (int i = 0; i < 3; ++i) hf[1 + 2 * d0 + i] = rew_state[i];
  CK(cudaMemcpyAsync(r->filt.p, hf, (size_t)(4 + 2 * d0) * 8, cudaMemcpyHostToDevice, st));
  CKP(PK_ROLLOUT, launch_rollout(a, r->env, act, pop, n_ctas, threads, smem, st), 1);

  // header + lengths + terminated (+ scores), then the collected rows only
  const int nh = ro_head_doubles(d0);
  int* h_len = (int*)(r->h_head + nh);
  CK(cudaMemcpyAsync(r->h_head, r->headbuf.p, (size_t)nh * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(h_len, r->lengths.p, (size_t)a.N * 4, cudaMemcpyDeviceToHost, st));
  CK(cudaMemcpyAsync(h_len + a.N, r->term.p, (size_t)a.N * 4, cudaMemcpyDeviceToHost, st));
  if (returns) CK(cudaMemcpyAsync(returns, r->returns.p, (size_t)a.N * 8, cudaMemcpyDeviceToHost, st));
  CK(cudaStreamSynchronize(st));
  const double* h = r->h_head;
  r->total = (long long)h[0];
  r->n_round = a.N;
  r->with_rows = want_rows != 0;
  r->with_states = want_rows && want_states;
  if (r->with_rows) {
    const RolloutLayout lay = rollout_layout(r->total, d0, r->sd, r->pd, ro_act_width(r), r->with_states);
    if (lay.end > r->h_body_cap) {
      if (r->h_body) cudaFreeHost(r->h_body);
      r->h_body = nullptr;
      r->h_body_cap = 0;
      CK(cudaMallocHost(&r->h_body, lay.end + lay.end / 4 + 256));
      r->h_body_cap = lay.end + lay.end / 4 + 256;
    }
    if (lay.end) CK(cudaMemcpyAsync(r->h_body, r->body.p, lay.end, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
  }
  if (ob_on) {
    for (int i = 0; i < 1 + 2 * d0; ++i) ob_state[i] = h[1 + i];
    if (ob_pushed) for (int i = 0; i < 1 + 2 * d0; ++i) ob_pushed[i] = h[2 + 2 * d0 + i];
  }
  if (rew_on) {
    for (int i = 0; i < 3; ++i) rew_state[i] = h[3 + 4 * d0 + i];
    if (rew_pushed) for (int i = 0; i < 3; ++i) rew_pushed[i] = h[6 + 4 * d0 + i];
  }
  *n_timesteps = r->total;
  return 0;
}

static const char* ro_env_name(const mrl_rollout* r) {
  switch (r->env) {
    case MRL_ENV_CARTPOLE: return "CartPole";
    case MRL_ENV_PENDULUM: return "Pendulum";
    case MRL_ENV_ACROBOT: return "Acrobot";
    case MRL_ENV_MOUNTAIN_CAR: return "MountainCar";
    case MRL_ENV_MOUNTAIN_CAR_CONTINUOUS: return "MountainCarContinuous";
    default: return rollout_user_name(r->env);
  }
}

extern "C" int mrl_rollout_run(mrl_rollout* r, mrl_net* policy, unsigned long long seed, int stochastic,
                               const mrl_zfilter_cfg* ob_cfg, double* ob_state, double* ob_pushed,
                               const mrl_zfilter_cfg* rew_cfg, double* rew_state, double* rew_pushed,
                               int want_states, long long* n_timesteps, void* stream) {
  if (!r || !policy || !n_timesteps) return fail("mrl_rollout_run: bad arguments");
  const bool ob_on = ob_cfg && ob_cfg->enabled, rew_on = rew_cfg && rew_cfg->enabled;
  if ((ob_on && !ob_state) || (rew_on && !rew_state)) return fail("mrl_rollout_run: an enabled filter needs its state");
  const NetGeom& g = policy->g;
  const char* env_name = ro_env_name(r);
  if (policy->device != r->device)
    return fail("mrl_rollout_run: the policy lives on device %d, the rollouts on device %d", policy->device, r->device);
  if (g.d[0] != r->d0)
    return fail("mrl_rollout_run: %s observations have %d entries, the policy takes %d", env_name, r->d0, g.d[0]);
  if (g.head != r->head || g.d[g.L] != r->dout)
    return fail("mrl_rollout_run: %s needs a %s head with %d outputs (the policy has a %s head with %d)", env_name,
                r->head == MRL_HEAD_CAT ? "Categorical" : "DiagGauss", r->dout,
                g.head == MRL_HEAD_CAT ? "Categorical" : (g.head == MRL_HEAD_GAUSS ? "DiagGauss" : "value"), g.d[g.L]);
  CK(cudaSetDevice(r->device));
  RolloutArgs a = {};
  a.N = r->N; a.T = r->T;
  ro_net_args(a, g.L, g.d);
  a.P = g.P;
  a.w_floats = (size_t)g.P * 4 <= 128 * 1024 ? g.P : 0;
  a.theta = policy->theta.as<float>();
  a.seed = seed;
  a.stochastic = stochastic != 0;
  return ro_round(r, a, g.act, false, "mrl_rollout_run", ob_cfg, ob_state, ob_pushed, rew_cfg, rew_state, rew_pushed,
                  nullptr, 1, want_states, n_timesteps, (cudaStream_t)stream);
}

extern "C" int mrl_rollout_run_population(mrl_rollout* r, int n_layers, const int* dims, int activation,
                                          const float* thetas, long long ld_theta, int theta_loc, int n_members,
                                          unsigned long long seed,
                                          const mrl_zfilter_cfg* ob_cfg, double* ob_state, double* ob_pushed,
                                          const mrl_zfilter_cfg* rew_cfg, double* rew_state, double* rew_pushed,
                                          double* returns, int want_rows, int want_states, long long* n_timesteps,
                                          void* stream) {
  const char* who = "mrl_rollout_run_population";
  if (!r || !dims || !thetas || !returns || !n_timesteps) return fail("%s: bad arguments", who);
  const bool ob_on = ob_cfg && ob_cfg->enabled, rew_on = rew_cfg && rew_cfg->enabled;
  if ((ob_on && !ob_state) || (rew_on && !rew_state)) return fail("%s: an enabled filter needs its state", who);
  if (want_states && !want_rows) return fail("%s: want_states = 1 needs want_rows = 1", who);
  if (n_layers < 1 || n_layers > MRL_MAX_LAYERS)
    return fail("%s: n_layers = %d; the rollout kernel runs 1..%d layers", who, n_layers, MRL_MAX_LAYERS);
  const char* env_name = ro_env_name(r);
  if (dims[0] != r->d0) return fail("%s: %s observations have %d entries, dims[0] = %d", who, env_name, r->d0, dims[0]);
  if (dims[n_layers] != r->dout)
    return fail("%s: %s actions take %d outputs, dims[%d] = %d", who, env_name, r->dout, n_layers, dims[n_layers]);
  long long P = 0;
  for (int l = 1; l <= n_layers; ++l) {
    if (dims[l] < 1 || dims[l] > 256) return fail("%s: dims[%d] = %d; widths must be in 1..256", who, l, dims[l]);
    P += (long long)dims[l - 1] * dims[l] + dims[l];
  }
  if (activation != MRL_ACT_TANH && activation != MRL_ACT_RELU && activation != MRL_ACT_SIGMOID)
    return fail("%s: unknown activation %d (0 tanh, 1 relu, 2 sigmoid)", who, activation);
  if (ld_theta < P) return fail("%s: ld_theta = %lld is smaller than the %lld Dense parameters", who, ld_theta, P);
  if (n_members < 1 || n_members > r->N)
    return fail("%s: n_members = %d; the handle runs 1..%d environments", who, n_members, r->N);
  if (theta_loc != MRL_HOST && theta_loc != MRL_DEVICE) return fail("%s: theta_loc = %d (MRL_HOST or MRL_DEVICE)", who, theta_loc);
  CK(cudaSetDevice(r->device));
  cudaStream_t st = (cudaStream_t)stream;
  const float* th = thetas;
  if (theta_loc == MRL_HOST) {
    const size_t bytes = (size_t)n_members * (size_t)ld_theta * 4;
    CK(r->thetas.reserve(bytes));
    CK(cudaMemcpyAsync(r->thetas.p, thetas, bytes, cudaMemcpyHostToDevice, st));
    th = r->thetas.as<float>();
  } else {
    cudaPointerAttributes pa;
    if (cudaPointerGetAttributes(&pa, thetas) != cudaSuccess) {
      cudaGetLastError();
      pa.type = cudaMemoryTypeUnregistered;
    }
    if ((pa.type != cudaMemoryTypeDevice && pa.type != cudaMemoryTypeManaged) || pa.device != r->device)
      return fail("%s: theta_loc = MRL_DEVICE but thetas is not device memory of device %d", who, r->device);
  }
  RolloutArgs a = {};
  a.N = n_members; a.T = r->T;
  ro_net_args(a, n_layers, dims);
  a.P = (int)P;
  a.w_floats = 0;                                 // each environment reads its own theta through L2
  a.theta = th;
  a.ld_theta = ld_theta;
  a.seed = seed;
  return ro_round(r, a, activation, true, who, ob_cfg, ob_state, ob_pushed, rew_cfg, rew_state, rew_pushed,
                  returns, want_rows, want_states, n_timesteps, st);
}

extern "C" int mrl_rollout_read(mrl_rollout* r, int* lengths, unsigned char* terminated, double* obs, void* act,
                                float* prob, double* reward, double* states) {
  if (!r) return fail("mrl_rollout_read: null handle");
  if (!r->with_rows && (obs || act || prob || reward || states))
    return fail("mrl_rollout_read: the last round did not record rows (want_rows = 0); only lengths and terminated");
  if (states && !r->with_states) return fail("mrl_rollout_read: the last round did not record states (want_states = 0)");
  const int N = r->n_round;
  const int* h_len = (const int*)(r->h_head + ro_head_doubles(r->d0));
  if (lengths) memcpy(lengths, h_len, (size_t)N * 4);
  if (terminated) for (int i = 0; i < N; ++i) terminated[i] = (unsigned char)h_len[N + i];
  const long long n = r->total;
  const RolloutLayout lay = rollout_layout(n, r->d0, r->sd, r->pd, ro_act_width(r), r->with_states);
  if (obs) memcpy(obs, r->h_body + lay.obs, (size_t)n * r->d0 * 8);
  if (reward) memcpy(reward, r->h_body + lay.rew, (size_t)n * 8);
  if (states) memcpy(states, r->h_body + lay.state, (size_t)n * r->sd * 8);
  if (prob) memcpy(prob, r->h_body + lay.prob, (size_t)n * r->pd * 4);
  if (act) memcpy(act, r->h_body + lay.act, (size_t)n * ro_act_width(r) * 4);
  return 0;
}

// ======================================================================== cross-entropy search (cem_search.cu)
struct mrl_cem_search {
  int device = 0, P = 0, M = 0, cur = 0;          // cur: the buffer of each pair that holds the current mean / var
  long long ld = 0;
  unsigned long long seed = 0;                    // of the last draw: the refit recomputes its rows
  bool drawn = false;
  DevBuf mean[2], var[2], dev, rows, scores, order;
};

// ptr must be device memory of `device` when loc == MRL_DEVICE
static int cs_check_loc(const char* who, const char* what, const void* ptr, int loc, int device) {
  if (loc != MRL_HOST && loc != MRL_DEVICE) return fail("%s: loc = %d (MRL_HOST or MRL_DEVICE)", who, loc);
  if (loc == MRL_HOST) return 0;
  cudaPointerAttributes pa;
  if (cudaPointerGetAttributes(&pa, ptr) != cudaSuccess) {
    cudaGetLastError();
    pa.type = cudaMemoryTypeUnregistered;
  }
  if ((pa.type != cudaMemoryTypeDevice && pa.type != cudaMemoryTypeManaged) || pa.device != device)
    return fail("%s: loc = MRL_DEVICE but %s is not device memory of device %d", who, what, device);
  return 0;
}

extern "C" int mrl_cem_search_destroy(mrl_cem_search* s) {
  if (!s) return 0;
  cudaSetDevice(s->device);
  DevBuf* bufs[] = {&s->mean[0], &s->mean[1], &s->var[0], &s->var[1], &s->dev, &s->rows, &s->scores, &s->order};
  for (DevBuf* d : bufs) d->release();
  delete s;
  return 0;
}

extern "C" int mrl_cem_search_create(mrl_cem_search** out, int device, long long P, int M, long long ld) {
  const char* who = "mrl_cem_search_create";
  if (!out) return fail("%s: null output", who);
  if (P < 1 || P > (1LL << 30)) return fail("%s: P = %lld; the search holds 1..%lld parameters", who, P, 1LL << 30);
  if (M < 1 || M > RO_MAX_ENVS)
    return fail("%s: M = %d; a generation is one rollout round of 1..%d members", who, M, RO_MAX_ENVS);
  if (ld < P || ld % 4) return fail("%s: ld = %lld; rows need ld >= P = %lld and a multiple of 4 (16 B)", who, ld, P);
  CK(cudaSetDevice(device));
  mrl_cem_search* s = new mrl_cem_search();
  s->device = device; s->P = (int)P; s->M = M; s->ld = ld;
  cudaError_t e = cudaSuccess;
  auto R = [&](DevBuf& b, size_t bytes) { if (e == cudaSuccess) e = b.reserve(bytes); };
  R(s->mean[0], P * 8); R(s->mean[1], P * 8); R(s->var[0], P * 8); R(s->var[1], P * 8); R(s->dev, P * 8);
  R(s->rows, (size_t)M * ld * 4); R(s->scores, (size_t)M * 8); R(s->order, (size_t)M * 4);
  if (e == cudaSuccess) e = cudaMemset(s->rows.p, 0, (size_t)M * ld * 4);     // the padding columns stay 0
  if (e != cudaSuccess) {
    mrl_cem_search_destroy(s);
    return fail("%s: %s", who, cudaGetErrorString(e));
  }
  *out = s;
  return 0;
}

// which: 0 mean, 1 var; to_lib: caller -> library
static int cs_copy(mrl_cem_search* s, int which, bool to_lib, void* x, int loc, void* stream, const char* who) {
  if (!s || !x) return fail("%s: bad arguments", who);
  RET(cs_check_loc(who, which ? "var" : "mean", x, loc, s->device));
  CK(cudaSetDevice(s->device));
  cudaStream_t st = (cudaStream_t)stream;
  void* lib = (which ? s->var : s->mean)[s->cur].p;
  const cudaMemcpyKind kind = loc == MRL_HOST ? (to_lib ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToHost)
                                              : cudaMemcpyDeviceToDevice;
  CK(cudaMemcpyAsync(to_lib ? lib : x, to_lib ? x : lib, (size_t)s->P * 8, kind, st));
  if (loc == MRL_HOST) CK(cudaStreamSynchronize(st));
  if (to_lib) s->drawn = false;                   // the rows of the last draw no longer follow from mean and dev
  return 0;
}
extern "C" int mrl_cem_search_set_mean(mrl_cem_search* s, const double* mean, int loc, void* stream) {
  return cs_copy(s, 0, true, (void*)mean, loc, stream, "mrl_cem_search_set_mean");
}
extern "C" int mrl_cem_search_set_var(mrl_cem_search* s, const double* var, int loc, void* stream) {
  return cs_copy(s, 1, true, (void*)var, loc, stream, "mrl_cem_search_set_var");
}
extern "C" int mrl_cem_search_get_mean(mrl_cem_search* s, double* mean, int loc, void* stream) {
  return cs_copy(s, 0, false, mean, loc, stream, "mrl_cem_search_get_mean");
}
extern "C" int mrl_cem_search_get_var(mrl_cem_search* s, double* var, int loc, void* stream) {
  return cs_copy(s, 1, false, var, loc, stream, "mrl_cem_search_get_var");
}

extern "C" int mrl_cem_search_draw(mrl_cem_search* s, unsigned long long seed, double extra_var, double noise_left,
                                   double* dev_out, int loc, void* stream) {
  const char* who = "mrl_cem_search_draw";
  if (!s) return fail("%s: null handle", who);
  if (dev_out) RET(cs_check_loc(who, "dev_out", dev_out, loc, s->device));
  CK(cudaSetDevice(s->device));
  cudaStream_t st = (cudaStream_t)stream;
  CKP(PK_CEM_SEARCH, launch_cem_draw(s->mean[s->cur].as<double>(), s->var[s->cur].as<double>(), s->dev.as<double>(),
                                     s->rows.as<float>(), s->P, s->M, s->ld, extra_var, noise_left, seed, st), 1);
  s->seed = seed;
  s->drawn = true;
  if (dev_out) {
    CK(cudaMemcpyAsync(dev_out, s->dev.p, (size_t)s->P * 8,
                       loc == MRL_HOST ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, st));
    if (loc == MRL_HOST) CK(cudaStreamSynchronize(st));
  }
  return 0;
}

extern "C" int mrl_cem_search_rows(mrl_cem_search* s, float** rows, long long* ld) {
  if (!s || !rows || !ld) return fail("mrl_cem_search_rows: bad arguments");
  *rows = s->rows.as<float>();
  *ld = s->ld;
  return 0;
}

extern "C" int mrl_cem_search_refit(mrl_cem_search* s, const double* scores, int loc, int keep, void* stream) {
  const char* who = "mrl_cem_search_refit";
  if (!s || !scores) return fail("%s: bad arguments", who);
  if (keep < 0) return fail("%s: keep = %d is negative (elite_frac < 0)", who, keep);
  if (!s->drawn) return fail("%s: no generation has been drawn (mrl_cem_search_draw)", who);
  RET(cs_check_loc(who, "scores", scores, loc, s->device));
  CK(cudaSetDevice(s->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int n = (keep == 0 || keep > s->M) ? s->M : keep;      // np.argsort(scores)[-keep:]: [-0:] is every member
  const double* sc = scores;
  if (loc == MRL_HOST) {
    CK(cudaMemcpyAsync(s->scores.p, scores, (size_t)s->M * 8, cudaMemcpyHostToDevice, st));
    sc = s->scores.as<double>();
  }
  const int nxt = s->cur ^ 1;
  CKP(PK_CEM_SEARCH, launch_cem_rank_refit(sc, s->M, n, s->order.as<int>(), s->mean[s->cur].as<double>(),
                                           s->dev.as<double>(), s->P, s->seed, s->mean[nxt].as<double>(),
                                           s->var[nxt].as<double>(), st), 2);
  s->cur = nxt;
  return 0;
}
