// Internal launcher declarations shared between the .cu translation units.
#pragma once
#include "common.cuh"

#include <string>

// ---- batch_params.cu
cudaError_t launch_pack_params(const NetGeom& g, const float* theta, float* img, float* WB, cudaStream_t st);
cudaError_t launch_reduce_partials(const NetGeom& g, const float* part1, const float* partm, int n_slabs,
                                   double scale, const float* theta, double l2c2, const float* vflat, double vls,
                                   float* out32, double* out64, const struct P2pPush* push, const struct P2pGather* gather,
                                   cudaStream_t st);
cudaError_t launch_reduce_losses(const double* parts, int n_slabs, double scale, double* out, cudaStream_t st);
cudaError_t launch_pack_tiles(const void* src, int dtype, long long ld, int ncols, int ncols_out, long long N,
                              float* dst, int rows_per_tile, int row_off, int n_tiles, cudaStream_t st);
cudaError_t launch_time_feature(const long long* offsets, int n_paths, long long N, double limit, int col, int* tindex,
                                float* XA, int xa_kgroups, float* XG, int xg_ftiles, cudaStream_t st);

cudaError_t launch_gather_rows(const int* idx, int n, long long n_src, const float* sXA, float* dXA, int xa_kg,
                               const float* sXG, float* dXG, int xg_ft, const float* sAux, float* dAux, int naux,
                               cudaStream_t st);
cudaError_t launch_adam_step(int P, const double* g64, float* theta, float* m, float* v, float a_t, float b1, float b2,
                             float eps, cudaStream_t st);
cudaError_t launch_accum_losses(const double* scal, double* acc, cudaStream_t st);

// ---- mlp_l1_tc.cu  (tcgen05 / TMEM layer-1 GEMMs, 3xTF32)
int l1tc_nu(const NetGeom& g);
size_t l1tc_wb_floats(const NetGeom& g);
bool l1tc_supported(const NetGeom& g);
size_t l1tc_xa_floats(int xa_kgroups, long long n_mtiles);
cudaError_t launch_l1_forward_tc(const NetGeom& g, const float* XA, int xa_kgroups, const float* WB, float* Zt,
                                 int n_tiles, cudaStream_t st);
cudaError_t launch_pack_xa(const void* src, int dtype, long long ld, int ncols, long long N, float* XA, int xa_kgroups,
                           long long n_mtiles, cudaStream_t st);
size_t l1tc_xg_floats(int xg_ftiles, long long n_tiles);
size_t l1tc_dg_floats(const NetGeom& g, long long n_tiles);
cudaError_t launch_pack_xg(const void* src, int dtype, long long ld, int ncols, long long N, float* XG, int xg_ftiles,
                           long long n_tiles, cudaStream_t st);
cudaError_t launch_l1_grad_tc(const NetGeom& g, const float* XG, int xg_ftiles, const float* DG, float* part1,
                              int slab_tiles, int n_tiles, int n_slabs, cudaStream_t st);

// ---- mlp_mid.cu
struct MidFwdArgs {
  const float* img;    // theta image
  const float* Zt;     // layer-1 pre-activations, tile-major [n_tiles][d1][LDT]
  const float* aux;    // side inputs, tile-major [n_tiles][naux][LDT] (nullptr: no losses)
  float* cache;        // activations + head output, tile-major [n_tiles][act_rows][LDT] (nullptr: none)
  float* head_out;     // row-major [N][d_L] head output (mean | probs | value), nullptr: none
  double* loss_part;   // [n_slabs][4]
  long long N;
  int n_tiles, slab_tiles, reverse_kl;
};
struct MidBwdArgs {
  const float* img;    // theta image
  const float* imgv;   // tangent image (Fvp mode)
  const float* Zt;     // Fvp: x . V1
  const float* aux;
  const float* cache;
  const double* coef;  // device: {c_surr, c_kl} (gradient mode)
  float* DG;           // out: delta_1 as the tcgen05 B operand, raw fp32 [tg][khalf][ngroup][8][4]
  int nu;              // padded layer-1 width of DG
  float* partm;        // out: [n_slabs][pmid]
  long long N;
  int n_tiles, slab_tiles, mode, reverse_kl;
};
// clip_eps (PPO clipped objective; a trailing kernel parameter, so that the argument layout of the other instances
// stays as it is): forward, > 0: surr is the clipped objective with this clip range and loss slot 3 the count of
// clipped rows; backward, the clip range of MRL_MODE_GRAD_CLIP.  Policy heads only.
size_t mid_forward_smem(const NetGeom& g);
size_t mid_backward_smem(const NetGeom& g, int mode);
cudaError_t launch_mid_forward(const NetGeom& g, const MidFwdArgs& a, int n_slabs, cudaStream_t st, float clip_eps = 0.f);
cudaError_t launch_mid_backward(const NetGeom& g, const MidBwdArgs& a, int n_slabs, cudaStream_t st, float clip_eps = 0.f);

// ---- mlp_layers.cu  (layer-by-layer path for nets whose mid_* kernels do not fit in shared memory, L >= 2)
// Same contract as launch_mid_*; R0 / R1: ping-pong buffers of layers_ws_floats each (deltas, R-activations).
// *launches: kernels launched.
size_t layers_ws_floats(const NetGeom& g, long long n_tiles);
cudaError_t launch_layers_forward(const NetGeom& g, const MidFwdArgs& a /* cache required */, int n_slabs,
                                  cudaStream_t st, int* launches, float clip_eps = 0.f);
cudaError_t launch_layers_backward(const NetGeom& g, const MidBwdArgs& a, float* R0, float* R1, int n_slabs,
                                   cudaStream_t st, int* launches, float clip_eps = 0.f);

// ---- mlp_chain.cu  (register-resident per-warp chains for the forward and gradient passes)
#define CH_WARPS 12          // backward chain: 12 warps x 16 timesteps = 3 cache tiles per pass
#define CH_NE 3             // weight-gradient entries per warp
#define CH_NTJ 4            // n-tiles (8 columns each) per entry
struct ChainEntry {
  int on;      // 1: active
  int gsoff;   // offset (floats) of the entry's accumulator blocks in shared memory: [n-tile][lane][4]
  int arow0;   // cache feature row of the m-tile's first input feature (off_act[l-1] + 16 mt)
  int amax;    // valid input features from there (d[l-1] - 16 mt; may exceed 16)
  int erow0;   // shared-memory delta row of the first n-tile
  int cnt;     // n-tiles
  int poff;    // offset of the block in the slab partial (off_W[l] + 16 mt ldw + 8 nt0)
  int ldw;
  int nmax;    // valid output features from the first n-tile (d[l] - 8 nt0)
};
struct ChainJobs { ChainEntry e[CH_WARPS][CH_NE]; };
int chain_bwd_shape(const NetGeom& g);   // 0: not covered by an instantiated chain shape
// gradient modes
cudaError_t launch_chain_backward(const NetGeom& g, const MidBwdArgs& a, int n_slabs, cudaStream_t st, float clip_eps = 0.f);
int chain_fwd_shape(const NetGeom& g);
cudaError_t launch_chain_forward(const NetGeom& g, const MidFwdArgs& a, int n_slabs, cudaStream_t st, float clip_eps = 0.f);

// ---- mlp_fvp_tc.cu  (tcgen05 / TMEM Fisher-vector chain of layers >= 2)
struct FvpTcArgs {
  const float* WC;      // chain weight images of theta   (launch_fvp_tc_pack, tangent = 0)
  const float* VC;      // chain weight images of the tangent (tangent = 1)
  const float* vflat;   // the tangent, flat
  const float* img;     // theta image (logstd block)
  const float* Zt;      // x . V_1, tile-major
  const float* cache;   // activation cache of theta
  float* DG;            // out: delta_1 operand of the layer-1 gradient GEMM, raw fp32 [tg][khalf][ngroup][8][4]
  float* partm;         // out: [n_slabs][pmid]
  long long N;
  int n_tiles, slab_tiles /* even */, n_slabs;
};
bool fvp_tc_supported(const NetGeom& g);
size_t fvp_tc_image_floats(const NetGeom& g, int tangent);
// WB1 != nullptr: also the layer-1 tensor-core operand of the same vector (one launch per tangent instead of two)
cudaError_t launch_fvp_tc_pack(const NetGeom& g, const float* src_flat, float* dst, int tangent, cudaStream_t st, float* WB1 = nullptr);
cudaError_t launch_fvp_tc(const NetGeom& g, const FvpTcArgs& a, cudaStream_t st);

// ---- vec_kernels.cu  (CG / line-search vector algebra on device-resident fp64 vectors)
struct CgState {   // device-resident scalars
  double rdotr, pz, alpha, beta, shs, lm, gdots, expected_rate, gmax;
  int done, iters, pad0, pad1;
};
cudaError_t launch_cg_init(int P, const float* g, double* b, double* x, double* r, double* p, float* p32,
                           CgState* s, cudaStream_t st);
#define CG_CTAS 32                              // co-resident CTAs of the CG iteration kernel
#define CG_SCRATCH_DOUBLES (2 * CG_CTAS + 40)   // two partial-sum rows + the grid barrier words
cudaError_t launch_cg_step(int P, const float* z32, double damping, double tol, double* x, double* r, double* p,
                           float* p32, CgState* s, double* scratch /* CG_SCRATCH_DOUBLES, zeroed once */,
                           cudaStream_t st);
cudaError_t launch_cg_prepare_shs(int P, const double* x, float* x32, cudaStream_t st);
cudaError_t launch_cg_finish(int P, const float* z32, double damping, double max_kl, const float* g,
                             const double* x, double* fullstep, CgState* s, cudaStream_t st);
cudaError_t launch_ls_candidate(int P, const float* theta_prev, const double* fullstep, double stepfrac,
                                float* theta_new, cudaStream_t st);
cudaError_t launch_ppo_coef(const double* losses, double kl_coeff, double kl_cutoff, double* coef,
                            double* pen_out, cudaStream_t st);

void cast_f64_f32(const double* x, float* y, long long N, cudaStream_t st);  // api.cu

// ---- scan_kernels.cu
cudaError_t launch_gae(const void* reward, int reward_f64, const void* baseline, int baseline_f64,
                       const long long* offsets, const unsigned char* terminated, int n_paths, long long N,
                       double gamma, double lam, double* ret, double* adv, cudaStream_t st);
#define MRL_MOMENTS_SCRATCH_DOUBLES 1792   // per-block Welford partials of launch_moments (caller-owned)
cudaError_t launch_standardize(double* adv, long long N, double* stats /* n, mean, M2 */, double* scratch,
                               float* adv32, cudaStream_t st);
cudaError_t launch_moments(const double* x, long long N, double* stats, double* scratch, cudaStream_t st);
cudaError_t launch_normalize(double* x, long long N, const double* stats, float* x32, cudaStream_t st);
cudaError_t launch_zfilter_scan(const void* x, int x_f64, long long N, int d, double n0, double* state_dev,
                                int demean, int destd, double clip, void* y, int y_f64, double* scratch,
                                cudaStream_t st);
long long zfilter_scratch_doubles(long long N, int d);

// ---- rollout.cu  (device-resident rollouts, one cluster launch per round; RolloutArgs: kernel_defs.cuh)
// observation entries, state entries, policy outputs, prob row width -> head, -1 for an unknown env
int rollout_env_dims(int env, int* d0, int* sd, int* dout, int* pd);
void rollout_shape(int N, int* n_ctas, int* per_cta, int* threads);
size_t rollout_smem_bytes(const RolloutArgs& a, int d0, int dout, bool pop);
// built-in and user environments; a user environment's kernels must be loaded (rollout_user_load) first
cudaError_t launch_rollout_kernel(const void* f, const RolloutArgs& a, int n_ctas, int threads, size_t smem,
                                  cudaStream_t st);
cudaError_t launch_rollout(const RolloutArgs& a, int env, int act, bool pop, int n_ctas, int threads, size_t smem,
                           cudaStream_t st);

// ---- rollout_user.cu  (user environments: the rollout kernel compiled by NVRTC at run time; host only)
// Compiles (or finds) the environment of snippet `source` with these shapes -> *env >= RO_USER_ENV0; else *err
int rollout_user_compile(const char* name, const char* source, int d0, int sd, int head, int dout, int* env,
                         std::string* err);
const std::string* rollout_user_log(int env);   // the ptxas lines of its six instances; nullptr for an unknown id
// rollout_env_dims for ids >= RO_USER_ENV0; -1 for an id that was never compiled
int rollout_user_dims(int env, int* d0, int* sd, int* dout, int* pd);
const char* rollout_user_name(int env);   // nullptr for an unknown id
// Loads the environment's six kernels (once per process)
int rollout_user_load(int env, std::string* err);
cudaError_t launch_rollout_user(const RolloutArgs& a, int env, int act, bool pop, int n_ctas, int threads,
                                size_t smem, cudaStream_t st);

// ---- cem_search.cu  (device search distribution of the cross-entropy method)
// rows[m][0..P) = float32(mean + dev * z[m]) for m < M, dev[j] = sqrt(var[j] + extra_var * noise_left); ld % 4 == 0
cudaError_t launch_cem_draw(const double* mean, const double* var, double* dev, float* rows, int P, int M,
                            long long ld, double extra_var, double noise_left, unsigned long long seed,
                            cudaStream_t st);
// elite = the last `keep` (1..M) of the stable ascending order of scores[M] (device); mean_out / var_out = their
// float64 mean and variance, rows recomputed from (mean, dev, seed).  order: int32 [M] scratch.  Two launches.
cudaError_t launch_cem_rank_refit(const double* scores, int M, int keep, int* order, const double* mean,
                                  const double* dev, int P, unsigned long long seed, double* mean_out, double* var_out,
                                  cudaStream_t st);
