// Definitions that both compilers take: nvcc, which builds the library, and NVRTC, which compiles the rollout kernel
// of a user environment at run time (rollout_user.cu).  Only device code and NVRTC-clean headers belong here: the
// library embeds this text and hands it to NVRTC.
#pragma once

#define MRL_MAX_LAYERS 6

enum { MRL_HEAD_GAUSS = 0, MRL_HEAD_CAT = 1, MRL_HEAD_VALUE = 2 };
enum { MRL_ACT_TANH = 0, MRL_ACT_RELU = 1, MRL_ACT_SIGMOID = 2 };

template <int ACT>
__device__ __forceinline__ float act_fn(float z) {
  if (ACT == MRL_ACT_TANH) return tanhf(z);
  if (ACT == MRL_ACT_RELU) return fmaxf(z, 0.f);
  return 1.f / (1.f + expf(-z));
}

// ---- device-resident rollouts (rollout_kernel.cuh)
#define RO_MAX_CTAS 8          // CTAs of the round's cluster (the portable cluster size)
#define RO_MAX_THREADS 512     // environments (threads) per CTA
#define RO_MIN_PER_CTA 32      // fewer environments per CTA than this: use fewer CTAs
#define RO_MAX_ENVS (RO_MAX_CTAS * RO_MAX_THREADS)
#define RO_USER_ENV0 64        // environment ids from here on: user environments, compiled at run time
#define RO_KMAX_OBS 6          // observation entries: the per-step scan carries them and the reward (RO_KMAX = 7)
struct RolloutArgs {
  int N, T, per_cta;           // environments, timestep limit, environments per CTA
  int L, d[MRL_MAX_LAYERS + 1], P;
  int w_floats;                // theta floats staged in shared memory (0: read through L2)
  int rows_chunk, ldh;         // forward: rows per chunk, activation row stride (floats)
  const float* theta;          // the policy's flat parameters (reference order), read in place
  unsigned long long seed;
  int stochastic;
  int ob_on, ob_demean, ob_destd, rew_on;
  double ob_clip;
  const double* filt_in;       // (n, M[d0], S[d0]) of the observation filter, then (n, M, S) of the reward filter
  // [T][N] staging rows
  double* s_obs; double* s_state /* nullptr: not recorded */; float* s_prob; void* s_act; double* s_rew;
  int* lengths; int* term;
  double* head;                // total, observation state, its round part, reward state, its round part
  char* body;                  // compacted path-major rows (rollout_layout)
  // population rounds (rollout_kernel<ENV, ACT, true>): environment e acts with theta + e * ld_theta
  long long ld_theta;
  double* returns;             // [N] the sum of each episode's raw rewards, in step order
  int want_rows;               // 0: no staging rows, no compaction (lengths, terminated, returns and the header only)
};
// Byte offsets of the compacted arrays for n timesteps: f64 sections first, so that every section stays aligned
struct RolloutLayout { size_t obs, rew, state, prob, act, end; };
__host__ __device__ inline RolloutLayout rollout_layout(long long n, int d0, int sd, int pd, int ad, int with_states) {
  RolloutLayout o;
  size_t p = 0;
  o.obs = p;   p += (size_t)n * d0 * 8;
  o.rew = p;   p += (size_t)n * 8;
  o.state = p; p += with_states ? (size_t)n * sd * 8 : 0;
  o.prob = p;  p += (size_t)n * pd * 4;
  o.act = p;   p += (size_t)n * ad * 4;     // int32 (Categorical) or float32 [d] (DiagGauss)
  o.end = p;
  return o;
}
