/* mrl_b200.h - C ABI of the B200-native modular_rl policy-update path.
 *
 * The reference (ddlau/modular_rl) has no FFI: its hot path is three compiled Theano
 * functions per updater plus scipy scans, called from Python.  Each entry point below
 * replaces one of those call sites; citations are file:line under /root/reference.
 * INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; mrl_last_error() gives the
 *     message for the calling thread.  No exceptions cross the ABI.  Soft failures of the
 *     algorithm (zero gradient, line-search failure) are reported as output flags, not errors.
 *   - `loc` says where a caller buffer lives: MRL_HOST (pageable or pinned) or MRL_DEVICE.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).  Calls enqueue on it;
 *     only functions that return scalars to the host synchronise it.
 *   - caller memory is borrowed for the duration of the call and never freed by the library.
 *   - one mrl_net / mrl_batch belongs to one (process, GPU).
 */
#ifndef MRL_B200_H
#define MRL_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define MRL_HOST 0
#define MRL_DEVICE 1
/* dtypes of caller arrays */
#define MRL_F32 0
#define MRL_F64 1
#define MRL_I32 2
#define MRL_I64 3
/* distribution heads: DiagGauss (core.py:402-438), Categorical (core.py:339-365), scalar value (agentzoo.py:53-59) */
#define MRL_GAUSS 0
#define MRL_CATEGORICAL 1
#define MRL_VALUE 2
/* hidden activations (Keras names, agentzoo.py:20-23) */
#define MRL_TANH 0
#define MRL_RELU 1
#define MRL_SIGMOID 2

typedef struct mrl_net mrl_net;
typedef struct mrl_batch mrl_batch;
typedef struct mrl_comm mrl_comm;

const char* mrl_last_error(void);
int mrl_version(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
long long mrl_launch_count(void);

/* measurement hooks (bench.py): per-kernel-class CUDA-event timing on the launching stream, and the FP32
 * FMA peak of the device.  mrl_profile_read synchronises the device; arrays have mrl_profile_kinds() entries. */
int mrl_profile_enable(int on);
int mrl_profile_kinds(void);
const char* mrl_profile_kind_name(int kind);
int mrl_profile_read(double* ms_out, long long* count_out);
int mrl_measure_fp32_tflops(int device, double* tflops_out);
/* measured mma.sync m16n8k8 TF32 throughput (dense TFLOP/s): the pipe of the register-chain kernels */
int mrl_measure_mma_tf32_tflops(int device, double* tflops_out);
/* measured tcgen05.mma kind::tf32 throughput (dense TFLOP/s, TS mode, M = 128, N = 128): the pipe of the layer-1 GEMMs
 * and of the Fisher-vector chain (mlp_l1_tc.cu, mlp_fvp_tc.cu); every algorithmic product costs three of these */
int mrl_measure_tcgen05_tf32_tflops(int device, double* tflops_out);

/* ---------------------------------------------------------------- batch (paths, flattened)
 * Replaces the `concat([path[k] for path in paths])` host copies of trpo.py:74-77,
 * ppo.py:61-64, core.py:653-654 and the per-call numpy->Theano downcast (keras_theano_setup.py:9). */
int mrl_batch_create(mrl_batch** out, int device, int ob_dim, int with_time_feature);
int mrl_batch_destroy(mrl_batch* b);
/* observations [N x ob_dim], row-major with leading dimension ld (elements) */
int mrl_batch_set_obs(mrl_batch* b, const void* ob, int dtype, long long ld, long long N, int loc, void* stream);
/* CSR trajectory structure: offsets int64[n_paths+1] (offsets[n_paths] == N), terminated uint8[n_paths].
 * Also materialises NnVf.preproc's feature t/timestep_limit (core.py:659-660) when the batch was
 * created with_time_feature. */
int mrl_batch_set_paths(mrl_batch* b, const long long* offsets, const unsigned char* terminated, int n_paths,
                        double timestep_limit, int loc, void* stream);
/* action [N] (int, Categorical) or [N x d] (float, DiagGauss); advantage [N]; oldprob [N x K] or [N x 2d]
 * = the args of trpo.py:66.  adv may be NULL to keep the advantages mrl_batch_gae left on the device. */
int mrl_batch_set_policy_inputs(mrl_batch* b, int head, int dout, const void* act, int act_dtype,
                                const void* adv, int adv_dtype, const void* oldprob, int oldprob_dtype,
                                int loc, void* stream);
/* regression target [N] for the value net, already mixed by the caller (core.py:624) */
int mrl_batch_set_vf_target(mrl_batch* b, const void* y, int dtype, int loc, void* stream);
/* target = mixfrac * return + (1 - mixfrac) * ypred_old (core.py:622-624) from what mrl_batch_gae and
 * mrl_net_predict_into_baseline left on the device (ypred_old == the GAE baseline: same theta) */
int mrl_batch_mix_vf_target(mrl_batch* b, double mixfrac, void* stream);
/* re-bind only the advantage column from the float32 advantages mrl_batch_gae left on the device */
int mrl_batch_refresh_advantages(mrl_batch* b, void* stream);
/* global timestep count when the batch is one shard of a data-parallel job (default: local N) */
int mrl_batch_set_global_n(mrl_batch* b, long long n_global);
long long mrl_batch_size(const mrl_batch* b);
/* within-path time index (int32[N]) computed on the device - the bit-exact integer contract */
int mrl_batch_get_time_index(mrl_batch* b, int* out, int loc, void* stream);

/* compute_advantage (core.py:63-105): reward [N]; baseline [N] (NULL: use the values left by
 * mrl_net_predict_into_baseline); writes return/advantage (float64, host or device, may be NULL) and keeps
 * float32 advantages on the device for the policy update.  standardize != 0 applies (adv-mean)/std with
 * population std and no epsilon (core.py:100-105); on a sharded batch the moments are merged over `comm`. */
int mrl_batch_gae(mrl_batch* b, const void* reward, int reward_dtype, const void* baseline, int baseline_dtype,
                  double gamma, double lam, int standardize, mrl_comm* comm, double* ret_out, double* adv_out,
                  int loc, void* stream);

/* ---------------------------------------------------------------- stand-alone scans */
/* misc_utils.discount over a CSR batch + GAE deltas, no batch object (core.py:69-75) */
int mrl_gae(const void* reward, int reward_dtype, const void* baseline, int baseline_dtype,
            const long long* offsets, const unsigned char* terminated, int n_paths, long long N, double gamma,
            double lam, double* ret_out, double* adv_out, int loc, void* stream);
/* in place (x-mean)/std, population std; stats_out[3] = {n, mean, M2} (may be NULL) */
int mrl_standardize(double* x, long long N, double* stats_out, int loc, void* stream);
/* ZFilter over N consecutive samples of dimension d (filters.py:30-38, running_stat.py:9-30): sample t is
 * normalised with running statistics that include samples 0..t and the incoming state {n, M[d], S[d]},
 * which is updated in place (host memory). */
int mrl_zfilter_scan(const void* x, int x_dtype, long long N, int d, double* state_n, double* state_M,
                     double* state_S, int demean, int destd, double clip, void* y, int y_dtype, int loc,
                     void* stream);

/* ---------------------------------------------------------------- network (policy or value MLP)
 * dims[0..n_layers] = input dim, hidden sizes..., output dim (agentzoo.py:25-61).  Parameters are the
 * reference's flat vector: per Dense layer [kernel(in,out) C-order, bias], then logstd (core.py:518-557).
 * Limits: 1..6 layers, every width <= 256, at most 64 outputs, and dims[0] x dims[1] within the tensor-memory
 * budget of the layer-1 kernels (376 inputs allow a first hidden layer of at most 144 units).  A net whose fused
 * layers->=2 kernels do not fit in shared memory (e.g. two hidden layers wider than about 88 units) runs those
 * layers one launch per layer instead; the choice is made here, from the shapes, and no entry point changes. */
int mrl_net_create(mrl_net** out, int device, int n_layers, const int* dims, int head, int activation);
int mrl_net_destroy(mrl_net* n);
long long mrl_net_num_params(const mrl_net* n);
int mrl_net_set_params(mrl_net* n, const void* theta, int dtype, int loc, void* stream); /* SetFromFlat, core.py:526-540 */
int mrl_net_get_params(mrl_net* n, float* theta, int loc, void* stream);                  /* GetFlat, core.py:518-523 */
int mrl_net_set_comm(mrl_net* n, mrl_comm* comm);

/* net output for every timestep of the batch, row-major [N x dout]: means (Gauss; std = exp(logstd) is
 * state independent), softmax probabilities (Categorical) or values.  core.py:270, core.py:608 */
int mrl_net_forward(mrl_net* n, mrl_batch* b, float* out, int loc, void* stream);
/* NnVf.predict over the whole batch, result kept on the device as the GAE baseline (core.py:70) */
int mrl_net_predict_into_baseline(mrl_net* n, mrl_batch* b, void* stream);
/* compute_losses (trpo.py:69, ppo.py:57): out = {surr, kl, ent} */
int mrl_net_losses(mrl_net* n, mrl_batch* b, double out[3], void* stream);
/* compute_policy_gradient (trpo.py:68): g[P]; losses may be NULL */
int mrl_net_policy_gradient(mrl_net* n, mrl_batch* b, float* g, int loc, double losses[3], void* stream);
/* compute_fisher_vector_product (trpo.py:70), WITHOUT the cg_damping term (trpo.py:86-92 adds it) */
int mrl_net_fvp(mrl_net* n, mrl_batch* b, const float* v, float* out, int loc, void* stream);
/* compute_lossgrad (ppo.py:56): pensurr and its flat gradient; losses = {surr, kl, ent} */
int mrl_net_ppo_lossgrad(mrl_net* n, mrl_batch* b, double kl_coeff, double kl_cutoff, int reverse_kl,
                         double* pensurr, double* g, double losses[3], void* stream);
/* NnRegression f_losses / f_lossgrad (core.py:613-617,670-671): losses = {loss, mse, l2}; g may be NULL */
int mrl_net_vf_lossgrad(mrl_net* n, mrl_batch* b, double l2coeff, double losses[3], double* g, void* stream);

/* TrpoUpdater.__call__ after the path concat (trpo.py:80-140): gradient, CG (trpo.py:165-200), step scaling
 * (trpo.py:119-124), backtracking line search (trpo.py:143-159), parameter update or rollback.
 * stats = {surr_before, surr_after, kl_before, kl_after, ent_before, ent_after};
 * info  = {skipped (zero gradient, trpo.py:102), linesearch_success, accepted_backtrack_index,
 *          cg_iterations_run, fvp_calls, loss_passes} */
typedef struct {
  double cg_damping, max_kl, residual_tol, accept_ratio;
  int cg_iters, max_backtracks;
} mrl_trpo_cfg;
int mrl_net_trpo_step(mrl_net* n, mrl_batch* b, const mrl_trpo_cfg* cfg, double stats[6], int info[6],
                      void* stream);
/* debugging / tests: last step direction and full step (float64[P], host) */
int mrl_net_get_trpo_vectors(mrl_net* n, double* stepdir, double* fullstep, double* scalars /* shs,lm,rate,rdotr */);

/* ---------------------------------------------------------------- data-parallel communicator (NCCL)
 * The reference is single-process (core.py:123-124 raises on `parallel`).  Sharding the timestep batch
 * adds one sum over ranks after each batch reduction; see DESIGN.md "Multi-GPU". */
int mrl_comm_unique_id(char id_out[128]);
int mrl_comm_create(mrl_comm** out, const char id[128], int rank, int world, int device);
int mrl_comm_destroy(mrl_comm* c);
int mrl_comm_allreduce_f64(mrl_comm* c, double* buf, long long n, void* stream); /* in place, device memory */
/* Peer-memory transport over NVLink / NVSwitch (CUDA IPC) for vectors of <= max_doubles: every rank exports its
 * receive buffer, the caller all-gathers the 64-byte handles (any side channel; torch.distributed in this repo)
 * and every rank connects.  Afterwards the slab reduce PUSHES each rank's gradient / Fvp partial straight into
 * its peers' buffers and a second kernel sums the slots in rank order (bit-identical on all ranks); NCCL stays
 * the fallback for longer vectors.  All operations on one communicator must be enqueued on one stream. */
int mrl_comm_p2p_export(mrl_comm* c, long long max_doubles, char handle_out[64]);
int mrl_comm_p2p_connect(mrl_comm* c, const char* handles /* [world][64] */);
int mrl_comm_p2p_enable(mrl_comm* c, int on);   /* after every rank connected successfully */

/* ---------------------------------------------------------------- PpoSgdUpdater (ppo.py:115-258), minibatches on the device
 * mrl_batch_gather: dst <- rows idx[0..n) of src (observations + policy side inputs), a device gather from the
 *   resident batch (the reference slices numpy arrays per minibatch, ppo.py:194-199); idx lives where `loc` says.
 * mrl_net_ppo_sgd_step: one `train` call (ppo.py:162-167): penalised-surrogate loss + gradient on the minibatch and
 *   the Adam update of adam_updates (ppo.py:231-258), no host synchronisation; the losses evaluated before the step
 *   are added to a running sum that mrl_net_ppo_sgd_read returns as a mean (and resets). */
int mrl_batch_gather(mrl_batch* dst, const mrl_batch* src, const int* idx, int n, int loc, void* stream);
int mrl_net_ppo_sgd_step(mrl_net* net, mrl_batch* minibatch, double kl_coeff, double kl_cutoff, int reverse_kl,
                         double stepsize, double beta1, double beta2, double epsilon, void* stream);
int mrl_net_ppo_sgd_read(mrl_net* net, double losses[3], long long* count, void* stream);
int mrl_net_adam_reset(mrl_net* net, void* stream);

/* ---------------------------------------------------------------- PPO with the clipped surrogate objective
 * L = -(1/N) sum_t min(r_t A_t, clip(r_t, 1 - clip_eps, 1 + clip_eps) A_t),  r_t = pi(a_t | s_t) / pi_old(a_t | s_t),
 * pi_old = the prob rows bound with mrl_batch_set_policy_inputs.  A row carries the surrogate's gradient unless
 * (A > 0 and r > 1 + clip_eps) or (A < 0 and r < 1 - clip_eps); at r = 1 +- clip_eps it does.  clip_eps > 0, +inf
 * means no clipping; a value net, NULL handles and clip_eps <= 0 or NaN are rejected.
 * mrl_net_ppo_clip_lossgrad: a full-batch pass: losses = {surr = L, kl = KL[old, new], ent, clipfrac = the fraction of
 *   rows with r outside [1 - clip_eps, 1 + clip_eps]} (may be NULL); g != NULL: dL/dtheta, float64 [P] (host), summed
 *   over the ranks of the net's communicator.  Synchronises `stream`.
 * mrl_net_ppo_clip_sgd_step: one minibatch step: the clipped gradient on the minibatch and the Adam update of
 *   mrl_net_ppo_sgd_step, on the same moments and step counter (mrl_net_adam_reset restarts them); no host
 *   synchronisation. */
int mrl_net_ppo_clip_lossgrad(mrl_net* net, mrl_batch* b, double clip_eps, double* g, double losses[4], void* stream);
int mrl_net_ppo_clip_sgd_step(mrl_net* net, mrl_batch* minibatch, double clip_eps, double stepsize, double beta1,
                              double beta2, double epsilon, void* stream);

/* ---------------------------------------------------------------- population forward (cross-entropy method)
 * cem.py:43-44 scores every candidate theta of an iteration by one rollout, one candidate at a time; this entry point
 * evaluates the net of ALL candidates at once: member m has its own flat theta (Dense kernels and biases in the
 * reference's order, no logstd; row stride ld_theta) and its own observation; out[m] is the raw output of the linear
 * last layer (agentzoo.py:63-81).  thetas / obs / out live where `loc` says. */
int mrl_population_forward(int device, int n_layers, const int* dims, int activation, const float* thetas,
                           long long ld_theta, const float* obs, int n_members, float* out, int loc, void* stream);

/* ---------------------------------------------------------------- device-resident rollouts (core.py:182-221)
 * The rollout loop of the built-in environments (modular_rl_b200/envs.py) on the device: one launch runs one ROUND,
 * n_envs environments from reset until every episode has ended or reached timestep_limit, in the lockstep order of
 * core.rollouts_vectorized: per step the observation ZFilter over the live environments in index order, the policy
 * forward on the net's parameters in place, the action draw, the float64 dynamics of envs.py and the reward ZFilter
 * statistics.  Resets and action noise come from Philox4x32-10 keyed by `seed` (DESIGN.md "Device rollouts").
 *   Environments (observation entries, action head, prob row width, state layout):
 *     MRL_ENV_CARTPOLE                 CartPole-v0               4, Categorical 2, 2, (x, x_dot, theta, theta_dot)
 *     MRL_ENV_PENDULUM                 Pendulum-v0               3, DiagGauss d = 1, 2, (theta, theta_dot)
 *     MRL_ENV_ACROBOT                  Acrobot-v1                6, Categorical 3, 3, (theta1, theta2, dtheta1, dtheta2)
 *     MRL_ENV_MOUNTAIN_CAR             MountainCar-v0            2, Categorical 3, 3, (position, velocity)
 *     MRL_ENV_MOUNTAIN_CAR_CONTINUOUS  MountainCarContinuous-v0  2, DiagGauss d = 1, 2, (position, velocity)
 *     The prob row holds K probabilities for a Categorical head with K outputs and [mean, std] (2d) for DiagGauss.
 *   mrl_rollout_env_info: the shapes of `env` above (host code, no device needed): observation entries, state
 *     entries, head (MRL_CATEGORICAL / MRL_GAUSS) and the policy's outputs.  Fails for an unknown env.
 *   mrl_rollout_create: one of the environments above; 1 <= n_envs <= mrl_rollout_max_envs().  Allocates the staging
 *     rows of a round, n_envs x timestep_limit rows of (observation, state, prob, action, reward), and a compacted
 *     output buffer of as many rows.  At 4096 environments that is about 0.2 GB each for Acrobot (500 steps, 104 B a
 *     row) and for MountainCarContinuous (999 steps, 52 B a row), computed from the row sizes.
 *   mrl_rollout_run: `policy` must live on the handle's device, take the environment's observation and end in its
 *     action head (the table above).  A NULL filter cfg or
 *     enabled == 0 is the identity.  ob_state = {n, M[ob_dim], S[ob_dim]} and rew_state = {n, M, S} (host) are read and
 *     replaced by the states after the round; *_pushed (may be NULL) receive the statistics of this round's samples
 *     alone.  want_states != 0 also records the raw environment state of every step.  Synchronises `stream`;
 *     *n_timesteps = timesteps collected.
 *   mrl_rollout_read: the last round, path-major (episode i = environment i): lengths int32[n_envs],
 *     terminated uint8[n_envs], observation f64 [n x ob_dim] (filtered), action int32 [n] (Categorical) or
 *     f32 [n x d] (DiagGauss), prob f32 [n x prob width] (probabilities or [mean, std]), raw reward f64 [n],
 *     states f64 [n x state_dim] (the state layouts above).  Any pointer may be NULL.  After a
 *     round without rows (mrl_rollout_run_population, want_rows = 0) only lengths and terminated may be non-NULL.
 *   mrl_rollout_run_population: one round in which environment m acts deterministically with its own theta_m (the
 *     cross-entropy method's population, cem.py:43-44,88-91).  n_members <= the handle's n_envs environments run;
 *     thetas [n_members x ld_theta] float32 where `theta_loc` says (MRL_HOST: one copy into a device buffer the handle
 *     keeps; MRL_DEVICE: read in place), each row the Dense kernels and biases of n_layers layers of widths dims[0..]
 *     (1..256) in the reference's flat order, no logstd block, ld_theta >= that count.  The action is taken from the
 *     raw last-layer output: for a Categorical head its argmax (first maximum; a NaN output wins as in numpy), for
 *     DiagGauss the output itself, which the dynamics clip (MountainCarContinuous penalises the unclipped value).
 *     returns[n_members] (host, float64) = the sum of each episode's raw rewards in step order.  Filters as
 *     mrl_rollout_run.  want_rows != 0 records the rows for mrl_rollout_read, the prob row then holding the raw
 *     outputs (Categorical: the K logits; DiagGauss: [mean, 1]); want_states (needs want_rows) the raw states.
 *     Synchronises `stream`; *n_timesteps = timesteps collected.
 *   User environments (ids >= 64) are accepted by every call above wherever an env is; see below. */
#define MRL_ENV_CARTPOLE 0
#define MRL_ENV_PENDULUM 1
#define MRL_ENV_ACROBOT 2
#define MRL_ENV_MOUNTAIN_CAR 3
#define MRL_ENV_MOUNTAIN_CAR_CONTINUOUS 4
typedef struct mrl_rollout mrl_rollout;
typedef struct {
  int enabled, demean, destd;
  double clip;   /* 0: no clipping */
} mrl_zfilter_cfg;
int mrl_rollout_max_envs(void);
int mrl_rollout_env_info(int env, int* ob_dim, int* state_dim, int* head, int* n_out);
int mrl_rollout_create(mrl_rollout** out, int device, int env, int n_envs, int timestep_limit);
int mrl_rollout_destroy(mrl_rollout* r);
int mrl_rollout_run(mrl_rollout* r, mrl_net* policy, unsigned long long seed, int stochastic,
                    const mrl_zfilter_cfg* ob_cfg, double* ob_state, double* ob_pushed,
                    const mrl_zfilter_cfg* rew_cfg, double* rew_state, double* rew_pushed,
                    int want_states, long long* n_timesteps, void* stream);
int mrl_rollout_run_population(mrl_rollout* r, int n_layers, const int* dims, int activation,
                               const float* thetas, long long ld_theta, int theta_loc, int n_members,
                               unsigned long long seed,
                               const mrl_zfilter_cfg* ob_cfg, double* ob_state, double* ob_pushed,
                               const mrl_zfilter_cfg* rew_cfg, double* rew_state, double* rew_pushed,
                               double* returns, int want_rows, int want_states,
                               long long* n_timesteps, void* stream);
int mrl_rollout_read(mrl_rollout* r, int* lengths, unsigned char* terminated, double* obs, void* act, float* prob,
                     double* reward, double* states);

/* ---------------------------------------------------------------- user environments in device rollouts
 * mrl_rollout_env_compile (host code, no device needed): compiles the rollout kernel for an environment given as CUDA
 *   source and returns its id (>= 64) in *env_out.  The library wraps `source` in
 *     template <> struct EnvT<id> { static constexpr int D0 = ob_dim, SD = state_dim, DOUT = n_out, PD = ..., HEAD = head;
 *                                   <source> };
 *   and `source` defines, in float64:
 *     __device__ static void reset(double* s, int env, uint32_t k0, uint32_t k1)   the start state of environment env
 *     __device__ static void obs(const double* s, double* x)                        its observation x[ob_dim]
 *     __device__ static bool step(double* s, int action, const float* a, double* reward)   -> terminated
 *   `action` is the Categorical index, `a` the n_out DiagGauss entries (float32).  reset draws its uniforms with
 *   reset_uniforms(env, block, k0, k1, &u0, &u1): the pair of Philox counter (env, 0, 0, block) in [0, 1).
 *   RO_PI is pi.  head: MRL_CATEGORICAL with 1 <= n_out <= 16 classes, or MRL_GAUSS with 1 <= n_out <= 8 entries;
 *   1 <= ob_dim <= 6 (the per-step filter scan carries the observation entries and the reward); 1 <= state_dim <= 16.
 *   NVRTC (libnvrtc.so.12, opened on first use) compiles the six (activation, population) instances for sm_100a, in
 *   seconds of host time; the same (source, shapes) returns the same id without compiling again.  A compile error
 *   fails with NVRTC's log in mrl_last_error(), its line numbers counted in `source`, whose file name is `name`.
 *   The kernels load at the first mrl_rollout_create of the id.
 * mrl_rollout_env_log: the compiler's report (ptxas registers and spills of the six instances) of a user environment,
 *   NUL-terminated and truncated to len bytes. */
int mrl_rollout_env_compile(const char* name, const char* source, int ob_dim, int state_dim, int head, int n_out,
                            int* env_out);
int mrl_rollout_env_log(int env, char* buf, int len);

/* ---------------------------------------------------------------- cross-entropy search on the device (cem.py:10-50)
 * The diagonal-Gaussian search distribution of the noisy cross-entropy method, resident on the device: the draw of a
 * generation's candidates and the refit of mean and variance to its elite (cem.py:10-50; here modular_rl_b200/cem.py
 * _GaussianSearch.draw / refit) run as kernels, so the candidates never cross to the host.  The normals come from
 * Philox4x32-10 (DESIGN.md 4b "Device search"), not from numpy's generator, so a run differs from the host search.
 *   mrl_cem_search_create: P parameters (the Dense kernels and biases of a DeterministicAgent, no logstd), M members
 *     (1..mrl_rollout_max_envs(): one population round), candidate rows of stride ld floats (ld >= P, a multiple of 4:
 *     16-byte rows, padding columns 0).  Holds mean and var (float64 [P], double-buffered), dev (float64 [P]), the rows
 *     (float32 [M x ld]) and M scores.  Mean and var start unset: set both before the first draw.
 *   mrl_cem_search_set_mean / _set_var / _get_mean / _get_var: float64 [P] where `loc` says (MRL_DEVICE: memory of the
 *     handle's device).  A get to the host synchronises `stream`.  A set discards the last draw (refit needs a new one).
 *   mrl_cem_search_draw: one launch.  dev[j] = sqrt(var[j] + extra_var * noise_left) with _GaussianSearch.draw's
 *     rounding; row m = float32(mean + dev * z_m), z_m the normals of member m under the key `seed` (the generation's
 *     round seed, which run_cem_algorithm also passes to mrl_rollout_run_population).  dev_out (may be NULL) receives
 *     dev where `loc` says; to the host it synchronises `stream`.
 *   mrl_cem_search_rows: the device pointer and stride of the rows, valid until mrl_cem_search_destroy; hand them to
 *     mrl_rollout_run_population with theta_loc = MRL_DEVICE.
 *   mrl_cem_search_refit: scores[M] float64 where `loc` says, of the rows of the last draw.  The elite is the last
 *     `keep` members of a stable ascending sort (np.argsort(scores, kind="stable")[-keep:]: ties go to the higher
 *     index, NaN sorts last); keep == 0 or keep > M selects all M, as numpy's slice does, and keep < 0 is an error.
 *     The new mean and var (two-pass, ddof 0) are those of the elite rows recomputed in float64 from the draw's
 *     counters, summed in ascending (score, index) order.  Two launches, no synchronisation. */
typedef struct mrl_cem_search mrl_cem_search;
int mrl_cem_search_create(mrl_cem_search** out, int device, long long P, int M, long long ld);
int mrl_cem_search_destroy(mrl_cem_search* s);
int mrl_cem_search_set_mean(mrl_cem_search* s, const double* mean, int loc, void* stream);
int mrl_cem_search_set_var(mrl_cem_search* s, const double* var, int loc, void* stream);
int mrl_cem_search_get_mean(mrl_cem_search* s, double* mean, int loc, void* stream);
int mrl_cem_search_get_var(mrl_cem_search* s, double* var, int loc, void* stream);
int mrl_cem_search_draw(mrl_cem_search* s, unsigned long long seed, double extra_var, double noise_left,
                        double* dev_out, int loc, void* stream);
int mrl_cem_search_rows(mrl_cem_search* s, float** rows, long long* ld);
int mrl_cem_search_refit(mrl_cem_search* s, const double* scores, int loc, int keep, void* stream);

#ifdef __cplusplus
}
#endif
#endif
