/*
 * cstr_b200.h — C ABI of the B200-native (sm_100a) two-series CSTR hot path.
 *
 * The reference (CHAINNEVERLIU/Pytorch-RL-EnhancedStableBaselines) is 100 % Python and has no
 * FFI of its own; its boundary for this path is three Python protocols (SURVEY.md §8b).  The
 * entry points below are what a ctypes binding placed under those protocols calls; each one
 * names the reference code it replaces.  INTEGRATION.md shows the reference-side stubs.
 *
 * Conventions
 *   - plain C, no torch types: raw DEVICE pointers + sizes + a CUDA stream handle (void*, the
 *     cudaStream_t; NULL = legacy default stream).  The caller owns every buffer.
 *   - every call is asynchronous and stream-ordered; nothing synchronises unless stated.
 *   - return value: 0 = ok; > 0 = cudaError_t of the failed launch/copy; < 0 = argument error
 *     (CSTR_EINVAL...).  cstr_last_error() returns a thread-local message for the last failure.
 *     NaN actions are DATA, handled with the reference's semantics, not errors.
 *   - layouts: state/obs (n,4) float32 (one float4 per reactor: C1,T1,C2,T2 normalised to [-1,1]),
 *     actions (n,2) float32, step_count/episode (n,) int32, rewards (n,) float32,
 *     done/timeout (n,) uint8.  The f64 entry points use double for state/action/reward.
 *   - not re-entrant on the same buffers; one CUDA context per process (one process per GPU).
 */
#ifndef CSTR_B200_H
#define CSTR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CSTR_B200_ABI_VERSION 18

#define CSTR_EINVAL (-1)   /* bad argument (null pointer, negative size, unknown mode) */
#define CSTR_EALIGN (-2)   /* pointer not aligned for the vectorised access the layout implies */

/* math_mode */
#define CSTR_MATH_STRICT 0 /* reference association, no FMA contraction, IEEE division, shared exp  */
#define CSTR_MATH_FAST 1   /* FMA contraction, reciprocal multiplies, ex2.approx (documented tolerance) */

/* init_mode (twoseriescstr.py:91-96) */
#define CSTR_INIT_RANDOM 0
#define CSTR_INIT_STATIC 1

/* Environment parameters shared by all entry points (twoseriescstr.py:63-112). */
typedef struct cstr_env_params {
    uint64_t seed;       /* Philox4x32-10 key of the device RNG (reset draws, exploration noise)   */
    int64_t env_offset;  /* global id of reactor 0 of this shard (multi-GPU: rank * n_per_rank)   */
    double target_c2;    /* TwoSeriesCSTREnv.target_C2 (default 0.20); rounded to float in fp32 mode */
    int32_t max_steps;   /* TwoSeriesCSTREnv.max_steps (400)                                      */
    int32_t init_mode;   /* CSTR_INIT_RANDOM | CSTR_INIT_STATIC                                   */
} cstr_env_params;

int cstr_b200_abi_version(void);
const char *cstr_last_error(void);
/* device properties the host needs for launch/roofline bookkeeping: SM count, SM clock (kHz) */
int cstr_device_info(int *sm_count, int *sm_clock_khz, int *cc_major, int *cc_minor);

/* ---- reset ------------------------------------------------------------------------------------
 * Replaces TwoSeriesCSTREnv.reset / generate_initial_state (twoseriescstr.py:226-269,167-224) for
 * the reactors whose mask byte is non-zero (mask == NULL: all).  Draws 8 unit doubles per reset
 * from Philox (counter = env id, episode; DESIGN.md "RNG"), float64 arithmetic as in the reference,
 * result stored normalised.  static_base: (n,4) double, required for CSTR_INIT_STATIC (quirk Q2:
 * the base state random-walks), may be NULL otherwise.  is_f64: state is double (n,4).             */
int cstr_reset(const cstr_env_params *p, int64_t n, const uint8_t *mask, void *state, int is_f64,
               int32_t *step_count, int32_t *episode, double *static_base, void *stream);

/* ---- one VecEnv step --------------------------------------------------------------------------
 * Replaces DummyVecEnv.step_wait over N TwoSeriesCSTREnv.step calls
 * (core/common/vec_env/dummy_vec_env.py:56-73; twoseriescstr.py:394-503,271-392).
 *   state        in: current normalised state; out: the observation step_wait returns
 *                (post-reset on done rows when auto_reset != 0, else the terminal observation)
 *   terminal_obs out (nullable): the new state before any reset (info["terminal_observation"] /
 *                the next_obs _store_transition stores)
 *   done = terminated or truncated; timeout = truncated and not terminated ("TimeLimit.truncated")
 * auto_reset == 0 leaves resetting to the caller (host PCG64 parity mode).
 * Episode statistics (Monitor semantics, core/common/monitor.py:85-111), all nullable:
 *   ep_return  (n,) double in/out running return; ep_final_return / ep_final_length (n,) out, written
 *   on done rows only: the finished episode's return and length (info["episode"]["r"/"l"]).          */
int cstr_vec_step_f32(const cstr_env_params *p, int64_t n, int math_mode, int auto_reset,
                      const float *actions, float *state, int32_t *step_count, int32_t *episode,
                      double *static_base, float *terminal_obs, float *reward, uint8_t *done,
                      uint8_t *timeout, double *ep_return, double *ep_final_return,
                      int32_t *ep_final_length, void *stream);
int cstr_vec_step_f64(const cstr_env_params *p, int64_t n, int auto_reset, const double *actions,
                      double *state, int32_t *step_count, int32_t *episode, double *static_base,
                      double *terminal_obs, double *reward, uint8_t *done, uint8_t *timeout,
                      double *ep_return, double *ep_final_return, int32_t *ep_final_length,
                      void *stream);

/* ---- T control intervals per launch, state held in registers ------------------------------------
 * Same semantics as T successive cstr_vec_step calls with auto-reset.
 *   actions  (T,n,2) tape, or NULL: actions are U(-1,1) from Philox (stream "action", counter
 *            t_base + t) generated in-kernel
 *   rewards (T,n), dones (T,n), obs_tape (T,n,4) = observation returned by each step: nullable
 *   reward_sum: nullable device double[1], atomically accumulates the sum of all rewards
 *   (size-independent checksum for large runs).                                                   */
int cstr_tape_f32(const cstr_env_params *p, int64_t n, int64_t T, int math_mode,
                  const float *actions, uint32_t t_base, float *state, int32_t *step_count,
                  int32_t *episode, double *static_base, float *rewards, uint8_t *dones,
                  float *obs_tape, double *reward_sum, void *stream);
int cstr_tape_f64(const cstr_env_params *p, int64_t n, int64_t T, const double *actions,
                  uint32_t t_base, double *state, int32_t *step_count, int32_t *episode,
                  double *static_base, double *rewards, uint8_t *dones, double *obs_tape,
                  double *reward_sum, void *stream);

/* Same as cstr_tape_f32 but with HOST buffers (pinned recommended): copies state/step_count/episode
 * and the action tape to scratch device memory owned by the library, runs the tape, copies state,
 * rewards and dones back, and synchronises.  This is the end-to-end call bench.py times ("e2e").   */
int cstr_tape_f32_host(const cstr_env_params *p, int64_t n, int64_t T, int math_mode,
                       const float *h_actions, float *h_state, int32_t *h_step_count,
                       int32_t *h_episode, float *h_rewards, uint8_t *h_dones, void *stream);

/* ---- ring replay buffer -------------------------------------------------------------------------
 * HBM layout: ONE 64-byte record per transition, records (rows, n_envs, 16) float32:
 *   [0:4] obs   [4:8] next_obs   [8:10] action   [10] reward   [11] done   [12] timeout   [13:16] pad
 * so that `add` is four coalesced 16-byte stores per reactor and a random-index `sample` reads two
 * whole 32-byte sectors per transition instead of six partial ones.  The reference's six arrays
 * (core/common/buffers.py:213-228: observations, next_observations, actions, rewards, dones,
 * timeouts) are exposed by the Python host as strided views of this tensor.
 *
 * cstr_replay_add replaces ReplayBuffer.add (buffers.py:247-283): writes ring row `pos`; the caller
 * advances pos/full (host ints, as in the reference).  done/timeout are uint8 device vectors
 * (timeout may be NULL = all False, the handle_timeout_termination=False case).                    */
#define CSTR_REC_FLOATS 16
#define CSTR_REC_OBS 0
#define CSTR_REC_NEXT_OBS 4
#define CSTR_REC_ACTION 8
#define CSTR_REC_REWARD 10
#define CSTR_REC_DONE 11
#define CSTR_REC_TIMEOUT 12

int cstr_replay_add(int64_t n_envs, int64_t pos, const float *obs, const float *next_obs,
                    const float *action, const float *reward, const uint8_t *done,
                    const uint8_t *timeout, float *records, void *stream);

/* Optional VecNormalize statistics applied inside the gather (ReplayBuffer._normalize_obs/_normalize_reward,
 * buffers.py:143-155,314-323): stats = the 16-double device block of cstr_norm_update.  NULL = no normalisation.      */
typedef struct cstr_norm_params {
    const double *stats;
    double epsilon, clip_obs, clip_reward; /* VecNormalize.epsilon / clip_obs / clip_reward */
    int32_t norm_obs, norm_reward;         /* VecNormalize.norm_obs / norm_reward           */
} cstr_norm_params;

/* cstr_replay_sample replaces ReplayBuffer._get_samples + to_torch (buffers.py:307-325,128-140):
 * gathers `batch` transitions at (batch_inds[i], env_inds[i]) into contiguous outputs
 * obs (B,4), act (B,2), next_obs (B,4), dones (B,1) = dones*(1-timeouts), rewards (B,1).
 * Index pairs are int64 device vectors (bit-exact mode: drawn on the host with the reference's two
 * np.random.randint calls).                                                                        */
int cstr_replay_sample(int64_t n_envs, int64_t batch, const int64_t *batch_inds,
                       const int64_t *env_inds, const float *records, float *out_obs,
                       float *out_act, float *out_next_obs, float *out_dones, float *out_rewards,
                       const cstr_norm_params *norm /* nullable */, void *stream);

/* Fast mode: indices drawn in-kernel from Philox (stream "sample", counter = (i, draw)): row uniform
 * in [0, upper), env uniform in [0, n_envs) by 32x32->64 multiply-shift.  Optionally returns the
 * drawn pairs (nullable).                                                                          */
int cstr_replay_sample_philox(uint64_t seed, uint64_t draw, int64_t n_envs, int64_t upper,
                              int64_t batch, const float *records, float *out_obs, float *out_act,
                              float *out_next_obs, float *out_dones, float *out_rewards,
                              int64_t *out_batch_inds, int64_t *out_env_inds,
                              const cstr_norm_params *norm /* nullable */, void *stream);
/* Same, with the draw counter read from device memory at execution time (no host scalar baked into the launch), so the call can
 * be captured in a CUDA graph and replayed; whoever owns the counter advances it (cstr_td3_update in graph mode does). */
int cstr_replay_sample_philox_dev(uint64_t seed, const int64_t *draw_dev, int64_t n_envs, int64_t upper,
                              int64_t batch, const float *records, float *out_obs, float *out_act,
                              float *out_next_obs, float *out_dones, float *out_rewards,
                              int64_t *out_batch_inds, int64_t *out_env_inds,
                              const cstr_norm_params *norm /* nullable */, void *stream);

/* ---- VecNormalize on the device ------------------------------------------------------------------------
 * cstr_norm_update replaces the statistics part of VecNormalize.step_wait (core/common/vec_env/vec_normalize.py:
 * 174-223) and RunningMeanStd.update (core/common/running_mean_std.py:36-56): obs (n,4) updates the observation
 * mean/var (NULL: skip); reward (n,) advances returns = returns*gamma + reward, updates the return mean/var and zeroes
 * returns on done rows (NULL: skip).  stats: 16 doubles on the device = obs mean[4], obs var[4], obs count, ret mean,
 * ret var, ret count (initialise mean 0, var 1, count 1e-4); scratch: 16 doubles, zero before the first call.
 * cstr_norm_apply replaces normalize_obs / normalize_reward (:225-259) for whole vectors (either side nullable).   */
int cstr_norm_update(int64_t n, const float *obs, const float *reward, const uint8_t *done, double *returns,
                     double gamma, double *stats, double *scratch, void *stream);
int cstr_norm_apply(int64_t n, const float *obs_in, const float *reward_in, const double *stats, double epsilon,
                    double clip_obs, double clip_reward, float *obs_out, float *reward_out, void *stream);

/* ---- TD3 gradient step (SURVEY §8f-1) ----------------------------------------------------------------
 * Replaces one iteration of the loop body of TD3.train (core/td3/td3.py:162-206) after the batch has been sampled:
 * target policy smoothing + twin-min target (:166-175), critic forward / MSE / backward (:178-186), Adam step of the
 * critic optimiser, and on every policy_delay-th update the actor loss -Q1(s, pi(s)).mean(), its backward, the
 * actor's Adam step and polyak_update of both target nets (:189-200, core/common/utils.py:457-481).
 * Networks: create_mlp(4, 2, [h1, h2]) + tanh for the actor, create_mlp(6, 1, [h1, h2]) for each of the two critics
 * (core/td3/policies.py:58, core/common/policies.py:966; torch nn.Linear layout), float32 arithmetic throughout.
 *
 * All five parameter-shaped blocks (params, targets, grads, adam_m, adam_v) use ONE flat layout of
 * cstr_td3_param_count(h1, h2) floats = [actor | critic0 | critic1], each net W1 b1 W2 b2 W3 b3 with every tensor
 * padded to a multiple of 4 floats; cstr_td3_layout writes the 18 tensor offsets (net-major) + the total.
 * counters are the values AFTER this update (1-based): n_updates decides the policy step, critic_step / actor_step
 * are the Adam step numbers used for the bias corrections.
 * phases: run a subset so a data-parallel caller can all-reduce `grads` between GRAD and APPLY.
 * noise: (batch,2) N(0, target_policy_noise) draws, or NULL = Philox (key seed, counter (row, n_updates), stream 5).
 * losses (nullable, 4 floats, device): [0] += critic loss, [1] += 1, [2] += actor loss, [3] += 1.                   */
typedef struct cstr_td3_config {
    int32_t h1, h2;       /* hidden sizes, multiples of 4 */
    int32_t batch;
    int32_t policy_delay;
    float gamma, tau, lr, beta1, beta2, eps, target_policy_noise, target_noise_clip;
    uint64_t seed;
    int32_t gemm_mode;    /* CSTR_TD3_GEMM_FP32: FFMA tiles (the reference's float32 arithmetic);                      */
    int32_t n_critics;    /* 2 (or 0) = TD3's twin critics; 1 = DDPG (core/ddpg/ddpg.py:100-109: TD3 with one critic,
                             policy_delay 1, target_noise_clip 0) — critic1's block of the layout stays unused              */
} cstr_td3_config;
#define CSTR_TD3_GEMM_FP32 0
#define CSTR_TD3_GEMM_TENSOR 1
#define CSTR_TD3_GEMM_BF16 2 /* tcgen05 with plain bf16 operands (fp32 accumulate): REDUCED precision, opt-in throughput mode */

/* ---- gradient all-reduce fused into the Adam step (multi-GPU, SURVEY §8e) -----------------------------------------
 * The data-parallel update's only collective is the mean of the flat gradient block over the ranks.  With a
 * cstr_peer_comm the APPLY phases do it themselves: every rank's `grads` block lives in memory the other ranks have mapped
 * (CUDA IPC, one process per GPU on one NVSwitch node), and the Adam kernel of rank r reads element i of ALL `world`
 * blocks over NVLink, sums them in rank order 0..world-1 (bit-identical result on every rank, no atomics), scales by
 * 1/world and goes straight into the Adam update — no separate collective launch, no second pass over the bucket.
 * Cross-GPU ordering: a per-CTA flag barrier over peer memory before the reads (every peer's backward pass has finished)
 * and after them (nobody overwrites its block while a peer still reads it); flags carry a per-launch epoch kept on the
 * device, so the launches can sit inside a CUDA graph.  A rank that waits longer than ~4 s (a dead peer) stops waiting,
 * raises the error word (cstr_peer_error) and skips the update instead of hanging the GPU; every later launch then skips
 * both the waits and the update at once (one bounded wait per broken group, never a hung stream).
 * cstr_peer_alloc returns device memory (cudaMalloc, zeroed) and its 64-byte IPC handle; cstr_peer_open maps a peer's
 * handle.  Layout of one rank's allocation, chosen by the caller: [grads block | pad to 256 B | cstr_peer_flag_bytes()]. */
#define CSTR_PEER_MAX_WORLD 8
typedef struct cstr_peer_comm {
    int32_t world, rank;
    float *grads[CSTR_PEER_MAX_WORLD];    /* grads[r]: rank r's flat gradient block as mapped in THIS process (grads[rank] = the local block) */
    uint32_t *flags[CSTR_PEER_MAX_WORLD]; /* flags[r]: rank r's barrier block (cstr_peer_flag_bytes() bytes, zero before the first update)  */
} cstr_peer_comm;
int64_t cstr_peer_flag_bytes(void);
int cstr_peer_alloc(int64_t bytes, void **ptr, void *handle64 /* 64 bytes out */);
int cstr_peer_open(const void *handle64, void **ptr);
int cstr_peer_close(void *ptr);
int cstr_peer_free(void *ptr);
/* non-zero after a peer wait timed out; *error is read from the local flag block (synchronises the stream)            */
int cstr_peer_error(const cstr_peer_comm *comm, uint32_t *error, void *stream);

typedef struct cstr_td3_state {
    float *params, *targets, *grads, *adam_m, *adam_v; /* device, cstr_td3_param_count floats each, 16-byte aligned */
    float *workspace;                                  /* device, >= cstr_td3_workspace_bytes(cfg)                  */
    int64_t workspace_bytes;
    float *losses;                                     /* device, 4 floats, or NULL                                 */
    int64_t *counters;                                 /* device, 4 x int64 {n_updates, critic_step, actor_step, sample_draw} BEFORE this
                                                          update, or NULL.  Non-NULL = graph mode: a one-thread kernel advances them at
                                                          the start of the update and derives the Philox counter of the smoothing noise and
                                                          the Adam bias corrections on the device, so nothing that changes from update to
                                                          update is baked into a launch and a cycle of policy_delay updates can be captured
                                                          in a CUDA graph and replayed (the by-value counters then only decide which
                                                          kernels are launched, i.e. whether this is a policy step)                     */
    const cstr_peer_comm *peer;                        /* NULL: single GPU, or the caller all-reduces `grads` between the GRAD and APPLY
                                                          phases itself.  Non-NULL: `grads` must be peer->grads[peer->rank] and the APPLY
                                                          phases average the gradient over the ranks inside the Adam kernel (see above)  */
} cstr_td3_state;

#define CSTR_TD3_CRITIC_GRAD 1
#define CSTR_TD3_CRITIC_APPLY 2
#define CSTR_TD3_ACTOR_GRAD 4
#define CSTR_TD3_ACTOR_APPLY 8
#define CSTR_TD3_ALL 15

int64_t cstr_td3_param_count(int32_t h1, int32_t h2);
int cstr_td3_layout(int32_t h1, int32_t h2, int64_t *offsets /* 19 */);
int64_t cstr_td3_workspace_bytes(const cstr_td3_config *cfg);
int cstr_td3_update(const cstr_td3_config *cfg, const cstr_td3_state *state, const float *obs, const float *actions,
                    const float *next_obs, const float *dones, const float *rewards, const float *noise,
                    int64_t n_updates, int64_t critic_step, int64_t actor_step, int32_t phases, void *stream);

/* ---- SAC gradient step (SURVEY §8f-1, second algorithm) -------------------------------------------------------
 * Replaces one iteration of the loop body of SAC.train (core/sac/sac.py:213-288) after the batch has been sampled:
 * squashed-Gaussian actor sample + log-prob (core/sac/policies.py:147-175, core/common/distributions.py:207-260), the
 * automatic entropy-coefficient Adam step (:226-243), the soft twin-min target from the CURRENT actor (:245-254), critic
 * forward / 0.5*sum MSE / backward / Adam (:256-268), actor loss (ent_coef*log_prob - min_i Q_i(s, a_pi)).mean() with its
 * backward through both critics and the tanh-Gaussian, actor Adam, polyak of the critic targets (:270-286).
 * Networks: actor = create_mlp(4, -, [h1, h2]) latent + [mu; log_std] head stored as ONE (4, h2) matrix (rows 0-1 mu,
 * rows 2-3 log_std); critics as for TD3.  Flat block = cstr_sac_param_count(h1, h2) floats = [actor | critic0 | critic1 |
 * log_ent_coef(+3 pad)]; cstr_sac_layout writes the 18 tensor offsets, the log_ent_coef offset and the block size.
 * The state struct is cstr_td3_state (targets: only the critic ranges are used; losses: 8 floats = critic, actor,
 * ent_coef_loss, ent_coef as {sum, count} pairs; counters as for TD3 — critic_step is the shared Adam step, the target
 * sync decision uses the by-value n_updates).  eps_pi / eps_next: (batch,2) standard-normal draws
 * of the two rsample() calls, or NULL = Philox (key seed, counter (row, n_updates), stream 5, call 0 / 1).
 * n_updates and adam_step are the values AFTER this update (1-based; all three optimisers share the step count).
 * phases: the CSTR_TD3_* bits.  CRITIC_GRAD = actor sample, d loss / d log_ent_coef (-> grads[log_ent_coef]), target,
 * critic gradients; CRITIC_APPLY = Adam on log_ent_coef and the critics; ACTOR_GRAD = actor loss backward; ACTOR_APPLY = actor
 * Adam + polyak.  A data-parallel caller all-reduces grads[critic0 .. log_ent_coef] after CRITIC_GRAD and grads[actor] after
 * ACTOR_GRAD; the intermediate activations of the earlier phases stay in the workspace.                               */
typedef struct cstr_sac_config {
    int32_t h1, h2, batch, target_update_interval;
    float gamma, tau, lr, beta1, beta2, eps, target_entropy, reserved0;
    uint64_t seed;
    int32_t gemm_mode;
    int32_t local_step;   /* which gradient step of the current SAC.train() call this is, 1-based: the reference's target sync tests the LOOP
                             index (`gradient_step % target_update_interval == 0`, core/sac/sac.py:284), which restarts at 0 on every
                             train() call.  0 = unknown: fall back to the global counter ((n_updates - 1) % interval)              */
    int32_t sde;          /* 1 = gSDE actor (use_sde=True, full_std, no expln), see below; 0 = the squashed Gaussian above            */
    float clip_mean;      /* gSDE: Hardtanh bound of the mean (<= 0: no Hardtanh)                                                   */
    uint64_t sde_seed;    /* gSDE: Philox key of the exploration eps, NOT keyed by the data-parallel rank (every rank draws one E)  */
} cstr_sac_config;
/* gSDE mode (sde = 1; core/sac/policies.py, core/common/distributions.py StateDependentNoiseDistribution with learn_features=True):
 * the actor's (4, h2) head slot holds [mu.weight (2,h2) | log_std (h2,2) row-major] and its 4-float bias slot [mu.bias (2) | 0 0]
 * (gradient 0 written to the pad); the layout, the Adam and the data-parallel ranges are unchanged.  Each update draws ONE exploration
 * matrix E = exp(log_std) * eps (reset_noise() with batch size 1 at the top of the loop body), eps (h2,2) from Philox (key sde_seed,
 * counter (k, n_updates), stream 10; in graph mode the update index comes from the device counters) or, for parity tests, from eps_pi
 * given as (h2,2) standard normals (eps_next must then be NULL).  mean = Hardtanh(mu(latent)), sigma = sqrt(latent^2 @ std^2 + 1e-6),
 * a = tanh(mean + latent @ E) for actions_pi and next_actions, log_prob = sum_j Normal(mean_j, sigma_j).log_prob(g_j) - sum_j log(1 -
 * tanh(g_j)^2 + 1e-6) with g = atanh(clamp(a, -1 + eps32, 1 - eps32)) (zero gradient where the clamp binds).  The actor loss reaches
 * log_std through sigma and through E.                                                                                            */

int64_t cstr_sac_param_count(int32_t h1, int32_t h2);
int cstr_sac_layout(int32_t h1, int32_t h2, int64_t *offsets /* 20 */);
int64_t cstr_sac_workspace_bytes(const cstr_sac_config *cfg);
int cstr_sac_update(const cstr_sac_config *cfg, const cstr_td3_state *state, const float *obs, const float *actions,
                    const float *next_obs, const float *dones, const float *rewards, const float *eps_pi,
                    const float *eps_next, int64_t n_updates, int64_t adam_step, int32_t phases, void *stream);

/* ---- BCQ gradient step (SURVEY §8f-1, third algorithm) ----------------------------------------------------------
 * Replaces one iteration of the loop body of BCQ.train (core/bcq/bcq.py:137-205) after the batch has been sampled, with the
 * networks of core/bcq/policies.py:21-166 for the CSTR spaces (obs 4, action 2):
 *   vae_enc   Linear(6, Hv) ReLU Linear(Hv, Hv) ReLU + the two heads stacked as ONE (2L, Hv) matrix [mean; log_std]   (:47-55)
 *   vae_dec   Linear(4 + L, Hv) ReLU Linear(Hv, Hv) ReLU Linear(Hv, 2) Tanh                                          (:58-65)
 *   pert      Linear(6, Hp) ReLU Linear(Hp, Hp) ReLU Linear(Hp, 2) Tanh, a + max_perturbation * xi clamped to [-1, 1]  (:147-160)
 *   critic0/1 create_mlp(6, 1, [h1, h2])                                                       (core/common/policies.py:966)
 * Steps: VAE (reconstruction MSE + 0.5 KL, Adam over encoder + decoder: :142-155); target from n_candidates latent draws through the
 * just-updated VAE (the "target VAE" is a plain copy of it, :158-159) and the TARGET perturbation net, twin-min, then the max over the
 * reference's (B, n_candidates) reshape of the candidate-major column AS WRITTEN (:165-172); twin critics (:174-186); on every
 * actor_delay-th update the perturbation step -Q1(s, pert(s, dec(s, z))).mean() (only the perturbation optimiser steps, :188-196) and
 * polyak of the critics and the perturbation net (:198-203).
 * Flat block (params, targets, grads, adam_m, adam_v) = [vae_enc | vae_dec | pert | critic0 | critic1], each net W1 b1 W2 b2 W3 b3
 * padded to multiples of 4 floats; cstr_bcq_layout writes 5 x 6 tensor offsets + the block size (31 values).  Of `targets` only the
 * pert and critic ranges are used.  Random draws: standard normal, UNclamped — eps_vae (B, L) of :76, z_next (n_candidates*B, L) of
 * sample_action (:122), z_actor (B, L) of the actor step's decode; NULL = Philox (key seed, counter (row, n_updates), streams 6/7/8).
 * State: cstr_td3_state (losses: 6 floats = vae, critic, actor as {sum, count}; counters as for TD3: critic_step is the Adam step of
 * the VAE and critic optimisers, actor_step that of the perturbation optimiser).  Counters are the values AFTER this update.
 * Data-parallel training goes through state->peer (the three Adam kernels average their gradient ranges over the ranks).       */
typedef struct cstr_bcq_config {
    int32_t latent;        /* L: vae_latent_dim, multiple of 4 in [4, 64]                       */
    int32_t vae_hidden;    /* Hv: vae_hidden_dim, multiple of 4                                 */
    int32_t pert_hidden;   /* Hp: perturbation_hidden_dim, multiple of 4                        */
    int32_t h1, h2;        /* critic hidden sizes                                               */
    int32_t batch, actor_delay, n_candidates;
    float gamma, tau, lr, beta1, beta2, eps, max_perturbation, reserved0;
    uint64_t seed;
    int32_t gemm_mode, reserved1;
} cstr_bcq_config;
int64_t cstr_bcq_param_count(const cstr_bcq_config *cfg);
int cstr_bcq_layout(const cstr_bcq_config *cfg, int64_t *offsets /* 31 */);
int64_t cstr_bcq_workspace_bytes(const cstr_bcq_config *cfg);
int cstr_bcq_update(const cstr_bcq_config *cfg, const cstr_td3_state *state, const float *obs, const float *actions, const float *next_obs,
                    const float *dones, const float *rewards, const float *eps_vae, const float *z_next, const float *z_actor,
                    int64_t n_updates, int64_t critic_step, int64_t actor_step, void *stream);

/* ---- MADDPG / IDDPG gradient step (SURVEY §8f-1, fourth and fifth algorithm) ---------------------------------------
 * Replaces one iteration of the loop body shared by MADDPG.train (core/maddpg/maddpg.py:127-185) and IDDPG.train
 * (core/iddpg/iddpg.py:127-185) for BASELINE config #5: the two reactors as two agents, observation_splits [[0,1],[2,3]],
 * action_splits [[0],[1]].  Per agent i: an actor create_mlp(2, 1, [h1, h2]) + Tanh on the agent's observation slice
 * (core/maddpg/policies.py:64-72) and n_critics q-networks — over ALL observations and actions (6 inputs) when centralised
 * (MADDPG, policies.py:236-241), over the agent's own slices (3 inputs) otherwise (IDDPG).
 * As written in the reference: the target actions of all agents are formed once, before the agent loop (:132-144); per agent the
 * critic step, then on every policy_delay-th update the actor step — which evaluates EVERY actor on agent i's observation slice
 * (:169-171) — and the polyak update of ALL agents' nets INSIDE the agent loop (:181-182).  Learning rates are per optimiser
 * (actor_lr[i], critic_lr[i]); the reference's _update_learning_rate pairing (base_class.py:1112-1136) makes them
 * learning_rate_list[0] for every actor and learning_rate_list[1] for every critic.
 * Flat block = [actor0 | actor1 | critic(0,0) .. critic(0,n_critics-1) | critic(1,0) ..]; cstr_ma_layout writes
 * (2 + 2 n_critics) x 6 tensor offsets + the block size.  noise: (2, B) N(0, target_policy_noise) draws (agent-major), NULL = Philox
 * (stream 9).  losses: 8 floats = critic0, actor0, critic1, actor1 as {sum, count}.  Counters as for TD3 (every agent's critic
 * optimiser has taken critic_step steps, every actor optimiser actor_step).  Data-parallel training goes through state->peer.   */
typedef struct cstr_ma_config {
    int32_t centralised;   /* 1 = MADDPG, 0 = IDDPG */
    int32_t h1, h2, batch, policy_delay, n_critics;
    float gamma, tau, beta1, beta2, eps, target_policy_noise, target_noise_clip, reserved0;
    float actor_lr[2], critic_lr[2];
    uint64_t seed;
    int32_t gemm_mode, reserved1;
} cstr_ma_config;
int64_t cstr_ma_param_count(const cstr_ma_config *cfg);
int cstr_ma_layout(const cstr_ma_config *cfg, int64_t *offsets /* (2 + 2 n_critics) * 6 + 1 */);
int64_t cstr_ma_workspace_bytes(const cstr_ma_config *cfg);
int cstr_ma_update(const cstr_ma_config *cfg, const cstr_td3_state *state, const float *obs, const float *actions, const float *next_obs,
                   const float *dones, const float *rewards, const float *noise, int64_t n_updates, int64_t critic_step, int64_t actor_step,
                   void *stream);

/* ---- fused rollout --------------------------------------------------------------------------------
 * Replaces, for K consecutive env steps of N reactors, OffPolicyAlgorithm._sample_action +
 * policy.predict (TD3 Actor.forward) + env.step + _store_transition + ReplayBuffer.add
 * (core/common/off_policy_algorithm.py:364-411,445-508,564; core/td3/policies.py:75-78;
 *  core/common/policies.py:331-413; core/common/buffers.py:247-283).
 * Actor = tanh(W3 relu(W2 relu(W1 x + b1) + b2) + b3), torch Linear layout (out,in), fp32.
 *   actor_mode 0: fp32 CUDA-core actor (parity path)
 *   actor_mode 1: bf16 tcgen05 tensor-core hidden layer, fp32 accumulate (throughput path);
 *                 needs the packed weights from cstr_actor_pack_bf16.
 * noise: TANH and SDE actors add sigma * N(0,1) exploration noise (NormalActionNoise) — from Philox (stream "noise") when
 * noise == NULL, else the (K,n,2) tensor is added as is.  GAUSSIAN actors use the same source as their eps ~ N(0,1)
 * (noise tensor = eps itself; sigma is ignored).
 * SDE actors (gSDE, use_sde=True) run on actor_mode 0 only and have no VecNormalize variant: both return CSTR_EINVAL.
 * warmup != 0: uniform random actions instead of the actor (learning_starts phase, :386-388).
 * Each step writes ring row (pos0 + k) % rows of the replay records and leaves `state` at the
 * observation to act on next.  rows = ring capacity in rows.                                       */
#define CSTR_ACTOR_TANH 0     /* TD3/DDPG actor: a = tanh(head)            core/td3/policies.py:75-78          */
#define CSTR_ACTOR_GAUSSIAN 1 /* SAC actor: a = tanh(mu + exp(clamp(log_std,-20,2)) * eps), eps ~ N(0,1)
                                 core/sac/policies.py:151-168, core/common/distributions.py:207-260           */
#define CSTR_ACTOR_SDE 2      /* SAC actor with gSDE: latent = relu(W2 relu(W1 x + b1) + b2), mean = hardtanh(W3 latent + b3, clip_mean),
                                 a = tanh(mean + latent @ explore[i]) with reactor i's (H2,2) exploration matrix
                                 (StateDependentNoiseDistribution, learn_features=True, full_std=True, use_expln=False)          */
typedef struct cstr_actor_f32 {
    const float *W1, *b1; /* (H1,4), (H1) */
    const float *W2, *b2; /* (H2,H1), (H2) */
    const float *W3, *b3; /* TANH, SDE: (2,H2), (2).  GAUSSIAN: (4,H2), (4) = rows [mu_0, mu_1, log_std_0, log_std_1] */
    int32_t H1, H2;
    int32_t kind;         /* CSTR_ACTOR_TANH | CSTR_ACTOR_GAUSSIAN | CSTR_ACTOR_SDE */
    float clip_mean;      /* SDE: the Hardtanh bound of mean (<= 0: no Hardtanh); 0 for the other kinds */
    const float *explore; /* SDE: (n,H2,2) per-reactor exploration matrices, std folded in (cstr_sde_sample), 8-byte aligned, row i =
                             local reactor i of this call; NULL for the other kinds */
} cstr_actor_f32;

/* gSDE exploration matrices for the SDE actor (StateDependentNoiseDistribution.sample_weights, core/common/distributions.py):
 * explore[i] = exp(log_std) * eps_i for the n reactors of this shard, eps_i (H2,2) standard normals from Philox keyed on
 * (seed, global reactor id env_offset + i, epoch) on the "sde" stream, so a row does not depend on how the reactors are sharded.
 * log_std: (H2,2) row-major; explore: (n,H2,2), 16-byte aligned.  The caller draws once per reset_noise() and passes a new epoch
 * each time; the rollout reads the stored matrices (at H2 = 256 they are 2 KiB per reactor).                                  */
int cstr_sde_sample(const float *log_std, int32_t h2, int64_t n, int64_t env_offset, uint64_t seed, uint32_t epoch, float *explore,
                    void *stream);

/* Monitor-style episode accounting for the fused rollout (core/common/monitor.py:85-111, the feed of
 * ep_info_buffer, core/common/base_class.py:462-481), all on the device: ep_return (n,) double is the running return of
 * every reactor (in/out); when an episode ends its (return, length) is appended to `finished` (capacity pairs of floats)
 * at index atomicAdd(count); entries beyond the capacity are counted but dropped.                                      */
typedef struct cstr_episode_stats {
    double *ep_return;   /* (n,) in/out */
    float *finished;     /* (capacity, 2): return, length */
    uint32_t *count;     /* device counter, caller-zeroed */
    uint32_t capacity;
    uint32_t reserved;
} cstr_episode_stats;

int cstr_rollout_fused(const cstr_env_params *p, int64_t n, int64_t K, int math_mode, int actor_mode,
                       const cstr_actor_f32 *actor, const void *packed_bf16, float sigma,
                       const float *noise, int warmup, uint32_t t_base, float *state,
                       int32_t *step_count, int32_t *episode, double *static_base, int64_t rows,
                       int64_t pos0, float *records, double *reward_sum, const cstr_episode_stats *stats /* nullable */,
                       void *stream);

/* VecNormalize variant.  Replaces, per env step, the same reference code as cstr_rollout_fused plus VecNormalize.step_wait's
 * statistics (core/common/vec_env/vec_normalize.py:174-223) and _store_transition's original-observation rule
 * (core/common/off_policy_algorithm.py:468-494):
 *   - the actor reads normalize_obs(obs) with the statistics in effect at that step (raw obs when norm_obs == 0);
 *   - training != 0: obs_rms is updated with the post-reset observations of ALL n reactors (norm_obs != 0), returns = returns * gamma
 *     + reward and ret_rms updated with them (whatever norm_reward is); returns of done rows are then zeroed (also when training == 0);
 *   - the records hold the raw obs, action, reward, done and timeout; next_obs of a done row is
 *     unnormalize_obs(normalize_obs(terminal obs)) with the statistics AFTER that step's update (differs from the terminal
 *     observation where clip_obs binds).
 * Each step needs statistics reduced over every reactor at the previous one, so the call enqueues one kernel launch per step (plus
 * one small launch that finishes the last step's done rows); the merge of the per-CTA sums is done in a fixed order, so the
 * statistics are the same bits from run to run.  No host synchronisation.  Arguments as for cstr_rollout_fused; the
 * multi-agent rollout has no VecNormalize variant.                                                                           */
typedef struct cstr_rollout_norm {
    double *stats;     /* 16 doubles on the device, the layout of cstr_norm_update (in/out)                                         */
    double *returns;   /* (n,) double VecNormalize.returns (in/out)                                                                 */
    void *workspace;   /* cstr_rollout_norm_workspace_bytes(n, actor_mode) bytes, 16-byte aligned, zeroed once before the first call */
    double gamma, epsilon, clip_obs; /* VecNormalize.gamma / epsilon / clip_obs */
    int32_t training, norm_obs;      /* VecNormalize.training / norm_obs        */
} cstr_rollout_norm;
int64_t cstr_rollout_norm_workspace_bytes(int64_t n, int actor_mode);
int cstr_rollout_fused_norm(const cstr_env_params *p, int64_t n, int64_t K, int math_mode, int actor_mode,
                            const cstr_actor_f32 *actor, const void *packed_bf16, float sigma,
                            const float *noise, int warmup, uint32_t t_base, float *state,
                            int32_t *step_count, int32_t *episode, double *static_base, int64_t rows,
                            int64_t pos0, float *records, double *reward_sum, const cstr_episode_stats *stats /* nullable */,
                            const cstr_rollout_norm *norm, void *stream);

/* Multi-agent variant (BASELINE config #5: the two reactors as two agents).  Replaces OffMultiAgentPolicyAlgorithm._sample_action +
 * MultiAgentBasePolicy.predict + env.step + _store_transition + ReplayBuffer.add
 * (core/common/multiagent_policy_algorithm.py:346-394,428-491,547; core/common/multi_agent_policies.py:500-563; core/maddpg/policies.py:88-121).
 * agent_actors: two cstr_actor_f32 (kind TANH, equal hidden sizes), agent i's 2 -> H1 -> H2 -> 1 net zero-padded to the single-agent shape:
 * W1 (H1,4) with the columns of the OTHER agent's observations zero, W3 (2,H2) with row i the agent's head and the other row zero, b3[i].
 * As written in the reference (quirk Q5) neither exploration noise nor per-agent rescaling is applied: the env receives, and the buffer
 * stores, u_i = low + 0.5 (mu_i + 1)(high - low); warm-up actions are the raw uniform draws.  fp32 CUDA-core actor.              */
int cstr_rollout_fused_multi(const cstr_env_params *p, int64_t n, int64_t K, int math_mode, const cstr_actor_f32 *agent_actors /* [2] */,
                             int warmup, uint32_t t_base, float *state, int32_t *step_count, int32_t *episode, double *static_base,
                             int64_t rows, int64_t pos0, float *records, double *reward_sum, const cstr_episode_stats *stats /* nullable */,
                             void *stream);

/* Packs W2 (H2,H1) fp32 into the bf16 UMMA shared-memory image the tensor-core path streams with
 * TMA-style bulk copies; returns the required size in bytes when dst == NULL.                      */
int64_t cstr_actor_pack_bf16(const cstr_actor_f32 *actor, void *dst, void *stream);

/* ---- measurement probes (bench.py roofline denominators) ------------------------------------------
 * FMA-chain microbenchmarks: every thread runs `iters` iterations of 8 independent FMA chains.
 * kind 0: fp32 FFMA, 1: fp64 DFMA, 2: fp32 separate FMUL+FADD (the non-contractible op mix),
 * 3: MUFU.EX2.  out: one value per thread (keeps the chains live); out[0] instead holds the SM clock in MHz that
 * thread 0 of block 0 observed over its own loop (clock64 cycles per globaltimer ns).  flops/launch =
 * grid*block*iters*8*(2 for kinds 0,1,2; 1 for kind 3).                                            */
int cstr_probe_pipe(int kind, int64_t iters, int grid, int block, float *out, void *stream);

/* Exhaustive device self-tests of the strict kernels' arithmetic shortcuts against the plain IEEE
 * operations they replace (0: -E/(R T) division, 1: normal-range exp scaling, 2: x/const Markstein
 * sequences for every constant divisor).  *mismatches (device uint64, caller-zeroed) must stay 0.  */
int cstr_selftest(int which, unsigned long long *mismatches, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* CSTR_B200_H */
