// K2 — fused rollout: actor MLP -> exploration noise -> action bounds -> CSTR step -> reward/done ->
// replay record, K env steps per launch with the reactor state resident in registers (sm_100a).
//
// Replaces, per env step (reference file:line):
//   OffPolicyAlgorithm._sample_action   core/common/off_policy_algorithm.py:364-411
//   BasePolicy.predict / scale / unscale core/common/policies.py:331-413
//   TD3 Actor.forward                   core/td3/policies.py:75-78 (create_mlp, torch_layers.py:110-183)
//   VecEnv.step -> TwoSeriesCSTREnv.step core/common/vec_env/dummy_vec_env.py:56-73, twoseriescstr.py:394-454
//   _store_transition + ReplayBuffer.add core/common/off_policy_algorithm.py:445-508, core/common/buffers.py:247-283
//
// actor_mode 0 (this file, fp32 CUDA cores): the parity path.  One CTA = 128 reactors and 16 warps; every lane works on
// four reactors.  Layer 1 (K=4) is computed by the reactor's threads and parked in shared memory k-major
// (h1[k][m]: conflict-free); layer 2 is a register-tiled contraction, 12 outputs per pass with the
// W2 rows fetched as warp-uniform 16-byte loads (L1-resident, 480 KB total streams from L2); layer 3
// (N=2) and tanh are folded into the layer-2 epilogue so h2 never exists in memory.
// actor_mode 1 (cstr_rollout_tc.cu): bf16 tcgen05 tensor-core hidden layer.
#include "cstr_abi.cuh"
#include "cstr_device.cuh"
#include "cstr_rollout_common.cuh"

namespace cstr {

constexpr int ROLL_M = 128;     // reactors per CTA (their h1 columns fill shared memory)
constexpr int ROLL_R = 4;       // reactors per thread in the actor: lane l works on reactors l, l+32, l+64, l+96
constexpr int ROLL_NB = 12;     // layer-2 outputs per register pass
constexpr int ROLL_PARTS = 16;  // warps per CTA; warp p takes the hidden units / output blocks p, p+16, ...
constexpr int ROLL_THREADS = ROLL_PARTS * 32;
// The kernel is bound by the L1 data pipe (ncu: 87 % of its wavefronts, FMA pipe 32 % with one reactor per thread): every
// warp-uniform 16-byte load of a W2 row piece and every h1 read is one wavefront.  Register-blocking FOUR reactors per thread
// makes one W2 load feed 16 FMAs per lane instead of 4: 28 wavefronts per 192 FMA instructions instead of 64.

// NORM (cstr_rollout_fused_norm, K == 1): the actor reads the normalised observation, done rows keep their raw terminal observation until
// the statistics that include this step exist, and the CTA's moment sums go to norm_merge.
// KIND == CSTR_ACTOR_SDE (gSDE): the layer-2 epilogue also accumulates noise = latent @ explore[i] into partial heads 2 and 3, each lane
// reading its own reactors' (H2,2) matrices (row i of `explore`); the head is then tanh(hardtanh(mu) + noise) plus the additive noise
// of the TANH kind.
template <int MODE, int KIND, bool NORM>
__global__ void __launch_bounds__(ROLL_THREADS, 1)
rollout_f32_kernel(cstr_env_params p, int64_t n, int64_t K, ActorNet actor_a, ActorNet actor_b, int n_agents, float sigma,
                   const float2 *__restrict__ noise, int warmup,
                   uint32_t t_base, float4 *__restrict__ state, int32_t *__restrict__ step_count, int32_t *__restrict__ episode,
                   double *static_base, int64_t rows, int64_t pos0, float4 *__restrict__ records, double *reward_sum, cstr_episode_stats stats,
                   int has_stats, NormLaunch nl, const float2 *__restrict__ explore) {
    extern __shared__ float h1[];  // [H1][ROLL_M] (reused for the partial heads [PARTS][4][ROLL_M] once layer 2 is done), then the state column
    constexpr bool SDE = KIND == CSTR_ACTOR_SDE;
    constexpr int NOUT = KIND == CSTR_ACTOR_GAUSSIAN ? 4 : 2;  // rows of W3
    constexpr int NPART = SDE ? 4 : NOUT;                      // partial heads per warp: [mu_0, mu_1, noise_0, noise_1] for SDE
    const int lane = threadIdx.x & 31, part = threadIdx.x >> 5;
    const bool owner = part < ROLL_M / 32;  // warps 0..3 own one reactor per lane: state registers, head, env step, record
    const int m = part * 32 + lane;         // the owned reactor (owners only)
    const int64_t i = (int64_t)blockIdx.x * ROLL_M + m;
    const bool live = owner && i < n;
    // n_agents == 2 (multi-agent, core/common/multiagent_policy_algorithm.py:346-394): the actor pass runs once per agent with that agent's
    // weights — its 2 -> H1 -> H2 -> 1 net zero-padded to the 4 -> H1 -> H2 -> 2 shape (W1 columns of the other agent's observations and the
    // other W3 row are zero, which adds exact zeros in the same summation order) — and output component `agent` is kept
    const int H1 = actor_a.H1, H2 = actor_a.H2;
    const size_t h1_floats = max((size_t)H1 * ROLL_M, (size_t)ROLL_PARTS * 4 * ROLL_M);
    float4 *s_state = reinterpret_cast<float4 *>(h1 + h1_floats);
    float *s_o = h1;
    float4 s = live ? state[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    int sc = live ? step_count[i] : 0, ep = live ? episode[i] : 0;
    const uint64_t env = (uint64_t)(p.env_offset + i);
    double acc_r = 0.0;
    double ep_ret = (has_stats && live) ? stats.ep_return[i] : 0.0;
    uint4 cache = make_uint4(0, 0, 0, 0);
    double nacc[NORM_SUMS];
    if constexpr (NORM) {
#pragma unroll
        for (int j = 0; j < NORM_SUMS; ++j) nacc[j] = 0.0;
        if (live) norm_fix_pending(nl, i, n, records);
    }

    for (int64_t k = 0; k < K; ++k) {
        const uint32_t g = t_base + (uint32_t)k;
        float2 env_a = make_float2(0.f, 0.f), buf_a = make_float2(0.f, 0.f);
        if (warmup) {
            if (owner) {
                // learning_starts phase: uniform action from the space (:386-388), then scale (:398)
                const float2 a = philox_action(p.seed, env, g, cache, k == 0 || (g & 1u) == 0);
                buf_a = make_float2(__fadd_rn(__fmul_rn(2.0f, __fmul_rn(__fadd_rn(a.x, 1.0f), 0.5f)), -1.0f),
                                    __fadd_rn(__fmul_rn(2.0f, __fmul_rn(__fadd_rn(a.y, 1.0f), 0.5f)), -1.0f));
                env_a = make_float2(__fadd_rn(-1.0f, __fmul_rn(__fmul_rn(0.5f, __fadd_rn(buf_a.x, 1.0f)), 2.0f)),
                                    __fadd_rn(-1.0f, __fmul_rn(__fmul_rn(0.5f, __fadd_rn(buf_a.y, 1.0f)), 2.0f)));
                if (n_agents > 1) env_a = buf_a = a;  // quirk Q5: the multi-agent path neither scales nor unscales (:369,390-392)
            }
        } else {
          float mu_agent[2] = {0.f, 0.f};
          for (int agent = 0; agent < n_agents; ++agent) {
            const ActorNet &actor = agent ? actor_b : actor_a;
            if constexpr (NORM) {
                if (owner) s_state[m] = nl.norm_obs ? norm_obs4(s, nl) : s;
            } else {
                if (owner) s_state[m] = s;
            }
            __syncthreads();
            float4 sv[ROLL_R];
#pragma unroll
            for (int r = 0; r < ROLL_R; ++r) sv[r] = s_state[lane + 32 * r];
            // ---- layer 1: h1 = relu(W1 s + b1), parked k-major in shared memory; warp p computes the hidden units p, p+16, ...
            for (int j = part; j < H1; j += ROLL_PARTS) {
                const float4 w = __ldg(reinterpret_cast<const float4 *>(actor.W1) + j);
                const float bj = __ldg(actor.b1 + j);
#pragma unroll
                for (int r = 0; r < ROLL_R; ++r) {
                    float v = bj;
                    v = fmaf(w.x, sv[r].x, v);
                    v = fmaf(w.y, sv[r].y, v);
                    v = fmaf(w.z, sv[r].z, v);
                    v = fmaf(w.w, sv[r].w, v);
                    h1[j * ROLL_M + lane + 32 * r] = fmaxf(v, 0.0f);
                }
            }
            __syncthreads();
            // ---- layer 2 + 3: out = W3 relu(W2 h1 + b2) + b3, 12 hidden units x 4 reactors per pass, passes dealt round-robin to the warps
            float o[ROLL_R][4];
#pragma unroll
            for (int r = 0; r < ROLL_R; ++r)
#pragma unroll
                for (int c = 0; c < 4; ++c) o[r][c] = 0.f;
            for (int nb = part * ROLL_NB; nb < H2; nb += ROLL_PARTS * ROLL_NB) {
                float acc[ROLL_NB][ROLL_R];
#pragma unroll
                for (int q = 0; q < ROLL_NB; ++q)
#pragma unroll
                    for (int r = 0; r < ROLL_R; ++r) acc[q][r] = 0.0f;
                const int H1v = H1 & ~3;
                for (int kk = 0; kk < H1v; kk += 4) {
                    float a[4][ROLL_R];
#pragma unroll
                    for (int c = 0; c < 4; ++c)
#pragma unroll
                        for (int r = 0; r < ROLL_R; ++r) a[c][r] = h1[(kk + c) * ROLL_M + lane + 32 * r];
#pragma unroll
                    for (int q = 0; q < ROLL_NB; ++q) {
                        const int row = min(nb + q, H2 - 1);  // clamp: tail lanes recompute the last row, discarded below
                        const float4 w = __ldg(reinterpret_cast<const float4 *>(actor.W2 + (size_t)row * H1 + kk));
#pragma unroll
                        for (int r = 0; r < ROLL_R; ++r) {  // same summation order per reactor as the one-reactor version
                            acc[q][r] = fmaf(w.x, a[0][r], acc[q][r]);
                            acc[q][r] = fmaf(w.y, a[1][r], acc[q][r]);
                            acc[q][r] = fmaf(w.z, a[2][r], acc[q][r]);
                            acc[q][r] = fmaf(w.w, a[3][r], acc[q][r]);
                        }
                    }
                }
                for (int kk = H1v; kk < H1; ++kk) {
#pragma unroll
                    for (int q = 0; q < ROLL_NB; ++q) {
                        const float w = __ldg(actor.W2 + (size_t)min(nb + q, H2 - 1) * H1 + kk);
#pragma unroll
                        for (int r = 0; r < ROLL_R; ++r) acc[q][r] = fmaf(w, h1[kk * ROLL_M + lane + 32 * r], acc[q][r]);
                    }
                }
#pragma unroll
                for (int q = 0; q < ROLL_NB; ++q) {
                    if (nb + q < H2) {
                        const float b2 = __ldg(actor.b2 + nb + q);
#pragma unroll
                        for (int c = 0; c < NOUT; ++c) {
                            const float w3 = __ldg(actor.W3 + (size_t)c * H2 + nb + q);
#pragma unroll
                            for (int r = 0; r < ROLL_R; ++r) o[r][c] = fmaf(w3, fmaxf(acc[q][r] + b2, 0.0f), o[r][c]);
                        }
                        if constexpr (SDE) {
#pragma unroll
                            for (int r = 0; r < ROLL_R; ++r) {  // past-the-end reactors read the last one's matrix; their heads are discarded
                                const int64_t ir = min((int64_t)blockIdx.x * ROLL_M + lane + 32 * r, n - 1);
                                const float2 e = __ldg(explore + (size_t)ir * H2 + nb + q);
                                const float lat = fmaxf(acc[q][r] + b2, 0.0f);
                                o[r][2] = fmaf(lat, e.x, o[r][2]);
                                o[r][3] = fmaf(lat, e.y, o[r][3]);
                            }
                        }
                    }
                }
            }
            __syncthreads();  // every warp is done with h1: its memory now carries the partial heads
#pragma unroll
            for (int r = 0; r < ROLL_R; ++r)
#pragma unroll
                for (int c = 0; c < NPART; ++c) s_o[(part * 4 + c) * ROLL_M + lane + 32 * r] = o[r][c];
            __syncthreads();
            if (owner) {
                float oo[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int c = 0; c < NOUT; ++c) {  // fixed order: bias, then warps 0..15
                    float v = __ldg(actor.b3 + c);
#pragma unroll
                    for (int q = 0; q < ROLL_PARTS; ++q) v += s_o[(q * 4 + c) * ROLL_M + m];
                    oo[c] = v;
                }
                if constexpr (SDE) {  // get_actions: tanh(mean + latent @ E), mean = Hardtanh(mu) when clip_mean > 0 (sac/policies.py)
                    float nse[2] = {0.f, 0.f};
#pragma unroll
                    for (int c = 0; c < 2; ++c)
#pragma unroll
                        for (int q = 0; q < ROLL_PARTS; ++q) nse[c] += s_o[(q * 4 + 2 + c) * ROLL_M + m];
                    const float cm = actor.clip_mean;
#pragma unroll
                    for (int c = 0; c < 2; ++c) oo[c] = __fadd_rn(cm > 0.0f ? fminf(fmaxf(oo[c], -cm), cm) : oo[c], nse[c]);
                }
                float2 nz;
                if (noise) nz = live ? noise[k * n + i] : make_float2(0.f, 0.f);
                else if (KIND == CSTR_ACTOR_GAUSSIAN) nz = philox_normal2(p.seed, env, g);
                else if (sigma != 0.0f) { nz = philox_normal2(p.seed, env, g); nz.x *= sigma; nz.y *= sigma; }
                else nz = make_float2(0.f, 0.f);
                float mu0, mu1;
                float2 add;
                actor_head<SDE ? CSTR_ACTOR_TANH : KIND>(oo, nz, mu0, mu1, add);
                if (n_agents == 1) {
                    action_maps(mu0, add.x, env_a.x, buf_a.x);
                    action_maps(mu1, add.y, env_a.y, buf_a.y);
                } else {
                    mu_agent[agent] = agent ? mu1 : mu0;
                    if (agent == n_agents - 1) {  // predict()'s unscale (multi_agent_policies.py:548-550,592) is all that happens: no noise, no rescale (Q5)
                        env_a = make_float2(__fadd_rn(-1.0f, __fmul_rn(__fmul_rn(0.5f, __fadd_rn(mu_agent[0], 1.0f)), 2.0f)),
                                            __fadd_rn(-1.0f, __fmul_rn(__fmul_rn(0.5f, __fadd_rn(mu_agent[1], 1.0f)), 2.0f)));
                        buf_a = env_a;
                    }
                }
            }
            if (agent + 1 < n_agents) __syncthreads();  // the owners are done with the partial heads before the next pass overwrites shared memory
          }
        }
        if (!owner) continue;  // (every thread has passed this step's barriers by now)
        // ---- env step + transition record
        const float4 obs = s;
        const StepResult r = (MODE == CSTR_MATH_STRICT) ? step_strict_f32(s, env_a, sc, (float)p.target_c2, p.max_steps)
                                                        : step_fast_f32(s, env_a, sc, (float)p.target_c2, p.max_steps);
        if (live) {
            const int64_t row = (pos0 + k) % rows;
            float4 next_obs = s;
            if constexpr (NORM) {
                if (r.truncated && nl.norm_obs) {
                    if (nl.training) nl.pending[i] = 1;  // the round trip needs S_{k+1}: the next launch (or the fix-up kernel) writes it
                    else next_obs = norm_round_trip4(s, nl);  // frozen statistics: S_{k+1} == S_k
                }
            }
            store_record(records + ((size_t)row * n + i) * 4, obs, next_obs, buf_a, r.reward, r.truncated);
            acc_r += (double)r.reward;
            episode_account(stats, has_stats != 0, ep_ret, r.reward, r.truncated, sc);
        }
        if (r.truncated) {
            if (live) s = reset_f32_env(p, i, ep, static_base);
            sc = 0;
        }
        if constexpr (NORM) {
            if (live) norm_account(nl, i, s, r.reward, r.truncated, nacc);
        }
    }
    if constexpr (NORM) {
        if (nl.training) norm_merge<ROLL_THREADS>(nl, n, nacc, reinterpret_cast<double *>(h1));
    }
    if (!owner) return;
    if (live) {
        state[i] = s;
        step_count[i] = sc;
        episode[i] = ep;
        if (has_stats) stats.ep_return[i] = ep_ret;
    }
    if (reward_sum) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc_r += __shfl_down_sync(0xffffffffu, acc_r, o);
        if (lane == 0) atomicAdd(reward_sum, acc_r);
    }
}

// the done rows of the last step of a call: their final next_obs, with the statistics that launch left
__global__ void __launch_bounds__(256) rollout_norm_fix_kernel(int64_t n, NormLaunch nl, float4 *__restrict__ records) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    norm_fix_pending(nl, i, n, records);
}

}  // namespace cstr

using namespace cstr;

// tensor-core path lives in cstr_rollout_tc.cu
int cstr_rollout_tc_launch(const cstr_env_params *p, int64_t n, int64_t K, int math_mode, const cstr_actor_f32 *actor,
                           const void *packed_bf16, float sigma, const float *noise, int warmup, uint32_t t_base, float *state,
                           int32_t *step_count, int32_t *episode, double *static_base, int64_t rows, int64_t pos0, float *records,
                           double *reward_sum, const cstr_episode_stats *stats, const NormLaunch *nl, void *stream);

static int rollout_fused_impl(const cstr_env_params *p, int64_t n, int64_t K, int math_mode, int actor_mode, const cstr_actor_f32 *actor,
                              const cstr_actor_f32 *actor_b, const void *packed_bf16, float sigma, const float *noise, int warmup, uint32_t t_base,
                              float *state, int32_t *step_count, int32_t *episode, double *static_base, int64_t rows, int64_t pos0, float *records,
                              double *reward_sum, const cstr_episode_stats *stats, const NormLaunch *nl, void *stream);

extern "C" int cstr_rollout_fused(const cstr_env_params *p, int64_t n, int64_t K, int math_mode, int actor_mode,
                                  const cstr_actor_f32 *actor, const void *packed_bf16, float sigma, const float *noise, int warmup,
                                  uint32_t t_base, float *state, int32_t *step_count, int32_t *episode, double *static_base,
                                  int64_t rows, int64_t pos0, float *records, double *reward_sum, const cstr_episode_stats *stats, void *stream) {
    return rollout_fused_impl(p, n, K, math_mode, actor_mode, actor, nullptr, packed_bf16, sigma, noise, warmup, t_base, state, step_count, episode,
                              static_base, rows, pos0, records, reward_sum, stats, nullptr, stream);
}

extern "C" int cstr_rollout_fused_multi(const cstr_env_params *p, int64_t n, int64_t K, int math_mode, const cstr_actor_f32 *agent_actors, int warmup,
                                        uint32_t t_base, float *state, int32_t *step_count, int32_t *episode, double *static_base, int64_t rows,
                                        int64_t pos0, float *records, double *reward_sum, const cstr_episode_stats *stats, void *stream) {
    if (!warmup) {
        if (!agent_actors) return fail_arg(CSTR_EINVAL, "rollout_multi: agent actors missing");
        if (agent_actors[0].H1 != agent_actors[1].H1 || agent_actors[0].H2 != agent_actors[1].H2 || agent_actors[0].kind != CSTR_ACTOR_TANH ||
            agent_actors[1].kind != CSTR_ACTOR_TANH)
            return fail_arg(CSTR_EINVAL, "rollout_multi: both agents need tanh actors of the same hidden sizes");
    }
    static const cstr_actor_f32 none = {};
    return rollout_fused_impl(p, n, K, math_mode, 0, agent_actors ? agent_actors : &none, agent_actors ? agent_actors + 1 : &none, nullptr, 0.0f, nullptr,
                              warmup, t_base, state, step_count, episode, static_base, rows, pos0, records, reward_sum, stats, nullptr, stream);
}

static int rollout_fused_impl(const cstr_env_params *p, int64_t n, int64_t K, int math_mode, int actor_mode, const cstr_actor_f32 *actor,
                              const cstr_actor_f32 *actor_b, const void *packed_bf16, float sigma, const float *noise, int warmup, uint32_t t_base,
                              float *state, int32_t *step_count, int32_t *episode, double *static_base, int64_t rows, int64_t pos0, float *records,
                              double *reward_sum, const cstr_episode_stats *stats, const NormLaunch *nl, void *stream) {
    if (!p || n < 0 || K < 0 || !state || !step_count || !episode || !records || rows <= 0 || pos0 < 0)
        return fail_arg(CSTR_EINVAL, "rollout: null pointer or bad size");
    if (p->init_mode == CSTR_INIT_STATIC && !static_base) return fail_arg(CSTR_EINVAL, "static init_mode needs static_base");
    if (math_mode != CSTR_MATH_STRICT && math_mode != CSTR_MATH_FAST) return fail_arg(CSTR_EINVAL, "unknown math_mode");
    if (!aligned(state, 16) || !aligned(records, 16) || (noise && !aligned(noise, 8))) return fail_arg(CSTR_EALIGN, "rollout: alignment");
    if (!warmup) {
        if (!actor || !actor->W1 || !actor->b1 || !actor->W2 || !actor->b2 || !actor->W3 || !actor->b3)
            return fail_arg(CSTR_EINVAL, "rollout: actor weights missing");
        if (actor->H1 <= 0 || actor->H2 <= 0 || (actor->H1 & 3)) return fail_arg(CSTR_EINVAL, "rollout: H1 must be a positive multiple of 4");
        if (actor->kind != CSTR_ACTOR_TANH && actor->kind != CSTR_ACTOR_GAUSSIAN && actor->kind != CSTR_ACTOR_SDE)
            return fail_arg(CSTR_EINVAL, "rollout: unknown actor kind");
        if (actor->kind == CSTR_ACTOR_SDE) {
            if (actor_mode != 0 || nl) return fail_arg(CSTR_EINVAL, "rollout: the gSDE actor runs on the fp32 kernel (actor_mode 0) without VecNormalize");
            if (!actor->explore) return fail_arg(CSTR_EINVAL, "rollout: the gSDE actor needs its exploration matrices (cstr_sde_sample)");
            if (!aligned(actor->explore, 8)) return fail_arg(CSTR_EALIGN, "rollout: explore 8 B alignment");
        }
        if (!aligned(actor->W1, 16) || !aligned(actor->W2, 16)) return fail_arg(CSTR_EALIGN, "rollout: W1/W2 16 B alignment");
    }
    if (stats && (!stats->ep_return || !stats->finished || !stats->count)) return fail_arg(CSTR_EINVAL, "rollout: episode stats pointers missing");
    if (n == 0 || K == 0) return 0;
    if (actor_b && !warmup) {
        if (!actor_b->W1 || !actor_b->b1 || !actor_b->W2 || !actor_b->b2 || !actor_b->W3 || !actor_b->b3 || !aligned(actor_b->W1, 16) || !aligned(actor_b->W2, 16))
            return fail_arg(CSTR_EINVAL, "rollout_multi: second agent's weights missing or misaligned");
    }
    if (actor_mode == 1 && !warmup)
        return cstr_rollout_tc_launch(p, n, K, math_mode, actor, packed_bf16, sigma, noise, warmup, t_base, state, step_count, episode,
                                      static_base, rows, pos0, records, reward_sum, stats, nl, stream);
    if (actor_mode != 0 && actor_mode != 1) return fail_arg(CSTR_EINVAL, "rollout: unknown actor_mode");
    ActorNet a = {}, b2nd = {};
    if (actor) a = actor_net(*actor);
    if (actor_b) b2nd = actor_net(*actor_b);
    const int n_agents = actor_b ? 2 : 1;
    const size_t h1_floats = (size_t)a.H1 * ROLL_M > (size_t)ROLL_PARTS * 4 * ROLL_M ? (size_t)a.H1 * ROLL_M : (size_t)ROLL_PARTS * 4 * ROLL_M;
    size_t smem = warmup ? 0 : h1_floats * sizeof(float) + ROLL_M * sizeof(float4);
    if (nl && smem < (ROLL_PARTS * NORM_SUMS + 1) * sizeof(double)) smem = (ROLL_PARTS * NORM_SUMS + 1) * sizeof(double);  // norm_merge's sums
    if (smem > 227 * 1024) return fail_arg(CSTR_EINVAL, "rollout: H1 too large for the fp32 path (max 448)");
    const int grid = (int)((n + ROLL_M - 1) / ROLL_M);
    cudaStream_t st = (cudaStream_t)stream;
    int rc = 0;
#define CSTR_LAUNCH_ROLL(MODE, KIND)                                                                                                       \
    do {                                                                                                                                   \
        rc = check_cuda(cudaFuncSetAttribute(rollout_f32_kernel<MODE, KIND, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "smem attr"); \
        if (!rc)                                                                                                                           \
            rollout_f32_kernel<MODE, KIND, false><<<grid, ROLL_THREADS, smem, st>>>(*p, n, K, a, b2nd, n_agents, sigma, (const float2 *)noise, warmup, t_base, (float4 *)state, \
                                                                       step_count, episode, static_base, rows, pos0, (float4 *)records, reward_sum, st_copy, has_stats, NormLaunch{},    \
                                                                       (const float2 *)(KIND == CSTR_ACTOR_SDE ? actor->explore : nullptr)); \
    } while (0)
    cstr_episode_stats st_copy = {};
    const int has_stats = stats != nullptr;
    if (stats) {
        st_copy = *stats;
    }
#define CSTR_LAUNCH_ROLL_NORM(MODE, KIND)                                                                                                  \
    do {                                                                                                                                   \
        rc = check_cuda(cudaFuncSetAttribute(rollout_f32_kernel<MODE, KIND, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem), "smem attr"); \
        if (!rc)                                                                                                                           \
            rollout_f32_kernel<MODE, KIND, true><<<grid, ROLL_THREADS, smem, st>>>(*p, n, K, a, b2nd, n_agents, sigma, (const float2 *)noise, warmup,     \
                                                                            t_base, (float4 *)state, step_count, episode, static_base, rows, pos0,  \
                                                                            (float4 *)records, reward_sum, st_copy, has_stats, *nl, nullptr);      \
    } while (0)
    const bool gauss = a.kind == CSTR_ACTOR_GAUSSIAN;
    if (!warmup && a.kind == CSTR_ACTOR_SDE) {
        if (math_mode == CSTR_MATH_STRICT) CSTR_LAUNCH_ROLL(CSTR_MATH_STRICT, CSTR_ACTOR_SDE);
        else CSTR_LAUNCH_ROLL(CSTR_MATH_FAST, CSTR_ACTOR_SDE);
    } else if (nl) {
        if (math_mode == CSTR_MATH_STRICT) { if (gauss) CSTR_LAUNCH_ROLL_NORM(CSTR_MATH_STRICT, CSTR_ACTOR_GAUSSIAN); else CSTR_LAUNCH_ROLL_NORM(CSTR_MATH_STRICT, CSTR_ACTOR_TANH); }
        else { if (gauss) CSTR_LAUNCH_ROLL_NORM(CSTR_MATH_FAST, CSTR_ACTOR_GAUSSIAN); else CSTR_LAUNCH_ROLL_NORM(CSTR_MATH_FAST, CSTR_ACTOR_TANH); }
    } else if (math_mode == CSTR_MATH_STRICT) { if (gauss) CSTR_LAUNCH_ROLL(CSTR_MATH_STRICT, CSTR_ACTOR_GAUSSIAN); else CSTR_LAUNCH_ROLL(CSTR_MATH_STRICT, CSTR_ACTOR_TANH); }
    else { if (gauss) CSTR_LAUNCH_ROLL(CSTR_MATH_FAST, CSTR_ACTOR_GAUSSIAN); else CSTR_LAUNCH_ROLL(CSTR_MATH_FAST, CSTR_ACTOR_TANH); }
#undef CSTR_LAUNCH_ROLL
#undef CSTR_LAUNCH_ROLL_NORM
    if (rc) return rc;
    return check_launch("rollout_f32_kernel");
}

// gSDE exploration matrices: thread t of reactor i writes explore[i][4t .. 4t+3] = exp(log_std[4t .. 4t+3]) * N(0,1) from one Philox
// call on counter (global id, epoch, "sde" stream | t): the Box-Muller pair of philox_normal4 in cstr_mlp.cuh
constexpr uint32_t STREAM_SDE = 11u;
__global__ void __launch_bounds__(256) sde_sample_kernel(const float *__restrict__ log_std, int h2, int64_t n, int64_t env_offset, uint64_t seed,
                                                          uint32_t epoch, float *__restrict__ explore) {
    const int per = (2 * h2 + 3) / 4;  // Philox calls per reactor (the last one is half used when h2 is odd)
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * per) return;
    const int64_t i = idx / per;
    const uint32_t t = (uint32_t)(idx - i * per);
    const uint64_t env = (uint64_t)(env_offset + i);
    // the call index takes the low byte of the counter's last word (as for the other streams) and, past 255, its top 16 bits
    const uint4 r = philox4x32_10(make_uint4((uint32_t)env, (uint32_t)(env >> 32), epoch, (STREAM_SDE << 8) | (t & 0xffu) | ((t >> 8) << 16)),
                                  (uint32_t)seed, (uint32_t)(seed >> 32));
    const float u1 = fmaf(u24(r.x), 1.0f, 5.9604644775390625e-08f), u2 = u24(r.y);
    const float u3 = fmaf(u24(r.z), 1.0f, 5.9604644775390625e-08f), u4 = u24(r.w);
    const float ra = sqrtf(-2.0f * logf(u1)), rb = sqrtf(-2.0f * logf(u3));
    float s1, c1, s2, c2;
    sincospif(2.0f * u2, &s1, &c1);
    sincospif(2.0f * u4, &s2, &c2);
    const float z[4] = {ra * c1, ra * s1, rb * c2, rb * s2};
    const int j0 = 4 * (int)t;
    float *out = explore + (size_t)i * 2 * h2;
#pragma unroll
    for (int c = 0; c < 4; ++c)
        if (j0 + c < 2 * h2) out[j0 + c] = __fmul_rn(expf(log_std[j0 + c]), z[c]);  // Normal(0, std).rsample() = 0 + eps * std
}

extern "C" int cstr_sde_sample(const float *log_std, int32_t h2, int64_t n, int64_t env_offset, uint64_t seed, uint32_t epoch, float *explore,
                               void *stream) {
    if (!log_std || !explore || h2 <= 0 || n < 0 || env_offset < 0) return fail_arg(CSTR_EINVAL, "sde_sample: null pointer or bad size");
    if (h2 > (1 << 23)) return fail_arg(CSTR_EINVAL, "sde_sample: h2 too large");
    if (!aligned(explore, 16)) return fail_arg(CSTR_EALIGN, "sde_sample: explore 16 B alignment");
    if (n == 0) return 0;
    const int64_t threads = n * ((2 * (int64_t)h2 + 3) / 4);
    sde_sample_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(log_std, h2, n, env_offset, seed, epoch, explore);
    return check_launch("sde_sample_kernel");
}

// workspace of cstr_rollout_fused_norm: [ticket (16 B)][partials: grid x NORM_SUMS doubles][pending: n bytes]; both kernels use 128-reactor CTAs
static int64_t norm_grid(int64_t n) { return (n + ROLL_M - 1) / ROLL_M; }

extern "C" int64_t cstr_rollout_norm_workspace_bytes(int64_t n, int actor_mode) {
    if (n < 0 || (actor_mode != 0 && actor_mode != 1)) return fail_arg(CSTR_EINVAL, "rollout_norm_workspace_bytes: bad size or actor_mode");
    return 16 + norm_grid(n) * NORM_SUMS * (int64_t)sizeof(double) + ((n + 15) & ~(int64_t)15);
}

extern "C" int cstr_rollout_fused_norm(const cstr_env_params *p, int64_t n, int64_t K, int math_mode, int actor_mode,
                                       const cstr_actor_f32 *actor, const void *packed_bf16, float sigma, const float *noise, int warmup,
                                       uint32_t t_base, float *state, int32_t *step_count, int32_t *episode, double *static_base,
                                       int64_t rows, int64_t pos0, float *records, double *reward_sum, const cstr_episode_stats *stats,
                                       const cstr_rollout_norm *norm, void *stream) {
    if (!norm || !norm->stats || !norm->returns || !norm->workspace) return fail_arg(CSTR_EINVAL, "rollout_norm: stats, returns or workspace missing");
    if (!aligned(norm->stats, 8) || !aligned(norm->returns, 8) || !aligned(norm->workspace, 16))
        return fail_arg(CSTR_EALIGN, "rollout_norm: stats/returns 8-byte, workspace 16-byte alignment");
    if (rows <= 0 || pos0 < 0 || K < 0) return fail_arg(CSTR_EINVAL, "rollout_norm: bad size");
    uint8_t *ws = (uint8_t *)norm->workspace;
    NormLaunch nl;
    nl.stats = norm->stats;
    nl.returns = norm->returns;
    nl.ticket = (uint32_t *)ws;
    nl.partials = (double *)(ws + 16);
    nl.pending = ws + 16 + norm_grid(n) * NORM_SUMS * sizeof(double);
    nl.gamma = norm->gamma;
    nl.eps = norm->epsilon;
    nl.clip = norm->clip_obs;
    nl.training = norm->training != 0;
    nl.norm_obs = norm->norm_obs != 0;
    // one launch per env step: step k+1 acts on statistics reduced over every reactor at step k
    for (int64_t k = 0; k < K; ++k) {
        nl.prev_row = (pos0 + k + rows - 1) % rows;
        const float *nz = noise ? noise + (size_t)k * n * 2 : nullptr;
        if (int rc = rollout_fused_impl(p, n, 1, math_mode, actor_mode, actor, nullptr, packed_bf16, sigma, nz, warmup, t_base + (uint32_t)k, state,
                                        step_count, episode, static_base, rows, pos0 + k, records, reward_sum, stats, &nl, stream))
            return rc;
    }
    if (n == 0 || K == 0 || !nl.training || !nl.norm_obs) return 0;
    nl.prev_row = (pos0 + K - 1) % rows;
    rollout_norm_fix_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, nl, (float4 *)records);
    return check_launch("rollout_norm_fix_kernel");
}
