// Pieces shared by the two fused-rollout kernels (fp32 CUDA-core actor, bf16 tcgen05 actor):
// the reference's float32 action plumbing, the Philox exploration noise and the replay record store.
#pragma once
#include "cstr_device.cuh"
#include "cstr_norm.cuh"

namespace cstr {

// float32 action plumbing for a Box(-1,1) action space, same association as the reference:
//   predict():        u = low + (0.5*(mu+1))*(high-low)                      policies.py:375,402-413
//   _sample_action(): s = clip(2*((u-low)/(high-low)) - 1 + noise, -1, 1)    off_policy_algorithm.py:398-402
//                     a = low + (0.5*(s+1))*(high-low)                       :405
// (x+1)-1 is not the identity in float32, so the three maps are applied, not skipped (SURVEY App. A).
__device__ __forceinline__ void action_maps(float mu, float noise, float &env_action, float &buffer_action) {
    const float u = __fadd_rn(-1.0f, __fmul_rn(__fmul_rn(0.5f, __fadd_rn(mu, 1.0f)), 2.0f));
    float s = __fadd_rn(__fmul_rn(2.0f, __fmul_rn(__fadd_rn(u, 1.0f), 0.5f)), -1.0f);
    s = clampf(__fadd_rn(s, noise), -1.0f, 1.0f);
    buffer_action = s;
    env_action = __fadd_rn(-1.0f, __fmul_rn(__fmul_rn(0.5f, __fadd_rn(s, 1.0f)), 2.0f));
}

// N(0,1) pair by Box-Muller from one Philox call (stream "noise", counter = global step)
__device__ __forceinline__ float2 philox_normal2(uint64_t seed, uint64_t env, uint32_t g) {
    const uint4 r = philox_env(seed, env, g, STREAM_NOISE, 0);
    const float u1 = fmaf(u24(r.x), 1.0f, 5.9604644775390625e-08f);  // (0,1]
    const float u2 = u24(r.y);
    const float rad = sqrtf(-2.0f * __logf(u1));
    float sn, cs;
    __sincosf(6.283185307179586f * u2, &sn, &cs);
    return make_float2(rad * cs, rad * sn);
}

// Actor head -> squashed action in [-1,1] and the additive exploration noise that follows it.
//   TANH (TD3):      a = tanh(o[0..1]);  noise = sigma*N(0,1) (or the caller's tensor)        td3/policies.py:75-78, noise.py:29-48
//   GAUSSIAN (SAC):  a = tanh(mu + exp(clamp(log_std,-20,2))*eps), no additive noise          sac/policies.py:151-168
template <int KIND>
__device__ __forceinline__ void actor_head(const float o[4], float2 nz, float &a0, float &a1, float2 &add_noise) {
    if (KIND == CSTR_ACTOR_TANH) {
        a0 = tanhf(o[0]);
        a1 = tanhf(o[1]);
        add_noise = nz;
    } else {
        const float s0 = expf(clampf(o[2], -20.0f, 2.0f)), s1 = expf(clampf(o[3], -20.0f, 2.0f));
        a0 = tanhf(fmaf(s0, nz.x, o[0]));
        a1 = tanhf(fmaf(s1, nz.y, o[1]));
        add_noise = make_float2(0.0f, 0.0f);
    }
}

// Monitor semantics on device: running return per reactor; finished episodes appended to a compact list.
__device__ __forceinline__ void episode_account(const cstr_episode_stats &st, bool enabled, double &ep_ret, float reward, bool done, int length) {
    if (!enabled) return;
    ep_ret += (double)reward;
    if (done) {
        const uint32_t idx = atomicAdd(st.count, 1u);
        if (idx < st.capacity) {
            st.finished[2 * idx] = (float)ep_ret;
            st.finished[2 * idx + 1] = (float)length;
        }
        ep_ret = 0.0;
    }
}

__device__ __forceinline__ void store_record(float4 *__restrict__ rec, float4 obs, float4 next_obs, float2 act, float reward, bool done) {
    rec[0] = obs;
    rec[1] = next_obs;
    rec[2] = make_float4(act.x, act.y, reward, done ? 1.0f : 0.0f);
    rec[3] = make_float4(done ? 1.0f : 0.0f, 0.0f, 0.0f, 0.0f);  // timeout == truncated (terminated is always False)
}

// ---- VecNormalize inside the rollout (cstr_rollout_fused_norm) ----------------------------------------------------------------
// The NORM kernel variants run ONE env step per launch: the statistics every reactor's next actor input and every done row's stored
// next_obs depend on are reduced over all N reactors at the end of the step, and the grid is not co-resident.
constexpr int NORM_SUMS = 10;  // per CTA: sum x[4], sum x^2[4] of the post-reset observations, sum r, sum r^2 of the updated returns

struct NormLaunch {
    double *stats;      // the 16-double block of cstr_norm_update: S_k on entry, S_{k+1} once the launch has finished
    double *returns;    // (n,) VecNormalize.returns
    double *partials;   // [grid][NORM_SUMS], one slot per CTA
    uint32_t *ticket;   // CTAs that have written their slot; the last one merges and puts it back to 0
    uint8_t *pending;   // (n,) 1 = the reactor's record in ring row prev_row still holds the raw terminal observation
    double gamma, eps, clip;
    int64_t prev_row;   // ring row of the previous env step
    int training, norm_obs;
};

// normalize_obs with the statistics block's obs mean [0:4] and var [4:8] (read where needed, not held in registers across the actor)
__device__ __forceinline__ float4 norm_obs4(float4 s, const NormLaunch &nl) {
    const double *st = nl.stats;
    return make_float4(normalize_obs_value(s.x, st[0], st[4], nl.eps, nl.clip), normalize_obs_value(s.y, st[1], st[5], nl.eps, nl.clip),
                       normalize_obs_value(s.z, st[2], st[6], nl.eps, nl.clip), normalize_obs_value(s.w, st[3], st[7], nl.eps, nl.clip));
}
// _store_transition's next_obs of a done row (off_policy_algorithm.py:468-481): unnormalize_obs(normalize_obs(terminal)), which is not the
// identity once clip_obs binds
__device__ __forceinline__ float4 norm_round_trip4(float4 s, const NormLaunch &nl) {
    const float4 z = norm_obs4(s, nl);
    const double *st = nl.stats;
    return make_float4(unnormalize_obs_value(z.x, st[0], st[4], nl.eps), unnormalize_obs_value(z.y, st[1], st[5], nl.eps),
                       unnormalize_obs_value(z.z, st[2], st[6], nl.eps), unnormalize_obs_value(z.w, st[3], st[7], nl.eps));
}
// a done row of the previous step gets its final next_obs now that the statistics include that step's observations
__device__ __forceinline__ void norm_fix_pending(const NormLaunch &nl, int64_t i, int64_t n, float4 *records) {
    if (!nl.pending[i]) return;
    float4 *next_obs = records + ((size_t)nl.prev_row * n + i) * 4 + 1;
    *next_obs = norm_round_trip4(*next_obs, nl);
    nl.pending[i] = 0;
}
// VecNormalize.step_wait after the env step, for one reactor (vec_normalize.py:188-198,218-221): the post-reset observation and the
// updated return enter the moment sums; the return restarts at 0 on done rows (also when the statistics are frozen)
__device__ __forceinline__ void norm_account(const NormLaunch &nl, int64_t i, float4 obs_next, float reward, bool done, double acc[NORM_SUMS]) {
    double ret = nl.returns[i];
    if (nl.training) {
        if (nl.norm_obs) {
            const double x[4] = {(double)obs_next.x, (double)obs_next.y, (double)obs_next.z, (double)obs_next.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) { acc[j] += x[j]; acc[4 + j] += x[j] * x[j]; }
        }
        ret = __dadd_rn(__dmul_rn(ret, nl.gamma), (double)reward);  // returns * gamma + reward in float64, as NumPy computes it
        acc[8] += ret;
        acc[9] += ret * ret;
    }
    nl.returns[i] = done ? 0.0 : ret;
}

// fixed-order CTA sum of acc[] into sred[warp][NORM_SUMS]
template <int NT>
__device__ __forceinline__ void norm_cta_sum(const double acc[NORM_SUMS], double *sred) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < NORM_SUMS; ++j) {
        double v = acc[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) sred[warp * NORM_SUMS + j] = v;
    }
    __syncthreads();
}

// Every thread of the CTA calls this at the end of the step (training only).  Each CTA writes its sums to its own slot; the last CTA
// to finish adds the slots up in a fixed order (strided by thread, then warp tree, then warps in order: no atomics on the values, so the
// statistics are the same bits on every run) and applies RunningMeanStd.update_from_moments.  sred: (NT/32)*NORM_SUMS+1 doubles of shared
// memory the step no longer uses.
template <int NT>
__device__ __noinline__ void norm_merge(const NormLaunch &nl, int64_t n, const double acc[NORM_SUMS], double *sred) {
    constexpr int NW = NT / 32;
    __syncthreads();  // sred may alias shared memory other warps were still reading during the step
    norm_cta_sum<NT>(acc, sred);
    if (threadIdx.x == 0) {
        for (int j = 0; j < NORM_SUMS; ++j) {
            double v = 0.0;
            for (int w = 0; w < NW; ++w) v += sred[w * NORM_SUMS + j];
            nl.partials[(size_t)blockIdx.x * NORM_SUMS + j] = v;
        }
        __threadfence();
        sred[NW * NORM_SUMS] = atomicAdd(nl.ticket, 1u) == gridDim.x - 1 ? 1.0 : 0.0;
    }
    __syncthreads();
    if (sred[NW * NORM_SUMS] == 0.0) return;
    __threadfence();
    double tot[NORM_SUMS];
#pragma unroll
    for (int j = 0; j < NORM_SUMS; ++j) tot[j] = 0.0;
    for (uint32_t c = threadIdx.x; c < gridDim.x; c += NT)
#pragma unroll
        for (int j = 0; j < NORM_SUMS; ++j) tot[j] += __ldcg(nl.partials + (size_t)c * NORM_SUMS + j);
    norm_cta_sum<NT>(tot, sred);  // (thread 0 read the first sums before its ticket; every thread has read the flag)
    if (threadIdx.x != 0) return;
    double s[NORM_SUMS];
    for (int j = 0; j < NORM_SUMS; ++j) {
        s[j] = 0.0;
        for (int w = 0; w < NW; ++w) s[j] += sred[w * NORM_SUMS + j];
    }
    const double bn = (double)n;
    double *st = nl.stats;
    if (nl.norm_obs) {  // obs_rms.update(obs) (vec_normalize.py:188-193): np.mean / np.var (population) of the batch
        const double cnt = st[8];
        double c = cnt;
        for (int j = 0; j < 4; ++j) {
            const double bmean = s[j] / bn;
            const double bvar = fmax(s[4 + j] / bn - bmean * bmean, 0.0);
            c = cnt;
            update_from_moments(st[j], st[4 + j], c, bmean, bvar, bn);
        }
        st[8] = c;
    }
    const double bmean = s[8] / bn;  // ret_rms.update(returns) (:197-198)
    const double bvar = fmax(s[9] / bn - bmean * bmean, 0.0);
    update_from_moments(st[9], st[10], st[11], bmean, bvar, bn);
    *nl.ticket = 0;
}

}  // namespace cstr
