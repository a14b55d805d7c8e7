// VecNormalize on the device (SURVEY §8f-4): running mean/variance of observations and of the discounted return,
// observation/reward normalisation, and the same normalisation fused into the replay gather.
//
// Replaces, for the CSTR path (reference file:line):
//   RunningMeanStd.update / update_from_moments     core/common/running_mean_std.py:4-56
//   VecNormalize.step_wait statistics + _update_reward core/common/vec_env/vec_normalize.py:174-223
//   VecNormalize.normalize_obs / normalize_reward   core/common/vec_env/vec_normalize.py:225-259
//   ReplayBuffer._get_samples(env=VecNormalize)     core/common/buffers.py:143-155,314-323 (fused in cstr_replay.cu)
//
// stats layout (device, 16 doubles): [0:4] obs mean, [4:8] obs var, [8] obs count, [9] ret mean, [10] ret var, [11] ret count.
// Arithmetic: float64 throughout, as in the reference (RunningMeanStd keeps float64; obs - mean promotes to float64);
// the batch moments are exact double sums (the reference's np.mean over float32 rows accumulates in float32, so the
// running statistics agree to ~1e-6 relative, not bit for bit); given equal statistics the normalised values are
// bit-identical (IEEE double sqrt/div, then the same float32 rounding).
#include "cstr_abi.cuh"
#include "cstr_norm.cuh"

namespace cstr {

// scratch: [0:4] sum obs, [4:8] sum obs^2, [8] sum ret, [9] sum ret^2   (zeroed by the finalise kernel for the next call)
__global__ void __launch_bounds__(256)
norm_reduce_kernel(int64_t n, const float4 *__restrict__ obs, const float *__restrict__ reward, const uint8_t *__restrict__ done,
                   double *__restrict__ returns, double gamma, int update_obs, int update_ret, double *__restrict__ scratch) {
    double acc[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (update_obs) {
            const float4 o = obs[i];
            const double x[4] = {(double)o.x, (double)o.y, (double)o.z, (double)o.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) { acc[j] += x[j]; acc[4 + j] += x[j] * x[j]; }
        }
        if (update_ret) {
            const double r = returns[i] * gamma + (double)reward[i];  // vec_normalize.py:221
            acc[8] += r;
            acc[9] += r * r;
            returns[i] = (done && done[i]) ? 0.0 : r;  // :218 (after the statistics update)
        }
    }
    __shared__ double sh[10][8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int j = 0; j < 10; ++j) {
        double v = acc[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        if (lane == 0) sh[j][warp] = v;
    }
    __syncthreads();
    if (threadIdx.x < 10) {
        double v = 0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) v += sh[threadIdx.x][w];
        atomicAdd(scratch + threadIdx.x, v);
    }
}

__global__ void norm_finalize_kernel(int64_t n, int update_obs, int update_ret, double *__restrict__ stats, double *__restrict__ scratch) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    const double bn = (double)n;
    if (update_obs) {
        double cnt = stats[8], c = cnt;
        for (int j = 0; j < 4; ++j) {
            const double bmean = scratch[j] / bn;
            const double bvar = fmax(scratch[4 + j] / bn - bmean * bmean, 0.0);  // np.var (population variance)
            c = cnt;
            update_from_moments(stats[j], stats[4 + j], c, bmean, bvar, bn);
        }
        stats[8] = c;
    }
    if (update_ret) {
        const double bmean = scratch[8] / bn;
        const double bvar = fmax(scratch[9] / bn - bmean * bmean, 0.0);
        update_from_moments(stats[9], stats[10], stats[11], bmean, bvar, bn);
    }
    for (int j = 0; j < 10; ++j) scratch[j] = 0.0;
}

__global__ void __launch_bounds__(256)
norm_apply_kernel(int64_t n, const float4 *__restrict__ obs_in, const float *__restrict__ rew_in, const double *__restrict__ stats,
                  double eps, double clip_obs, double clip_reward, float4 *__restrict__ obs_out, float *__restrict__ rew_out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (obs_in && obs_out) {
        const float4 o = obs_in[i];
        obs_out[i] = make_float4(normalize_obs_value(o.x, stats[0], stats[4], eps, clip_obs), normalize_obs_value(o.y, stats[1], stats[5], eps, clip_obs),
                                 normalize_obs_value(o.z, stats[2], stats[6], eps, clip_obs), normalize_obs_value(o.w, stats[3], stats[7], eps, clip_obs));
    }
    if (rew_in && rew_out) rew_out[i] = normalize_reward_value(rew_in[i], stats[10], eps, clip_reward);
}

}  // namespace cstr

using namespace cstr;

extern "C" {

int cstr_norm_update(int64_t n, const float *obs, const float *reward, const uint8_t *done, double *returns, double gamma, double *stats,
                     double *scratch, void *stream) {
    if (n <= 0 || !stats || !scratch) return fail_arg(CSTR_EINVAL, "norm_update: bad size or null stats/scratch");
    const int update_obs = obs != nullptr, update_ret = reward != nullptr;
    if (update_ret && !returns) return fail_arg(CSTR_EINVAL, "norm_update: returns missing");
    if (obs && !aligned(obs, 16)) return fail_arg(CSTR_EALIGN, "norm_update: obs must be 16-byte aligned");
    if (!update_obs && !update_ret) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int block = 256;
    int grid = (int)((n + block - 1) / block);
    const int cap = sm_count() * 8;
    if (grid > cap) grid = cap;
    norm_reduce_kernel<<<grid, block, 0, st>>>(n, (const float4 *)obs, reward, done, returns, gamma, update_obs, update_ret, scratch);
    if (int rc = check_launch("norm_reduce_kernel")) return rc;
    norm_finalize_kernel<<<1, 32, 0, st>>>(n, update_obs, update_ret, stats, scratch);
    return check_launch("norm_finalize_kernel");
}

int cstr_norm_apply(int64_t n, const float *obs_in, const float *reward_in, const double *stats, double epsilon, double clip_obs,
                    double clip_reward, float *obs_out, float *reward_out, void *stream) {
    if (n < 0 || !stats) return fail_arg(CSTR_EINVAL, "norm_apply: bad size or null stats");
    if ((obs_in && !aligned(obs_in, 16)) || (obs_out && !aligned(obs_out, 16))) return fail_arg(CSTR_EALIGN, "norm_apply: obs 16-byte alignment");
    if (n == 0) return 0;
    const int block = 256, grid = (int)((n + block - 1) / block);
    norm_apply_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(n, (const float4 *)obs_in, reward_in, stats, epsilon, clip_obs, clip_reward,
                                                                (float4 *)obs_out, reward_out);
    return check_launch("norm_apply_kernel");
}

}  // extern "C"
