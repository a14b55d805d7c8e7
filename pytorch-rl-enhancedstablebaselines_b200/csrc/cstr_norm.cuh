// VecNormalize value maps (core/common/vec_env/vec_normalize.py:225-259), float64 arithmetic as in the reference.
#pragma once
#include <cuda_runtime.h>

namespace cstr {

// np.clip((obs - mean) / np.sqrt(var + eps), -clip, clip).astype(float32)
__device__ __forceinline__ float normalize_obs_value(float x, double mean, double var, double eps, double clip) {
    const double z = ((double)x - mean) / sqrt(var + eps);
    return (float)fmin(fmax(z, -clip), clip);
}
// np.clip(reward / np.sqrt(ret_var + eps), -clip, clip).astype(float32)
__device__ __forceinline__ float normalize_reward_value(float r, double ret_var, double eps, double clip) {
    const double z = (double)r / sqrt(ret_var + eps);
    return (float)fmin(fmax(z, -clip), clip);
}
// unnormalize_obs (:212-219) of a float32 normalised value, stored as float32: obs * np.sqrt(var + eps) + mean in float64, no FMA
__device__ __forceinline__ float unnormalize_obs_value(float z, double mean, double var, double eps) {
    return (float)__dadd_rn(__dmul_rn((double)z, sqrt(var + eps)), mean);
}

// RunningMeanStd.update_from_moments (running_mean_std.py:43-56) for the 4 observation dims and the return
__device__ __forceinline__ void update_from_moments(double &mean, double &var, double &count, double bmean, double bvar, double bcount) {
    const double delta = bmean - mean;
    const double tot = count + bcount;
    const double new_mean = mean + delta * bcount / tot;
    const double m2 = var * count + bvar * bcount + delta * delta * count * bcount / (count + bcount);
    mean = new_mean;
    var = m2 / (count + bcount);
    count = bcount + count;
}

}  // namespace cstr
