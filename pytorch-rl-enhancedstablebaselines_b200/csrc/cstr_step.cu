// K1 — the CSTR environment step kernels and their C-ABI entry points (sm_100a).
//
//   vec_step_*   one control interval for N reactors with DummyVecEnv.step_wait semantics
//                (reference core/common/vec_env/dummy_vec_env.py:56-73 over twoseriescstr.py:394-454)
//   tape_*       T control intervals per launch; the float4 state, step counter and episode counter
//                stay in registers for the whole launch, HBM is touched only for the action tape
//                (8 B/step) and the requested outputs (reward 4 B, done 1 B, obs 16 B per step)
//   reset        TwoSeriesCSTREnv.reset / generate_initial_state (twoseriescstr.py:167-269)
//
// Roofline: FP32 issue (FMA + ALU pipes) for the tape kernels, HBM for the single-step kernel at
// large N (70 B/step).  See DESIGN.md §Kernels for the per-step instruction and byte budgets.
#include "cstr_abi.cuh"
#include "cstr_device.cuh"

namespace cstr {

char *last_error_buf() {
    static thread_local char buf[256] = {0};
    return buf;
}

int sm_count() {
    static int cached = 0;
    if (cached == 0) {
        int dev = 0, v = 0;
        if (cudaGetDevice(&dev) == cudaSuccess &&
            cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0)
            cached = v;
        else
            return 148;
    }
    return cached;
}

enum { MODE_STRICT = CSTR_MATH_STRICT, MODE_FAST = CSTR_MATH_FAST };

template <int MODE>
__device__ __forceinline__ StepResult step_f32(float4 &s, float2 a, int &sc, float target, int max_steps) {
    if (MODE == MODE_STRICT) return step_strict_f32(s, a, sc, target, max_steps);
    return step_fast_f32(s, a, sc, target, max_steps);
}

// ---------------------------------------------------------------------------------------------------
// reset
// ---------------------------------------------------------------------------------------------------
__global__ void reset_kernel(cstr_env_params p, int64_t n, const uint8_t *__restrict__ mask, void *state, int is_f64,
                             int32_t *__restrict__ step_count, int32_t *__restrict__ episode, double *static_base) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || (mask && !mask[i])) return;
    double o[4];
    const int ep = episode[i];
    reset_draw(p.seed, (uint64_t)(p.env_offset + i), (uint32_t)ep, p.init_mode, static_base ? static_base + 4 * i : nullptr, o);
    if (is_f64) {
        double2 *s = reinterpret_cast<double2 *>(state) + 2 * i;
        s[0] = make_double2(o[0], o[1]);
        s[1] = make_double2(o[2], o[3]);
    } else {
        reinterpret_cast<float4 *>(state)[i] = make_float4((float)o[0], (float)o[1], (float)o[2], (float)o[3]);
    }
    step_count[i] = 0;
    episode[i] = ep + 1;
}

// ---------------------------------------------------------------------------------------------------
// one VecEnv step
// ---------------------------------------------------------------------------------------------------
// Monitor-style episode accounting (core/common/monitor.py:85-111) on device
__device__ __forceinline__ void episode_stats(int64_t i, double reward, bool done, int length, double *ep_return,
                                              double *ep_final_return, int32_t *ep_final_length) {
    if (!ep_return) return;
    double er = ep_return[i] + reward;
    if (done) {
        if (ep_final_return) ep_final_return[i] = er;
        if (ep_final_length) ep_final_length[i] = length;
        er = 0.0;
    }
    ep_return[i] = er;
}

template <int MODE>
__global__ void __launch_bounds__(256)
vec_step_f32_kernel(cstr_env_params p, int64_t n, int auto_reset, const float2 *__restrict__ actions, float4 *__restrict__ state,
                    int32_t *__restrict__ step_count, int32_t *__restrict__ episode, double *static_base,
                    float4 *__restrict__ terminal_obs, float *__restrict__ reward, uint8_t *__restrict__ done,
                    uint8_t *__restrict__ timeout, double *__restrict__ ep_return, double *__restrict__ ep_final_return,
                    int32_t *__restrict__ ep_final_length) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float4 s = state[i];
    const float2 a = actions[i];
    int sc = step_count[i];
    const StepResult r = step_f32<MODE>(s, a, sc, (float)p.target_c2, p.max_steps);
    if (terminal_obs) terminal_obs[i] = s;
    reward[i] = r.reward;
    done[i] = (uint8_t)r.truncated;
    if (timeout) timeout[i] = (uint8_t)r.truncated;  // terminated is always False -> timeout == truncated
    episode_stats(i, (double)r.reward, r.truncated, sc, ep_return, ep_final_return, ep_final_length);
    if (r.truncated && auto_reset) {
        int ep = episode[i];
        s = reset_f32_env(p, i, ep, static_base);
        episode[i] = ep;
        sc = 0;
    }
    state[i] = s;
    step_count[i] = sc;
}

__global__ void __launch_bounds__(256)
vec_step_f64_kernel(cstr_env_params p, int64_t n, int auto_reset, const double2 *__restrict__ actions, double2 *__restrict__ state,
                    int32_t *__restrict__ step_count, int32_t *__restrict__ episode, double *static_base,
                    double2 *__restrict__ terminal_obs, double *__restrict__ reward, uint8_t *__restrict__ done,
                    uint8_t *__restrict__ timeout, double *__restrict__ ep_return, double *__restrict__ ep_final_return,
                    int32_t *__restrict__ ep_final_length) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double2 s01 = state[2 * i], s23 = state[2 * i + 1];
    double s[4] = {s01.x, s01.y, s23.x, s23.y};
    const double2 a = actions[i];
    int sc = step_count[i];
    const StepResult64 r = step_f64(s, a.x, a.y, sc, p.target_c2, p.max_steps);
    if (terminal_obs) {
        terminal_obs[2 * i] = make_double2(s[0], s[1]);
        terminal_obs[2 * i + 1] = make_double2(s[2], s[3]);
    }
    reward[i] = r.reward;
    done[i] = (uint8_t)r.truncated;
    if (timeout) timeout[i] = (uint8_t)r.truncated;
    episode_stats(i, r.reward, r.truncated, sc, ep_return, ep_final_return, ep_final_length);
    if (r.truncated && auto_reset) {
        const int ep = episode[i];
        reset_draw(p.seed, (uint64_t)(p.env_offset + i), (uint32_t)ep, p.init_mode, static_base ? static_base + 4 * i : nullptr, s);
        episode[i] = ep + 1;
        sc = 0;
    }
    state[2 * i] = make_double2(s[0], s[1]);
    state[2 * i + 1] = make_double2(s[2], s[3]);
    step_count[i] = sc;
}

// ---------------------------------------------------------------------------------------------------
// T steps per launch, state in registers
// ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ void block_sum_to(double v, double *dst) {
    // warp shuffle reduce, then one atomic per warp
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(dst, v);
}

// SUM / OBS are compile-time so the common launch (rewards + dones only) carries no dead work.
// After the first step the register state is always "in the box" (it is either this kernel's own
// output or a fresh reset: a bad/NaN row truncates and is reset at once), so the loop runs the
// clamp-free cores; strict keeps the normalised state, fast keeps the RAW state across steps.
constexpr int TAPE_PF = 8;  // action loads in flight per thread

// Per-thread cursor of the tape kernel: everything one control interval touches, passed by reference so the
// unrolled loops below share one definition of "a step".  The tapes are addressed by element index t*n + i: a 32-bit
// index (IDX = uint32_t, when n*T < 2^31) makes each per-step address one IMAD.WIDE.U32 off the base and the advance one
// 32-bit add, where 64-bit pointers cost two adds per pointer and step.
template <typename IDX>
struct TapeCursor {
    float4 s;        // strict: normalised state; fast: RAW state
    int sc, ep;
    bool bad_state, unboxed;
    double acc;
    IDX ia;  // element index of the next action to prefetch for this thread
    IDX io;  // element index of this step's reward / done / obs slot
};

template <int MODE, bool CHECK, bool SUM, bool OBS, bool REW, bool DONE, typename IDX>
__device__ __forceinline__ void tape_step(const cstr_env_params &p, int64_t i, IDX n, float target, double *static_base, float2 a,
                                          float *__restrict__ rewards, uint8_t *__restrict__ dones, float4 *__restrict__ obs_tape,
                                          TapeCursor<IDX> &c) {
    StepResult r;
    if (MODE == MODE_STRICT) {
        // a state that did not come out of step_strict_core may lie outside the box (caller-injected, or a static-mode
        // reset, which the reference does not clip: twoseriescstr.py:245-253) -> clamp it on first use
        float4 sx = c.s;
        if (c.unboxed) sx = clamp_unit4(c.s);
        r = step_strict_core<CHECK>(c.s, sx, a, c.bad_state, c.sc, target, p.max_steps);
        c.unboxed = r.bad;  // a bad row keeps its (possibly unboxed) state
    } else {
        // no commit: a bad row is truncated, so the reset below overwrites whatever state it computed
        r = step_fast_raw<CHECK>(c.s, a, c.bad_state, c.sc, target, p.max_steps);
    }
    c.bad_state = false;
    if (REW) rewards[c.io] = r.reward;
    if (DONE) dones[c.io] = (uint8_t)r.truncated;
    if (SUM) c.acc += (double)r.reward;
    bool wrote_obs = false;
    if (r.truncated) {
        c.s = reset_f32_env(p, i, c.ep, static_base);
        if (OBS && MODE != MODE_STRICT) { obs_tape[c.io] = c.s; wrote_obs = true; }
        if (MODE != MODE_STRICT) c.s = fast_denorm(c.s);
        c.unboxed = p.init_mode != CSTR_INIT_RANDOM;
        c.sc = 0;
    }
    if (OBS && !wrote_obs) obs_tape[c.io] = (MODE == MODE_STRICT) ? c.s : fast_norm(c.s);
    c.io += n;
}

// SUM / OBS / REW / DONE are compile-time so the common launch (rewards + dones only) carries no dead work and no
// per-step pointer tests.
// After the first step the register state is always "in the box" (it is either this kernel's own
// output or a fresh reset: a bad/NaN row truncates and is reset at once), so the loop runs the
// clamp-free cores; strict keeps the normalised state, fast keeps the RAW state across steps.
//
// Action prefetch: a step is only ~100-240 instructions and a scheduler holds 3-4 warps at 65,536 reactors, so
// every thread keeps TAPE_PF action loads in flight in a REGISTER ring.  The main loop is unrolled by TAPE_PF with
// unconditional refills, which makes every ring slot a fixed register (a rolled loop with predicated refills made
// ptxas copy each freshly loaded value at once and exposed the full HBM latency: 70 % long-scoreboard stalls);
// the last <= 2*TAPE_PF-1 steps run through a guarded copy of the same body.
template <int MODE, bool PHILOX, bool SUM, bool OBS, bool REW, bool DONE, typename IDX>
__global__ void __launch_bounds__(256, 2)
tape_f32_kernel(cstr_env_params p, int64_t n64, int64_t T64, const float2 *__restrict__ actions, uint32_t t_base,
                float4 *__restrict__ state, int32_t *__restrict__ step_count, int32_t *__restrict__ episode, double *static_base,
                float *__restrict__ rewards, uint8_t *__restrict__ dones, float4 *__restrict__ obs_tape, double *reward_sum, float target) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < n64;
    const int T = (int)T64;
    const IDX n = (IDX)n64;
    TapeCursor<IDX> c;
    c.acc = 0.0;
    if (live) {
        c.s = state[i];
        c.bad_state = any_nan4(c.s);
        if (MODE != MODE_STRICT) c.s = fast_denorm(c.s);  // fast: RAW state in registers (clipped); strict: normalised
        c.unboxed = true;
        c.sc = step_count[i];
        c.ep = episode[i];
        c.io = (IDX)i;
        if (PHILOX) {
            const uint64_t env = (uint64_t)(p.env_offset + i);
            uint4 cache = make_uint4(0, 0, 0, 0);
            for (int t = 0; t < T; ++t) {
                const uint32_t g = t_base + (uint32_t)t;
                const float2 a = philox_action(p.seed, env, g, cache, t == 0 || (g & 1u) == 0);
                tape_step<MODE, false, SUM, OBS, REW, DONE>(p, i, n, target, static_base, a, rewards, dones, obs_tape, c);
            }
        } else {
            float2 ring[TAPE_PF];
            c.ia = (IDX)i;
#pragma unroll
            for (int j = 0; j < TAPE_PF; ++j) {
                ring[j] = (j < T) ? actions[c.ia] : make_float2(0.f, 0.f);
                if (j + 1 < T) c.ia += n;  // ends up at step min(TAPE_PF, T-1)... only dereferenced when in range
            }
            int t = 0;
            // full groups: every refill t+TAPE_PF+j (j < TAPE_PF) is in range  <=>  t + 2*TAPE_PF <= T.
            // All TAPE_PF refills of a group are issued up front, before its first step: each load then has a whole group
            // (~TAPE_PF x 100+ instructions x the resident warps) to land.  (Refilling slot j inside step j left one slot whose
            // loop-carried register copy sat right behind its load: 20 % of the stall samples on that single MOV.)
            for (; t + 2 * TAPE_PF <= T; t += TAPE_PF) {
                float2 cur[TAPE_PF];
#pragma unroll
                for (int j = 0; j < TAPE_PF; ++j) cur[j] = ring[j];
#pragma unroll
                for (int j = 0; j < TAPE_PF; ++j) {
                    ring[j] = actions[c.ia];  // action of step t + TAPE_PF + j
                    c.ia += n;
                }
#pragma unroll
                for (int j = 0; j < TAPE_PF; ++j)
                    tape_step<MODE, true, SUM, OBS, REW, DONE>(p, i, n, target, static_base, cur[j], rewards, dones, obs_tape, c);
            }
            // tail: fewer than 2*TAPE_PF steps left; refills are guarded
            for (; t < T; t += TAPE_PF) {
#pragma unroll
                for (int j = 0; j < TAPE_PF; ++j) {
                    if (t + j < T) {
                        const float2 a = ring[j];
                        if (t + TAPE_PF + j < T) {
                            ring[j] = actions[c.ia];
                            if (t + TAPE_PF + j + 1 < T) c.ia += n;
                        }
                        tape_step<MODE, true, SUM, OBS, REW, DONE>(p, i, n, target, static_base, a, rewards, dones, obs_tape, c);
                    }
                }
            }
        }
        state[i] = (MODE == MODE_STRICT) ? c.s : fast_norm(c.s);
        step_count[i] = c.sc;
        episode[i] = c.ep;
    }
    if (SUM) block_sum_to(c.acc, reward_sum);
}

template <bool PHILOX>
__global__ void __launch_bounds__(256)
tape_f64_kernel(cstr_env_params p, int64_t n, int64_t T, const double2 *__restrict__ actions, uint32_t t_base,
                double2 *__restrict__ state, int32_t *__restrict__ step_count, int32_t *__restrict__ episode, double *static_base,
                double *__restrict__ rewards, uint8_t *__restrict__ dones, double2 *__restrict__ obs_tape, double *reward_sum) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = i < n;
    double acc = 0.0;
    if (live) {
        const double2 s01 = state[2 * i], s23 = state[2 * i + 1];
        double s[4] = {s01.x, s01.y, s23.x, s23.y};
        int sc = step_count[i], ep = episode[i];
        const uint64_t env = (uint64_t)(p.env_offset + i);
        uint4 cache = make_uint4(0, 0, 0, 0);
        for (int64_t t = 0; t < T; ++t) {
            double a0, a1;
            if (PHILOX) {
                const uint32_t g = t_base + (uint32_t)t;
                const float2 a = philox_action(p.seed, env, g, cache, t == 0 || (g & 1u) == 0);
                a0 = (double)a.x;
                a1 = (double)a.y;
            } else {
                const double2 a = actions[t * n + i];
                a0 = a.x;
                a1 = a.y;
            }
            const StepResult64 r = step_f64(s, a0, a1, sc, p.target_c2, p.max_steps);
            if (rewards) rewards[t * n + i] = r.reward;
            if (dones) dones[t * n + i] = (uint8_t)r.truncated;
            if (reward_sum) acc += r.reward;
            if (r.truncated) {
                reset_draw(p.seed, env, (uint32_t)ep, p.init_mode, static_base ? static_base + 4 * i : nullptr, s);
                ep += 1;
                sc = 0;
            }
            if (obs_tape) {
                obs_tape[2 * (t * n + i)] = make_double2(s[0], s[1]);
                obs_tape[2 * (t * n + i) + 1] = make_double2(s[2], s[3]);
            }
        }
        state[2 * i] = make_double2(s[0], s[1]);
        state[2 * i + 1] = make_double2(s[2], s[3]);
        step_count[i] = sc;
        episode[i] = ep;
    }
    if (reward_sum) block_sum_to(acc, reward_sum);
}

// host scratch for cstr_tape_f32_host (grow-only, per process)
struct HostTapeScratch {
    void *buf = nullptr;
    size_t cap = 0;
    int ensure(size_t bytes) {
        if (bytes <= cap) return 0;
        if (buf) cudaFree(buf);
        buf = nullptr;
        cap = 0;
        const int rc = check_cuda(cudaMalloc(&buf, bytes), "cudaMalloc(tape scratch)");
        if (rc == 0) cap = bytes;
        return rc;
    }
};
static HostTapeScratch g_scratch;

}  // namespace cstr

using namespace cstr;

extern "C" {

int cstr_b200_abi_version(void) { return CSTR_B200_ABI_VERSION; }

const char *cstr_last_error(void) { return last_error_buf(); }

int cstr_device_info(int *sm_count_out, int *sm_clock_khz, int *cc_major, int *cc_minor) {
    int dev = 0;
    int rc = check_cuda(cudaGetDevice(&dev), "cudaGetDevice");
    if (rc) return rc;
    int v = 0;
    if (sm_count_out) {
        if ((rc = check_cuda(cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev), "attr"))) return rc;
        *sm_count_out = v;
    }
    if (sm_clock_khz) {
        if ((rc = check_cuda(cudaDeviceGetAttribute(&v, cudaDevAttrClockRate, dev), "attr"))) return rc;
        *sm_clock_khz = v;
    }
    if (cc_major) {
        if ((rc = check_cuda(cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMajor, dev), "attr"))) return rc;
        *cc_major = v;
    }
    if (cc_minor) {
        if ((rc = check_cuda(cudaDeviceGetAttribute(&v, cudaDevAttrComputeCapabilityMinor, dev), "attr"))) return rc;
        *cc_minor = v;
    }
    return 0;
}

static int check_env_args(const cstr_env_params *p, int64_t n, const void *state, const void *step_count, const void *episode,
                          const void *static_base, size_t state_align) {
    if (!p || n < 0 || !state || !step_count || !episode) return fail_arg(CSTR_EINVAL, "null pointer or negative n");
    if (p->init_mode != CSTR_INIT_RANDOM && p->init_mode != CSTR_INIT_STATIC) return fail_arg(CSTR_EINVAL, "unknown init_mode");
    if (p->init_mode == CSTR_INIT_STATIC && !static_base) return fail_arg(CSTR_EINVAL, "static init_mode needs static_base");
    if (!aligned(state, state_align)) return fail_arg(CSTR_EALIGN, "state must be 16-byte aligned");
    return 0;
}

int cstr_reset(const cstr_env_params *p, int64_t n, const uint8_t *mask, void *state, int is_f64, int32_t *step_count,
               int32_t *episode, double *static_base, void *stream) {
    if (int rc = check_env_args(p, n, state, step_count, episode, static_base, 16)) return rc;
    if (n == 0) return 0;
    const int block = 128, grid = (int)((n + block - 1) / block);
    reset_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(*p, n, mask, state, is_f64, step_count, episode, static_base);
    return check_launch("reset_kernel");
}

int cstr_vec_step_f32(const cstr_env_params *p, int64_t n, int math_mode, int auto_reset, const float *actions, float *state,
                      int32_t *step_count, int32_t *episode, double *static_base, float *terminal_obs, float *reward,
                      uint8_t *done, uint8_t *timeout, double *ep_return, double *ep_final_return, int32_t *ep_final_length,
                      void *stream) {
    if (int rc = check_env_args(p, n, state, step_count, episode, static_base, 16)) return rc;
    if (!actions || !reward || !done) return fail_arg(CSTR_EINVAL, "null actions/reward/done");
    if (!aligned(actions, 8) || (terminal_obs && !aligned(terminal_obs, 16))) return fail_arg(CSTR_EALIGN, "actions 8 B / terminal_obs 16 B alignment");
    if (math_mode != CSTR_MATH_STRICT && math_mode != CSTR_MATH_FAST) return fail_arg(CSTR_EINVAL, "unknown math_mode");
    if (n == 0) return 0;
    int grid, block;
    env_launch_geometry(n, grid, block);
    cudaStream_t st = (cudaStream_t)stream;
    if (math_mode == CSTR_MATH_STRICT)
        vec_step_f32_kernel<MODE_STRICT><<<grid, block, 0, st>>>(*p, n, auto_reset, (const float2 *)actions, (float4 *)state, step_count,
                                                                 episode, static_base, (float4 *)terminal_obs, reward, done, timeout,
                                                                 ep_return, ep_final_return, ep_final_length);
    else
        vec_step_f32_kernel<MODE_FAST><<<grid, block, 0, st>>>(*p, n, auto_reset, (const float2 *)actions, (float4 *)state, step_count,
                                                               episode, static_base, (float4 *)terminal_obs, reward, done, timeout,
                                                               ep_return, ep_final_return, ep_final_length);
    return check_launch("vec_step_f32_kernel");
}

int cstr_vec_step_f64(const cstr_env_params *p, int64_t n, int auto_reset, const double *actions, double *state, int32_t *step_count,
                      int32_t *episode, double *static_base, double *terminal_obs, double *reward, uint8_t *done, uint8_t *timeout,
                      double *ep_return, double *ep_final_return, int32_t *ep_final_length, void *stream) {
    if (int rc = check_env_args(p, n, state, step_count, episode, static_base, 16)) return rc;
    if (!actions || !reward || !done) return fail_arg(CSTR_EINVAL, "null actions/reward/done");
    if (!aligned(actions, 16) || (terminal_obs && !aligned(terminal_obs, 16))) return fail_arg(CSTR_EALIGN, "16 B alignment");
    if (n == 0) return 0;
    int grid, block;
    env_launch_geometry(n, grid, block);
    vec_step_f64_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(*p, n, auto_reset, (const double2 *)actions, (double2 *)state, step_count,
                                                                   episode, static_base, (double2 *)terminal_obs, reward, done, timeout,
                                                                   ep_return, ep_final_return, ep_final_length);
    return check_launch("vec_step_f64_kernel");
}

int cstr_tape_f32(const cstr_env_params *p, int64_t n, int64_t T, int math_mode, const float *actions, uint32_t t_base, float *state,
                  int32_t *step_count, int32_t *episode, double *static_base, float *rewards, uint8_t *dones, float *obs_tape,
                  double *reward_sum, void *stream) {
    if (int rc = check_env_args(p, n, state, step_count, episode, static_base, 16)) return rc;
    if (T < 0) return fail_arg(CSTR_EINVAL, "negative T");
    if ((actions && !aligned(actions, 8)) || (obs_tape && !aligned(obs_tape, 16))) return fail_arg(CSTR_EALIGN, "actions 8 B / obs_tape 16 B alignment");
    if (math_mode != CSTR_MATH_STRICT && math_mode != CSTR_MATH_FAST) return fail_arg(CSTR_EINVAL, "unknown math_mode");
    if (n == 0 || T == 0) return 0;
    int grid, block;
    env_launch_geometry(n, grid, block);
    cudaStream_t st = (cudaStream_t)stream;
    const bool idx32 = n <= INT32_MAX / T;  // every tape element index t*n + i fits in 31 bits
#define CSTR_LAUNCH_TAPE_IDX(MODE, PH, SUM, OBS, REW, DONE, IDX)                                                                 \
    tape_f32_kernel<MODE, PH, SUM, OBS, REW, DONE, IDX><<<grid, block, 0, st>>>(*p, n, T, (const float2 *)actions, t_base,            \
                                                                                (float4 *)state, step_count, episode, static_base,   \
                                                                                rewards, dones, (float4 *)obs_tape, reward_sum,     \
                                                                                (float)p->target_c2)
#define CSTR_LAUNCH_TAPE_RD(MODE, PH, SUM, OBS, REW, DONE)                                   \
    do {                                                                                     \
        if (idx32) CSTR_LAUNCH_TAPE_IDX(MODE, PH, SUM, OBS, REW, DONE, uint32_t);            \
        else CSTR_LAUNCH_TAPE_IDX(MODE, PH, SUM, OBS, REW, DONE, int64_t);                   \
    } while (0)
#define CSTR_LAUNCH_TAPE(MODE, PH, SUM, OBS)                                                       \
    do {                                                                                           \
        if (rewards) {                                                                             \
            if (dones) CSTR_LAUNCH_TAPE_RD(MODE, PH, SUM, OBS, true, true);                        \
            else CSTR_LAUNCH_TAPE_RD(MODE, PH, SUM, OBS, true, false);                             \
        } else {                                                                                   \
            if (dones) CSTR_LAUNCH_TAPE_RD(MODE, PH, SUM, OBS, false, true);                       \
            else CSTR_LAUNCH_TAPE_RD(MODE, PH, SUM, OBS, false, false);                            \
        }                                                                                          \
    } while (0)
#define CSTR_TAPE_FLAGS(MODE, PH)                                         \
    do {                                                                  \
        if (reward_sum) {                                                 \
            if (obs_tape) CSTR_LAUNCH_TAPE(MODE, PH, true, true);         \
            else CSTR_LAUNCH_TAPE(MODE, PH, true, false);                 \
        } else {                                                          \
            if (obs_tape) CSTR_LAUNCH_TAPE(MODE, PH, false, true);        \
            else CSTR_LAUNCH_TAPE(MODE, PH, false, false);                \
        }                                                                 \
    } while (0)
    if (math_mode == CSTR_MATH_STRICT) {
        if (actions) CSTR_TAPE_FLAGS(MODE_STRICT, false); else CSTR_TAPE_FLAGS(MODE_STRICT, true);
    } else {
        if (actions) CSTR_TAPE_FLAGS(MODE_FAST, false); else CSTR_TAPE_FLAGS(MODE_FAST, true);
    }
#undef CSTR_TAPE_FLAGS
#undef CSTR_LAUNCH_TAPE
#undef CSTR_LAUNCH_TAPE_RD
#undef CSTR_LAUNCH_TAPE_IDX
    return check_launch("tape_f32_kernel");
}

int cstr_tape_f64(const cstr_env_params *p, int64_t n, int64_t T, const double *actions, uint32_t t_base, double *state,
                  int32_t *step_count, int32_t *episode, double *static_base, double *rewards, uint8_t *dones, double *obs_tape,
                  double *reward_sum, void *stream) {
    if (int rc = check_env_args(p, n, state, step_count, episode, static_base, 16)) return rc;
    if (T < 0) return fail_arg(CSTR_EINVAL, "negative T");
    if ((actions && !aligned(actions, 16)) || (obs_tape && !aligned(obs_tape, 16))) return fail_arg(CSTR_EALIGN, "16 B alignment");
    if (n == 0 || T == 0) return 0;
    int grid, block;
    env_launch_geometry(n, grid, block);
    cudaStream_t st = (cudaStream_t)stream;
    if (actions)
        tape_f64_kernel<false><<<grid, block, 0, st>>>(*p, n, T, (const double2 *)actions, t_base, (double2 *)state, step_count, episode,
                                                       static_base, rewards, dones, (double2 *)obs_tape, reward_sum);
    else
        tape_f64_kernel<true><<<grid, block, 0, st>>>(*p, n, T, nullptr, t_base, (double2 *)state, step_count, episode, static_base,
                                                      rewards, dones, (double2 *)obs_tape, reward_sum);
    return check_launch("tape_f64_kernel");
}

int cstr_tape_f32_host(const cstr_env_params *p, int64_t n, int64_t T, int math_mode, const float *h_actions, float *h_state,
                       int32_t *h_step_count, int32_t *h_episode, float *h_rewards, uint8_t *h_dones, void *stream) {
    if (!p || n < 0 || T < 0 || !h_actions || !h_state || !h_step_count || !h_episode)
        return fail_arg(CSTR_EINVAL, "null pointer or negative size");
    if (p->init_mode != CSTR_INIT_RANDOM) return fail_arg(CSTR_EINVAL, "host tape supports init_mode=random only");
    if (n == 0 || T == 0) return 0;
    // Reactors are independent, so the batch is cut into chunks that flow through a 3-stream pipeline:
    // while chunk c computes, chunk c+1's action tape is on its way down (H2D) and chunk c-1's rewards are
    // on their way up (D2H) — PCIe is full duplex, so the end-to-end time approaches max(H2D, D2H) instead
    // of H2D + kernel + D2H.  2-D copies cut the (T, n, .) host arrays into per-chunk compact device tiles.
    static cudaStream_t streams[3] = {nullptr, nullptr, nullptr};
    int rc;
    for (int k = 0; k < 3; ++k)
        if (!streams[k] && (rc = check_cuda(cudaStreamCreateWithFlags(&streams[k], cudaStreamNonBlocking), "cudaStreamCreate"))) return rc;
    if ((rc = check_cuda(cudaStreamSynchronize((cudaStream_t)stream), "cudaStreamSynchronize(caller)"))) return rc;
    int64_t chunk = (n + 7) / 8;
    chunk = (chunk + 63) & ~(int64_t)63;
    if (chunk < 4096) chunk = n < 4096 ? n : 4096;
    const int64_t nchunks = (n + chunk - 1) / chunk;
    auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t per_chunk = up((size_t)chunk * 16) + 2 * up((size_t)chunk * 4) + up((size_t)T * chunk * 8) + up((size_t)T * chunk * 4) +
                             up((size_t)T * chunk);
    if ((rc = g_scratch.ensure(per_chunk * (size_t)nchunks))) return rc;
    for (int64_t c = 0; c < nchunks; ++c) {
        const int64_t c0 = c * chunk, cnt = (c0 + chunk <= n) ? chunk : n - c0;
        cudaStream_t st = streams[c % 3];
        char *d = (char *)g_scratch.buf + per_chunk * (size_t)c;
        char *d_state = d, *d_sc = d_state + up((size_t)chunk * 16), *d_ep = d_sc + up((size_t)chunk * 4);
        char *d_act = d_ep + up((size_t)chunk * 4), *d_rew = d_act + up((size_t)T * chunk * 8), *d_done = d_rew + up((size_t)T * chunk * 4);
        if ((rc = check_cuda(cudaMemcpyAsync(d_state, h_state + 4 * c0, (size_t)cnt * 16, cudaMemcpyHostToDevice, st), "H2D state"))) return rc;
        if ((rc = check_cuda(cudaMemcpyAsync(d_sc, h_step_count + c0, (size_t)cnt * 4, cudaMemcpyHostToDevice, st), "H2D step_count"))) return rc;
        if ((rc = check_cuda(cudaMemcpyAsync(d_ep, h_episode + c0, (size_t)cnt * 4, cudaMemcpyHostToDevice, st), "H2D episode"))) return rc;
        if ((rc = check_cuda(cudaMemcpy2DAsync(d_act, (size_t)cnt * 8, h_actions + 2 * c0, (size_t)n * 8, (size_t)cnt * 8, (size_t)T,
                                               cudaMemcpyHostToDevice, st), "H2D actions"))) return rc;
        cstr_env_params pc = *p;
        pc.env_offset = p->env_offset + c0;
        rc = cstr_tape_f32(&pc, cnt, T, math_mode, (const float *)d_act, 0u, (float *)d_state, (int32_t *)d_sc, (int32_t *)d_ep, nullptr,
                           h_rewards ? (float *)d_rew : nullptr, h_dones ? (uint8_t *)d_done : nullptr, nullptr, nullptr, (void *)st);
        if (rc) return rc;
        if (h_rewards && (rc = check_cuda(cudaMemcpy2DAsync(h_rewards + c0, (size_t)n * 4, d_rew, (size_t)cnt * 4, (size_t)cnt * 4, (size_t)T,
                                                            cudaMemcpyDeviceToHost, st), "D2H rewards"))) return rc;
        if (h_dones && (rc = check_cuda(cudaMemcpy2DAsync(h_dones + c0, (size_t)n, d_done, (size_t)cnt, (size_t)cnt, (size_t)T,
                                                          cudaMemcpyDeviceToHost, st), "D2H dones"))) return rc;
        if ((rc = check_cuda(cudaMemcpyAsync(h_state + 4 * c0, d_state, (size_t)cnt * 16, cudaMemcpyDeviceToHost, st), "D2H state"))) return rc;
        if ((rc = check_cuda(cudaMemcpyAsync(h_step_count + c0, d_sc, (size_t)cnt * 4, cudaMemcpyDeviceToHost, st), "D2H step_count"))) return rc;
        if ((rc = check_cuda(cudaMemcpyAsync(h_episode + c0, d_ep, (size_t)cnt * 4, cudaMemcpyDeviceToHost, st), "D2H episode"))) return rc;
    }
    for (int k = 0; k < 3; ++k)
        if ((rc = check_cuda(cudaStreamSynchronize(streams[k]), "cudaStreamSynchronize"))) return rc;
    return 0;
}

}  // extern "C"
