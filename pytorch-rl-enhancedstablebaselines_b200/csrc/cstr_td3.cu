// TD3 gradient step on the device (SURVEY §8f-1): everything between `replay_buffer.sample()` and the end of one
// iteration of the loop in TD3.train, as a fixed sequence of hand-written float32 kernels on one stream.
//
// Replaces (reference file:line):
//   TD3.train loop body                     core/td3/td3.py:162-206
//   Actor / ContinuousCritic forward        core/td3/policies.py:58,75-78, core/common/policies.py:966-987 (create_mlp, torch_layers.py:110-183)
//   autograd backward of those MLPs         (torch autograd; restated in oracle/td3_oracle.py::mlp_backward)
//   th.optim.Adam.step (defaults)           torch/optim/adam.py single-tensor path
//   polyak_update                           core/common/utils.py:457-481
//
// Arithmetic: float32 FFMA (the reference's torch default: no TF32/BF16), so parity with the oracle is summation-order
// tolerance (tests/test_gpu_td3.py).  Everything is deterministic: no atomics; batch reductions go through fixed-order
// partial sums.
//
// Parameter block (floats): [actor | critic0 | critic1], each net = W1 (H1,in) b1 W2 (H2,H1) b2 W3 (out,H2) b3 in torch nn.Linear
// layout, every tensor padded to a multiple of 4 floats (16-byte aligned rows for float4 access).  `params`, `targets`,
// `grads`, `adam_m`, `adam_v` all share that layout, so Adam / polyak / the NCCL gradient bucket are single flat ranges.
#include "cstr_abi.cuh"
#include "cstr_device.cuh"

#include <algorithm>
#include <cstdlib>
#include <cstring>

namespace cstr {

constexpr int OBS = 4, ACT = 2;

// Programmatic dependent launch: the update is a chain of 25-50 short kernels on one stream (one CUDA graph at small batches), so
// the gap between two kernels costs as much as the kernels.  Every kernel here starts with pdl_enter(): wait until the kernel before
// it has completed and its writes are visible (same ordering as a plain stream), then let the kernel after it be launched — its CTAs
// become resident and stop at their own wait while this one computes, which hides the launch latency of the next node.  At most one
// kernel runs ahead, and never past its wait, so data dependencies (including write-after-read on the reused workspace slabs) hold.
// Measured (B200, [400,300] nets): launch by launch 0.174 -> 0.141 ms per TD3 update at batch 256 (SAC 0.216 -> 0.159), 0.568 -> 0.542 at
// 4096; inside a captured CUDA graph the node-to-node latency is already that low and the early-resident CTAs cost a few percent, so
// the attribute is left off while the stream is capturing.  CSTR_TD3_PDL=0: never; 2: also under capture (griddepcontrol.* are no-ops
// in a kernel launched without the attribute).
__device__ __forceinline__ void pdl_enter() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;");
}

static int pdl_mode() {
    static const int mode = [] {
        const char *e = std::getenv("CSTR_TD3_PDL");
        return (e && e[0] >= '0' && e[0] <= '2') ? e[0] - '0' : 1;
    }();
    return mode;
}

static bool pdl_for(cudaStream_t st) {
    const int mode = pdl_mode();
    if (mode != 1) return mode == 2;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    return cudaStreamIsCapturing(st, &cs) == cudaSuccess && cs == cudaStreamCaptureStatusNone;
}

template <typename... KArgs, typename... Args>
static inline void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid, cfg.blockDim = block, cfg.dynamicSmemBytes = smem, cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr, cfg.numAttrs = pdl_for(st) ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);  // errors surface through check_launch (cudaGetLastError)
}

struct NetLayout {  // offsets (floats) inside one net block
    int in, out, h1, h2;
    int64_t w1, b1, w2, b2, w3, b3, size;
};

__host__ __device__ inline int64_t pad4(int64_t n) { return (n + 3) & ~(int64_t)3; }

inline NetLayout net_layout(int in, int out, int h1, int h2) {
    NetLayout L;
    L.in = in, L.out = out, L.h1 = h1, L.h2 = h2;
    int64_t o = 0;
    L.w1 = o, o += pad4((int64_t)h1 * in);
    L.b1 = o, o += pad4(h1);
    L.w2 = o, o += pad4((int64_t)h2 * h1);
    L.b2 = o, o += pad4(h2);
    L.w3 = o, o += pad4((int64_t)out * h2);
    L.b3 = o, o += pad4(out);
    L.size = o;
    return L;
}

struct Td3Layout {
    NetLayout actor, critic;
    int64_t actor_off, critic_off[2], total;
};

inline Td3Layout td3_layout(int h1, int h2, int actor_out = ACT) {  // actor_out = 2 (TD3: tanh head) or 4 (SAC: [mu; log_std] head)
    Td3Layout T;
    T.actor = net_layout(OBS, actor_out, h1, h2);
    T.critic = net_layout(OBS + ACT, 1, h1, h2);
    T.actor_off = 0;
    T.critic_off[0] = T.actor.size;
    T.critic_off[1] = T.actor.size + T.critic.size;
    T.total = T.actor.size + 2 * T.critic.size;
    return T;
}

// ------------------------------------------------------------------------------------------------------------------
// layer 1: h1[z][b][j] = relu(b1[j] + sum_i x[b][i] W1[j][i]),  x = [obs | act]  (K = 4 or 6: no GEMM needed)
// ------------------------------------------------------------------------------------------------------------------
constexpr int L1_ROWS = 8;  // batch rows per thread: the 4 x IN weights of the thread's four units stay in registers

template <int IN>
__global__ void __launch_bounds__(256)
td3_layer1_kernel(int B, int H1, const float4 *__restrict__ obs, const float2 *__restrict__ act, const float *__restrict__ W1, const float *__restrict__ b1,
                  int64_t w_stride_z, float *__restrict__ h1, int64_t h_stride_z) {
    pdl_enter();
    const int q = H1 >> 2;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int row_groups = (B + L1_ROWS - 1) / L1_ROWS;
    if (i >= (int64_t)row_groups * q) return;
    const int b0 = (int)(i / q) * L1_ROWS, j = (int)(i % q) * 4;  // a warp covers 32 consecutive unit-quads of one row group
    const int z = blockIdx.y;
    const float *W = W1 + z * w_stride_z + (int64_t)j * IN;
    float w[4][IN];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int k = 0; k < IN; ++k) w[c][k] = __ldg(W + c * IN + k);
    const float4 bias = *reinterpret_cast<const float4 *>(b1 + z * w_stride_z + j);
    float *out = h1 + z * h_stride_z + j;
#pragma unroll
    for (int r = 0; r < L1_ROWS; ++r) {
        const int b = b0 + r;
        if (b >= B) break;
        const float4 o = obs[b];
        float x[IN];
        x[0] = o.x, x[1] = o.y, x[2] = o.z, x[3] = o.w;
        if (IN == 6) {
            const float2 a = act[b];
            x[4] = a.x, x[5] = a.y;
        }
        float v[4] = {bias.x, bias.y, bias.z, bias.w};
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int k = 0; k < IN; ++k) v[c] = fmaf(x[k], w[c][k], v[c]);
        *reinterpret_cast<float4 *>(out + (int64_t)b * H1) = make_float4(fmaxf(v[0], 0.f), fmaxf(v[1], 0.f), fmaxf(v[2], 0.f), fmaxf(v[3], 0.f));
    }
}

// ------------------------------------------------------------------------------------------------------------------
// the hidden-layer GEMM (H1 x H2), three roles from one tiled FFMA kernel:
//   FWD    h2  = relu(h1  @ W2^T + b2)        A = h1  (M=B, K=H1, k-contiguous)   Bm = W2 (N=H2 rows, k-contiguous)
//   DGRAD  dz1 = (dz2 @ W2) * (h1 > 0)        A = dz2 (M=B, K=H2, k-contiguous)   Bm = W2 (K=H2 rows, n-contiguous)
//   WGRAD  dW2 = dz2^T @ h1   (split over B)  A = dz2 (K=B rows, m-contiguous)    Bm = h1 (K=B rows, n-contiguous)
// CTA tile 128 x 64 x 16, 256 threads, 8 x 4 accumulators per thread, double-buffered shared memory.
// ------------------------------------------------------------------------------------------------------------------
enum { G_FWD = 0, G_DGRAD = 1, G_WGRAD = 2 };
constexpr int BM = 128, BN = 64, BK = 16, LDA_S = BM + 4, LDB_S = BN + 4;

struct GemmArgs {
    const float *A, *Bm, *aux;
    float *C;
    int M, N, K, lda, ldb, ldc, ldaux;
    int64_t a_z, b_z, c_z, aux_z;  // per-net strides (floats)
    int splits, k_per_split;
    int64_t c_split;               // split-K: slab stride
    int raw_partials;              // FWD/DGRAD split over K (small batches): store raw partial sums, td3_splitk_finish_kernel applies the epilogue
    float *split_buf;              // scratch for those partials (NULL: never split)
    int64_t split_cap;             // its capacity in floats
};

template <int MODE, bool RAW = false>  // RAW: forward / dgrad split over K, raw partial sums out (compile-time so the main path keeps its registers)
__global__ void __launch_bounds__(256, 2) td3_gemm_kernel(GemmArgs g) {
    pdl_enter();
    __shared__ __align__(16) float As[2][BK][LDA_S];
    __shared__ __align__(16) float Bs[2][BK][LDB_S];
    const int tid = threadIdx.x, tn = tid & 15, tm = tid >> 4;
    const int z = blockIdx.z / g.splits, split = blockIdx.z % g.splits;
    const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
    const float *A = g.A + z * g.a_z, *Bm = g.Bm + z * g.b_z;
    int k_begin = 0, k_end = g.K;
    constexpr bool partial = MODE == G_WGRAD || RAW;
    if (partial) {
        k_begin = split * g.k_per_split;
        k_end = min(g.K, k_begin + g.k_per_split);
    }
    float acc[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    float4 ra[2], rb;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    auto load_global = [&](int k0) {
        if (MODE == G_WGRAD) {  // A rows = k, m-contiguous: 16 x 128 floats = 512 float4
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int idx = tid + i * 256, kk = idx >> 5, mq = (idx & 31) * 4;
                const int k = k0 + kk, m = m0 + mq;
                ra[i] = (k < k_end && m < g.M) ? *reinterpret_cast<const float4 *>(A + (int64_t)k * g.lda + m) : zero4;
            }
        } else {  // A rows = m, k-contiguous: 128 x 16 floats
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int idx = tid + i * 256, row = idx >> 2, kq = (idx & 3) * 4;
                const int m = m0 + row, k = k0 + kq;
                ra[i] = (m < g.M && k < k_end) ? *reinterpret_cast<const float4 *>(A + (int64_t)m * g.lda + k) : zero4;
            }
        }
        if (MODE == G_FWD) {  // Bm rows = n, k-contiguous: 64 x 16
            const int row = tid >> 2, kq = (tid & 3) * 4;
            const int n = n0 + row, k = k0 + kq;
            rb = (n < g.N && k < k_end) ? *reinterpret_cast<const float4 *>(Bm + (int64_t)n * g.ldb + k) : zero4;
        } else {  // Bm rows = k, n-contiguous: 16 x 64
            const int kk = tid >> 4, nq = (tid & 15) * 4;
            const int k = k0 + kk, n = n0 + nq;
            rb = (k < k_end && n < g.N) ? *reinterpret_cast<const float4 *>(Bm + (int64_t)k * g.ldb + n) : zero4;
        }
    };
    auto store_shared = [&](int buf) {
        if (MODE == G_WGRAD) {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int idx = tid + i * 256, kk = idx >> 5, mq = (idx & 31) * 4;
                *reinterpret_cast<float4 *>(&As[buf][kk][mq]) = ra[i];
            }
        } else {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int idx = tid + i * 256, row = idx >> 2, kq = (idx & 3) * 4;
                As[buf][kq + 0][row] = ra[i].x;
                As[buf][kq + 1][row] = ra[i].y;
                As[buf][kq + 2][row] = ra[i].z;
                As[buf][kq + 3][row] = ra[i].w;
            }
        }
        if (MODE == G_FWD) {
            const int row = tid >> 2, kq = (tid & 3) * 4;
            Bs[buf][kq + 0][row] = rb.x;
            Bs[buf][kq + 1][row] = rb.y;
            Bs[buf][kq + 2][row] = rb.z;
            Bs[buf][kq + 3][row] = rb.w;
        } else {
            const int kk = tid >> 4, nq = (tid & 15) * 4;
            *reinterpret_cast<float4 *>(&Bs[buf][kk][nq]) = rb;
        }
    };

    const int n_iter = (k_end - k_begin + BK - 1) / BK;
    if (n_iter > 0) {
        load_global(k_begin);
        store_shared(0);
    }
    __syncthreads();
    for (int it = 0; it < n_iter; ++it) {
        const int buf = it & 1;
        if (it + 1 < n_iter) load_global(k_begin + (it + 1) * BK);
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            const float4 a0 = *reinterpret_cast<const float4 *>(&As[buf][kk][tm * 8]);
            const float4 a1 = *reinterpret_cast<const float4 *>(&As[buf][kk][tm * 8 + 4]);
            const float4 b = *reinterpret_cast<const float4 *>(&Bs[buf][kk][tn * 4]);
            const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        if (it + 1 < n_iter) store_shared(buf ^ 1);
        __syncthreads();
    }

    const int n = n0 + tn * 4;
    if (n >= g.N) return;
    float *C = g.C + z * g.c_z + (partial ? split * g.c_split : 0);
    float4 bias = zero4;
    if (MODE == G_FWD && !RAW) bias = *reinterpret_cast<const float4 *>(g.aux + z * g.aux_z + n);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = m0 + tm * 8 + i;
        if (m >= g.M) break;
        float4 v = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        if (RAW) {
        } else if (MODE == G_FWD) {
            v = make_float4(fmaxf(v.x + bias.x, 0.f), fmaxf(v.y + bias.y, 0.f), fmaxf(v.z + bias.z, 0.f), fmaxf(v.w + bias.w, 0.f));
        } else if (MODE == G_DGRAD) {
            const float4 h = *reinterpret_cast<const float4 *>(g.aux + z * g.aux_z + (int64_t)m * g.ldaux + n);
            v = make_float4(h.x > 0.f ? v.x : 0.f, h.y > 0.f ? v.y : 0.f, h.z > 0.f ? v.z : 0.f, h.w > 0.f ? v.w : 0.f);
        }
        *reinterpret_cast<float4 *>(C + (int64_t)m * g.ldc + n) = v;
    }
}

// second stage of a split-K forward / dgrad GEMM: sum the partial slabs in order, then bias+relu or the relu mask
template <int MODE>
__global__ void __launch_bounds__(256) td3_splitk_finish_kernel(GemmArgs g, const float *__restrict__ slabs, int splits, int64_t slab_stride, float *__restrict__ out) {
    pdl_enter();
    const int n4 = g.N >> 2, z = blockIdx.y;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (int64_t)g.M * n4) return;
    const int m = (int)(i / n4), n = (int)(i % n4) * 4;
    const float *p = slabs + (int64_t)z * g.M * g.N + (int64_t)m * g.N + n;
    float4 v = *reinterpret_cast<const float4 *>(p);
    for (int s = 1; s < splits; ++s) {
        const float4 u = *reinterpret_cast<const float4 *>(p + s * slab_stride);
        v.x += u.x, v.y += u.y, v.z += u.z, v.w += u.w;
    }
    if (MODE == G_FWD) {
        const float4 b = *reinterpret_cast<const float4 *>(g.aux + z * g.aux_z + n);
        v = make_float4(fmaxf(v.x + b.x, 0.f), fmaxf(v.y + b.y, 0.f), fmaxf(v.z + b.z, 0.f), fmaxf(v.w + b.w, 0.f));
    } else {
        const float4 h = *reinterpret_cast<const float4 *>(g.aux + z * g.aux_z + (int64_t)m * g.ldaux + n);
        v = make_float4(h.x > 0.f ? v.x : 0.f, h.y > 0.f ? v.y : 0.f, h.z > 0.f ? v.z : 0.f, h.w > 0.f ? v.w : 0.f);
    }
    *reinterpret_cast<float4 *>(out + z * g.c_z + (int64_t)m * g.ldc + n) = v;
}

}  // namespace cstr
#include "cstr_td3_tc.cuh"
namespace cstr {

// ------------------------------------------------------------------------------------------------------------------
// row heads: one warp per batch row
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__device__ __forceinline__ float row_dot(const float *__restrict__ h, const float *__restrict__ w, int H, int lane) {
    float s = 0.f;
    for (int k = lane * 4; k < H; k += 128) {
        const float4 a = *reinterpret_cast<const float4 *>(h + k), b = *reinterpret_cast<const float4 *>(w + k);
        s = fmaf(a.x, b.x, s), s = fmaf(a.y, b.y, s), s = fmaf(a.z, b.z, s), s = fmaf(a.w, b.w, s);
    }
    return warp_sum(s);
}

// actor head: a = tanh(h2 @ W3^T + b3) [+ clip(noise) -> clamp(-1,1)]                              td3.py:168-170 / policies.py:75-78
__global__ void __launch_bounds__(256)
td3_actor_head_kernel(int B, int H2, const float *__restrict__ h2, const float *__restrict__ W3, const float *__restrict__ b3, int smooth,
                      const float2 *__restrict__ noise, float sigma, float clip, uint64_t seed, uint32_t update_index, const float *__restrict__ dev_scalars,
                      float2 *__restrict__ out) {
    pdl_enter();
    const int lane = threadIdx.x & 31, b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    const float *h = h2 + (int64_t)b * H2;
    const float p0 = row_dot(h, W3, H2, lane) + b3[0], p1 = row_dot(h, W3 + H2, H2, lane) + b3[1];
    if (lane) return;
    float a0 = tanhf(p0), a1 = tanhf(p1);
    if (smooth) {
        float2 nz;
        if (noise) nz = noise[b];
        else {
            const uint32_t ui = dev_scalars ? __float_as_uint(dev_scalars[4]) : update_index;  // graph mode: counter lives on the device
            const uint4 r = philox_env(seed, (uint64_t)b, ui, STREAM_TD3, 0);
            const float u1 = fmaf(u24(r.x), 1.0f, 5.9604644775390625e-08f), u2 = u24(r.y);
            const float rad = sqrtf(-2.0f * logf(u1));
            float sn, cs;
            sincospif(2.0f * u2, &sn, &cs);
            nz = make_float2(sigma * rad * cs, sigma * rad * sn);
        }
        a0 = fminf(fmaxf(a0 + fminf(fmaxf(nz.x, -clip), clip), -1.f), 1.f);
        a1 = fminf(fmaxf(a1 + fminf(fmaxf(nz.y, -clip), clip), -1.f), 1.f);
    }
    out[b] = make_float2(a0, a1);
}

// target head: target = r + (1 - done) * gamma * min(q1_target, q2_target)                         td3.py:173-175
__global__ void __launch_bounds__(256)
td3_target_head_kernel(int B, int H2, const float *__restrict__ h2, int64_t h_z, const float *__restrict__ W3, const float *__restrict__ b3, int64_t w_z,
                       const float *__restrict__ rewards, const float *__restrict__ dones, float gamma, int n_critics, float *__restrict__ target) {
    pdl_enter();
    const int lane = threadIdx.x & 31, b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    float q = row_dot(h2 + (int64_t)b * H2, W3, H2, lane) + b3[0];
    if (n_critics > 1) q = fminf(q, row_dot(h2 + h_z + (int64_t)b * H2, W3 + w_z, H2, lane) + b3[w_z]);  // DDPG (n_critics = 1): no min
    if (lane == 0) target[b] = rewards[b] + (1.f - dones[b]) * gamma * q;
}

// critic head (z = critic): q = h2 . w3 + b3; loss += (q-target)^2; dq = 2 (q-target)/B; dz2 = dq * w3 * (h2 > 0)   td3.py:178-186
// policy head  (POLICY):    q1 = h2 . w3 + b3; loss += q1;          dq = -1/B                                        td3.py:191
template <bool POLICY>
__global__ void __launch_bounds__(256)
td3_critic_head_kernel(int B, int H2, const float *__restrict__ h2, int64_t h_z, const float *__restrict__ W3, const float *__restrict__ b3, int64_t w_z,
                       const float *__restrict__ target, float dq_scale, float *__restrict__ dq_out, float *__restrict__ dz2,
                       float *__restrict__ loss_partial) {
    pdl_enter();
    __shared__ float sl[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, b = blockIdx.x * 8 + warp, z = blockIdx.y;
    float contrib = 0.f;
    if (b < B) {
        const float *h = h2 + z * h_z + (int64_t)b * H2, *w = W3 + z * w_z;
        const float q = row_dot(h, w, H2, lane) + b3[z * w_z];
        float dq;
        if (POLICY) {
            contrib = q;
            dq = -1.f / (float)B;
        } else {
            const float diff = q - target[b];
            contrib = diff * diff;
            dq = dq_scale * diff;  // TD3: sum_i mse -> 2/B; SAC: 0.5 * sum_i mse -> 1/B
        }
        if (lane == 0) dq_out[(int64_t)z * B + b] = dq;
        float *d = dz2 + z * h_z + (int64_t)b * H2;
        for (int k = lane * 4; k < H2; k += 128) {
            const float4 a = *reinterpret_cast<const float4 *>(h + k), ww = *reinterpret_cast<const float4 *>(w + k);
            *reinterpret_cast<float4 *>(d + k) =
                make_float4(a.x > 0.f ? dq * ww.x : 0.f, a.y > 0.f ? dq * ww.y : 0.f, a.z > 0.f ? dq * ww.z : 0.f, a.w > 0.f ? dq * ww.w : 0.f);
        }
    }
    if (lane == 0) sl[warp] = contrib;
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.f;
        for (int i = 0; i < 8; ++i) s += sl[i];
        loss_partial[(int64_t)z * gridDim.x + blockIdx.x] = s;
    }
}

// policy gradient through the critic input and the tanh:  da = dz1c @ W1c[:, 4:6];  dpre = da * (1 - a^2);
// dz2a = (dpre @ W3a) * (h2a > 0)                                                                   td3.py:191-196 (autograd)
__global__ void __launch_bounds__(256)
td3_actor_bwd_head_kernel(int B, int H1, int H2, const float *__restrict__ dz1c, const float *__restrict__ W1c, const float2 *__restrict__ a_pi,
                          const float *__restrict__ W3a, const float *__restrict__ h2a, float2 *__restrict__ dpre_out, float *__restrict__ dz2a) {
    pdl_enter();
    const int lane = threadIdx.x & 31, b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    const float *d = dz1c + (int64_t)b * H1;
    float s0 = 0.f, s1 = 0.f;
    for (int j = lane; j < H1; j += 32) {
        const float v = d[j];
        s0 = fmaf(v, __ldg(W1c + j * (OBS + ACT) + OBS), s0);
        s1 = fmaf(v, __ldg(W1c + j * (OBS + ACT) + OBS + 1), s1);
    }
    s0 = warp_sum(s0), s1 = warp_sum(s1);
    const float2 a = a_pi[b];
    const float p0 = s0 * (1.f - a.x * a.x), p1 = s1 * (1.f - a.y * a.y);
    if (lane == 0) dpre_out[b] = make_float2(p0, p1);
    const float *h = h2a + (int64_t)b * H2;
    float *o = dz2a + (int64_t)b * H2;
    for (int k = lane * 4; k < H2; k += 128) {
        const float4 hh = *reinterpret_cast<const float4 *>(h + k);
        const float4 w0 = *reinterpret_cast<const float4 *>(W3a + k), w1 = *reinterpret_cast<const float4 *>(W3a + H2 + k);
        *reinterpret_cast<float4 *>(o + k) = make_float4(hh.x > 0.f ? fmaf(p1, w1.x, p0 * w0.x) : 0.f, hh.y > 0.f ? fmaf(p1, w1.y, p0 * w0.y) : 0.f,
                                                         hh.z > 0.f ? fmaf(p1, w1.z, p0 * w0.z) : 0.f, hh.w > 0.f ? fmaf(p1, w1.w, p0 * w0.w) : 0.f);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// SAC heads (core/sac/sac.py:213-281, core/sac/policies.py:147-175, core/common/distributions.py:207-260)
// ------------------------------------------------------------------------------------------------------------------
constexpr float SAC_LOG_STD_MIN = -20.f, SAC_LOG_STD_MAX = 2.f, SAC_SQUASH_EPS = 1e-6f, SAC_HALF_LOG_2PI = 0.91893853320467274f;

// squashed-Gaussian actor head: [mean; log_std] = h2 @ W3^T + b3 (W3 is (4,H2)), u = mean + std*eps, a = tanh(u),
// log_prob = sum_i [-(u-mean)^2/(2 std^2) - log_std - 0.5 log 2pi] - sum_i log(1 - a^2 + 1e-6).
// call 0 = actions_pi (keeps what the backward needs), call 1 = next_actions (no grad).
__global__ void __launch_bounds__(256)
sac_actor_head_kernel(int B, int H2, const float *__restrict__ h2, const float *__restrict__ W3, const float *__restrict__ b3, const float2 *__restrict__ eps_in,
                      uint64_t seed, uint32_t update_index, const float *__restrict__ dev_scalars, uint32_t call, float2 *__restrict__ act_out,
                      float *__restrict__ logp_out,
                      float2 *__restrict__ std_eps_out, float2 *__restrict__ raw_out, float *__restrict__ lp_partial) {
    pdl_enter();
    __shared__ float sl[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, b = blockIdx.x * 8 + warp;
    float lp = 0.f;
    if (b < B) {
        const float *h = h2 + (int64_t)b * H2;
        float y[4];
#pragma unroll
        for (int o = 0; o < 4; ++o) y[o] = row_dot(h, W3 + (int64_t)o * H2, H2, lane) + b3[o];
        if (lane == 0) {
            float2 e;
            if (eps_in) e = eps_in[b];
            else {
                const uint32_t ui = dev_scalars ? __float_as_uint(dev_scalars[4]) : update_index;
                const uint4 r = philox_env(seed, (uint64_t)b, ui, STREAM_TD3, call);
                const float u1 = fmaf(u24(r.x), 1.0f, 5.9604644775390625e-08f), u2 = u24(r.y);
                const float rad = sqrtf(-2.0f * logf(u1));
                float sn, cs;
                sincospif(2.0f * u2, &sn, &cs);
                e = make_float2(rad * cs, rad * sn);
            }
            const float ev[2] = {e.x, e.y};
            float a[2], se[2];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const float ls = fminf(fmaxf(y[2 + i], SAC_LOG_STD_MIN), SAC_LOG_STD_MAX), sd = expf(ls);
                se[i] = sd * ev[i];
                const float u = y[i] + se[i], d = u - y[i];
                a[i] = tanhf(u);
                lp += -(d * d) / (2.f * sd * sd) - ls - SAC_HALF_LOG_2PI - logf(1.f - a[i] * a[i] + SAC_SQUASH_EPS);
            }
            act_out[b] = make_float2(a[0], a[1]);
            logp_out[b] = lp;
            if (std_eps_out) std_eps_out[b] = make_float2(se[0], se[1]);
            if (raw_out) raw_out[b] = make_float2(y[2], y[3]);
        }
    }
    if (lp_partial) {
        if (lane == 0) sl[warp] = lp;
        __syncthreads();
        if (threadIdx.x == 0) {
            float t = 0.f;
            for (int i = 0; i < 8; ++i) t += sl[i];
            lp_partial[blockIdx.x] = t;
        }
    }
}

// entropy coefficient: ent_coef = exp(log_ent_coef) BEFORE the step (used by this update's target and actor loss),
// loss = -(log_ent_coef * (log_prob + target_entropy)).mean(), one Adam step on the scalar            sac.py:226-243
// scalars[5] = ent_coef of this update.  losses: [4] += ent_coef_loss, [5] += 1, [6] += ent_coef, [7] += 1.
// mode bit 0: form the gradient (-> grad[0]); bit 1: Adam step from grad[0] (split for the data-parallel all-reduce in between).
__global__ void sac_ent_coef_kernel(int B, int n_partial, const float *__restrict__ lp_partial, float target_entropy, float *__restrict__ log_ent_coef,
                                    float *__restrict__ grad, float *__restrict__ m, float *__restrict__ v, float beta1, float beta2, float eps,
                                    float step_size_arg, float bc2_sqrt_arg, int use_dev_scalars, float *__restrict__ scalars, float *__restrict__ losses,
                                    int mode) {
    pdl_enter();
    __shared__ float sl[256];
    if (mode & 1) {
        float s = 0.f;
        for (int k = threadIdx.x; k < n_partial; k += 256) s += lp_partial[k];
        sl[threadIdx.x] = s;
        __syncthreads();
        for (int o = 128; o > 0; o >>= 1) {
            if ((int)threadIdx.x < o) sl[threadIdx.x] += sl[threadIdx.x + o];
            __syncthreads();
        }
    }
    if (threadIdx.x) return;
    const float step_size = use_dev_scalars ? scalars[0] : step_size_arg, bc2_sqrt = use_dev_scalars ? scalars[1] : bc2_sqrt_arg;
    const float le = log_ent_coef[0];
    if (mode & 1) {
        const float mean_term = sl[0] / (float)B + target_entropy;  // mean(log_prob + target_entropy)
        grad[0] = -mean_term;
        scalars[5] = expf(le);
        if (losses) {
            losses[4] += -(le * mean_term), losses[5] += 1.f;
            losses[6] += scalars[5], losses[7] += 1.f;
        }
    }
    if (!(mode & 2)) return;
    const float g = grad[0];
    float mm = m[0], vv = v[0];
    mm = mm + (g - mm) * (1.f - beta1);
    vv = vv * beta2 + (1.f - beta2) * g * g;
    log_ent_coef[0] = le - step_size * (mm / (sqrtf(vv) / bc2_sqrt + eps));
    m[0] = mm, v[0] = vv;
}

// target = r + (1 - done) * gamma * (min(q1_t, q2_t) - ent_coef * next_log_prob)                      sac.py:246-254
__global__ void __launch_bounds__(256)
sac_target_head_kernel(int B, int H2, const float *__restrict__ h2, int64_t h_z, const float *__restrict__ W3, const float *__restrict__ b3, int64_t w_z,
                       const float *__restrict__ rewards, const float *__restrict__ dones, const float *__restrict__ next_logp,
                       const float *__restrict__ scalars, float gamma, float *__restrict__ target) {
    pdl_enter();
    const int lane = threadIdx.x & 31, b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    const float q0 = row_dot(h2 + (int64_t)b * H2, W3, H2, lane) + b3[0];
    const float q1 = row_dot(h2 + h_z + (int64_t)b * H2, W3 + w_z, H2, lane) + b3[w_z];
    if (lane == 0) target[b] = rewards[b] + (1.f - dones[b]) * gamma * (fminf(q0, q1) - scalars[5] * next_logp[b]);
}

// actor loss head: q_i(s, a_pi) for both critics, min -> the gradient -1/B goes to the smaller one (first on ties, as torch.min);
// loss partial = ent_coef * log_prob - min q; dz2[z] = dq[z] * w3[z] * (h2[z] > 0)                                 sac.py:271-276
__global__ void __launch_bounds__(256)
sac_qmin_head_kernel(int B, int H2, const float *__restrict__ h2, int64_t h_z, const float *__restrict__ W3, const float *__restrict__ b3, int64_t w_z,
                     const float *__restrict__ logp, const float *__restrict__ scalars, float *__restrict__ dz2, float *__restrict__ loss_partial) {
    pdl_enter();
    __shared__ float sl[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, b = blockIdx.x * 8 + warp;
    float contrib = 0.f;
    if (b < B) {
        const float *h0 = h2 + (int64_t)b * H2, *h1 = h0 + h_z;
        const float q0 = row_dot(h0, W3, H2, lane) + b3[0], q1 = row_dot(h1, W3 + w_z, H2, lane) + b3[w_z];
        const bool pick0 = q0 <= q1;
        contrib = scalars[5] * logp[b] - (pick0 ? q0 : q1);
        const float g = -1.f / (float)B;
        for (int z = 0; z < 2; ++z) {
            const float dq = (z == 0) == pick0 ? g : 0.f;
            const float *h = z ? h1 : h0, *w = W3 + z * w_z;
            float *d = dz2 + z * h_z + (int64_t)b * H2;
            for (int k = lane * 4; k < H2; k += 128) {
                const float4 a = *reinterpret_cast<const float4 *>(h + k), ww = *reinterpret_cast<const float4 *>(w + k);
                *reinterpret_cast<float4 *>(d + k) =
                    make_float4(a.x > 0.f ? dq * ww.x : 0.f, a.y > 0.f ? dq * ww.y : 0.f, a.z > 0.f ? dq * ww.z : 0.f, a.w > 0.f ? dq * ww.w : 0.f);
            }
        }
    }
    if (lane == 0) sl[warp] = contrib;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
        for (int i = 0; i < 8; ++i) t += sl[i];
        loss_partial[blockIdx.x] = t;
    }
}

// through the critics' input layers and the squashed Gaussian into the actor head:
//   da = sum_z dz1c[z] @ W1c[z][:, 4:6];  du = da (1-a^2) + (ent_coef/B) 2a(1-a^2)/(1-a^2+1e-6);  dmean = du;
//   dlog_std = (du * std*eps - ent_coef/B) * [log_std not clamped];  dz2a = ([dmean, dlog_std] @ W3a) * (h2a > 0)
__global__ void __launch_bounds__(256)
sac_actor_bwd_head_kernel(int B, int H1, int H2, const float *__restrict__ dz1c, int64_t dz_z, const float *__restrict__ W1c, int64_t w_z,
                          const float2 *__restrict__ a_pi, const float2 *__restrict__ std_eps, const float2 *__restrict__ raw, const float *__restrict__ scalars,
                          const float *__restrict__ W3a, const float *__restrict__ h2a, float4 *__restrict__ dpre_out, float *__restrict__ dz2a) {
    pdl_enter();
    const int lane = threadIdx.x & 31, b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    float s0 = 0.f, s1 = 0.f;
    for (int z = 0; z < 2; ++z) {
        const float *d = dz1c + z * dz_z + (int64_t)b * H1, *W = W1c + z * w_z;
        for (int j = lane; j < H1; j += 32) {
            const float v = d[j];
            s0 = fmaf(v, __ldg(W + j * (OBS + ACT) + OBS), s0);
            s1 = fmaf(v, __ldg(W + j * (OBS + ACT) + OBS + 1), s1);
        }
    }
    s0 = warp_sum(s0), s1 = warp_sum(s1);
    const float2 a = a_pi[b], se = std_eps[b], rw = raw[b];
    const float c = scalars[5] / (float)B;
    const float om0 = 1.f - a.x * a.x, om1 = 1.f - a.y * a.y;
    const float du0 = s0 * om0 + c * (2.f * a.x * om0 / (om0 + SAC_SQUASH_EPS)), du1 = s1 * om1 + c * (2.f * a.y * om1 / (om1 + SAC_SQUASH_EPS));
    const float g0 = (rw.x >= SAC_LOG_STD_MIN && rw.x <= SAC_LOG_STD_MAX) ? du0 * se.x - c : 0.f;
    const float g1 = (rw.y >= SAC_LOG_STD_MIN && rw.y <= SAC_LOG_STD_MAX) ? du1 * se.y - c : 0.f;
    if (lane == 0) dpre_out[b] = make_float4(du0, du1, g0, g1);
    const float p[4] = {du0, du1, g0, g1};
    const float *h = h2a + (int64_t)b * H2;
    float *o = dz2a + (int64_t)b * H2;
    for (int k = lane * 4; k < H2; k += 128) {
        const float4 hh = *reinterpret_cast<const float4 *>(h + k);
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int r = 0; r < 4; ++r) {
            const float4 w = *reinterpret_cast<const float4 *>(W3a + (int64_t)r * H2 + k);
            acc.x = fmaf(p[r], w.x, acc.x), acc.y = fmaf(p[r], w.y, acc.y), acc.z = fmaf(p[r], w.z, acc.z), acc.w = fmaf(p[r], w.w, acc.w);
        }
        *reinterpret_cast<float4 *>(o + k) = make_float4(hh.x > 0.f ? acc.x : 0.f, hh.y > 0.f ? acc.y : 0.f, hh.z > 0.f ? acc.z : 0.f, hh.w > 0.f ? acc.w : 0.f);
    }
}

// ------------------------------------------------------------------------------------------------------------------
// SAC with gSDE (use_sde=True: StateDependentNoiseDistribution, learn_features=True, full_std=True, use_expln=False; core/sac/policies.py,
// core/common/distributions.py).  The actor head slot holds [mu.weight (2,H2) | log_std (H2,2)], the bias slot [mu.bias (2) | 0 0].
// One exploration matrix E = exp(log_std) * eps (H2,2) per update (reset_noise() with batch size 1 at the top of sac.py's loop) serves
// every row of actions_pi, next_actions and the actor loss; it is an rsample, so the loss reaches log_std through E as well.
// ------------------------------------------------------------------------------------------------------------------
constexpr uint32_t STREAM_SAC_SDE = 10u;
constexpr float SDE_VAR_EPS = 1e-6f, SDE_ATANH_EPS = 1.1920928955078125e-07f;  // proba_distribution's variance epsilon; finfo(float32).eps

// sde[0 : 2H2] = E, sde[2H2 : 4H2] = std^2, with std = exp(log_std); eps from eps_in (H2,2) or Philox (key seed = the UN-rank-keyed seed,
// counter (k, update index), stream 10): every data-parallel rank draws the same E
__global__ void __launch_bounds__(256)
sac_sde_draw_kernel(int H2, const float *__restrict__ log_std, const float2 *__restrict__ eps_in, uint64_t seed, uint32_t update_index,
                    const float *__restrict__ dev_scalars, float *__restrict__ sde) {
    pdl_enter();
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= H2) return;
    float2 e;
    if (eps_in) e = eps_in[k];
    else {
        const uint32_t ui = dev_scalars ? __float_as_uint(dev_scalars[4]) : update_index;
        const uint4 r = philox_env(seed, (uint64_t)k, ui, STREAM_SAC_SDE, 0);
        const float u1 = fmaf(u24(r.x), 1.0f, 5.9604644775390625e-08f), u2 = u24(r.y);
        const float rad = sqrtf(-2.0f * logf(u1));
        float sn, cs;
        sincospif(2.0f * u2, &sn, &cs);
        e = make_float2(rad * cs, rad * sn);
    }
    const float s0 = expf(log_std[2 * k]), s1 = expf(log_std[2 * k + 1]);
    sde[2 * k] = s0 * e.x, sde[2 * k + 1] = s1 * e.y;
    sde[2 * H2 + 2 * k] = s0 * s0, sde[2 * H2 + 2 * k + 1] = s1 * s1;
}

// log_prob of the gSDE distribution at the squashed action a (distributions.py log_prob: the tanh is INVERTED, g = atanh(clamp(a)))
__device__ __forceinline__ float sde_gauss_arg(float a) {
    const float y = fminf(fmaxf(a, -1.f + SDE_ATANH_EPS), 1.f - SDE_ATANH_EPS);
    return 0.5f * (log1pf(y) - log1pf(-y));
}

// per row: mu_raw = h2 @ Wmu^T + b, mean = hardtanh(mu_raw), var = h2^2 @ std^2, sigma = sqrt(var + 1e-6), noise = h2 @ E,
// a = tanh(mean + noise), log_prob = sum_j Normal(mean_j, sigma_j).log_prob(g_j) - sum_j log(1 - tanh(g_j)^2 + 1e-6)
__global__ void __launch_bounds__(256)
sac_sde_head_kernel(int B, int H2, const float *__restrict__ h2, const float *__restrict__ W3, const float *__restrict__ b3, const float *__restrict__ sde,
                    float clip_mean, float2 *__restrict__ act_out, float *__restrict__ logp_out, float2 *__restrict__ mu_raw_out,
                    float2 *__restrict__ sigma_out, float *__restrict__ lp_partial) {
    pdl_enter();
    __shared__ float sl[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, b = blockIdx.x * 8 + warp;
    float lp = 0.f;
    if (b < B) {
        const float *h = h2 + (int64_t)b * H2;
        const float m0 = row_dot(h, W3, H2, lane) + b3[0], m1 = row_dot(h, W3 + H2, H2, lane) + b3[1];
        const float2 *E = reinterpret_cast<const float2 *>(sde), *S2 = E + H2;
        float n0 = 0.f, n1 = 0.f, v0 = 0.f, v1 = 0.f;
        for (int k = lane; k < H2; k += 32) {
            const float x = h[k], x2 = x * x;
            const float2 e = E[k], s2 = S2[k];
            n0 = fmaf(x, e.x, n0), n1 = fmaf(x, e.y, n1), v0 = fmaf(x2, s2.x, v0), v1 = fmaf(x2, s2.y, v1);
        }
        n0 = warp_sum(n0), n1 = warp_sum(n1), v0 = warp_sum(v0), v1 = warp_sum(v1);
        if (lane == 0) {
            const float mr[2] = {m0, m1}, nz[2] = {n0, n1}, vr[2] = {v0, v1};
            float a[2], sg[2];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const float mean = clip_mean > 0.f ? fminf(fmaxf(mr[i], -clip_mean), clip_mean) : mr[i];
                sg[i] = sqrtf(vr[i] + SDE_VAR_EPS);
                a[i] = tanhf(mean + nz[i]);
                const float g = sde_gauss_arg(a[i]), d = g - mean, t = tanhf(g);
                lp += -(d * d) / (2.f * sg[i] * sg[i]) - logf(sg[i]) - SAC_HALF_LOG_2PI - logf(1.f - t * t + SAC_SQUASH_EPS);
            }
            act_out[b] = make_float2(a[0], a[1]);
            logp_out[b] = lp;
            if (mu_raw_out) mu_raw_out[b] = make_float2(m0, m1);
            if (sigma_out) sigma_out[b] = make_float2(sg[0], sg[1]);
        }
    }
    if (lp_partial) {
        if (lane == 0) sl[warp] = lp;
        __syncthreads();
        if (threadIdx.x == 0) {
            float t = 0.f;
            for (int i = 0; i < 8; ++i) t += sl[i];
            lp_partial[blockIdx.x] = t;
        }
    }
}

// actor-loss backward through the gSDE head, per row (c = ent_coef / B, s = dL/da from the critics):
//   d = g - mean;  dlp/dg = -d/sigma^2 + 2t(1-t^2)/(1-t^2+1e-6) (t = tanh g), 0 where the atanh clamp binds;  du = s (1-a^2) + c dlp/dg
//   dmean = du + c d/sigma^2 -> dmu_raw (0 outside the open Hardtanh interval);  dnoise = du;  dvar = c (d^2/sigma^3 - 1/sigma) / (2 sigma)
//   dlatent = (dmu_raw @ Wmu + dnoise @ E^T + 2 h2 * (dvar @ std2^T)) * (h2 > 0)
// Y rows: y4[b] = [dmu_raw_0, dmu_raw_1, dnoise_0, dnoise_1], y2[b] = [dvar_0, dvar_1] (for sac_sde_wgrad_kernel)
__global__ void __launch_bounds__(256)
sac_sde_bwd_head_kernel(int B, int H1, int H2, const float *__restrict__ dz1c, int64_t dz_z, const float *__restrict__ W1c, int64_t w_z,
                        const float2 *__restrict__ a_pi, const float2 *__restrict__ mu_raw, const float2 *__restrict__ sigma, const float *__restrict__ scalars,
                        const float *__restrict__ W3a, const float *__restrict__ sde, float clip_mean, const float *__restrict__ h2a,
                        float4 *__restrict__ y4, float2 *__restrict__ y2, float *__restrict__ dz2a) {
    pdl_enter();
    const int lane = threadIdx.x & 31, b = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (b >= B) return;
    float s[2] = {0.f, 0.f};
    for (int z = 0; z < 2; ++z) {
        const float *d = dz1c + z * dz_z + (int64_t)b * H1, *W = W1c + z * w_z;
        for (int j = lane; j < H1; j += 32) {
            const float v = d[j];
            s[0] = fmaf(v, __ldg(W + j * (OBS + ACT) + OBS), s[0]);
            s[1] = fmaf(v, __ldg(W + j * (OBS + ACT) + OBS + 1), s[1]);
        }
    }
    s[0] = warp_sum(s[0]), s[1] = warp_sum(s[1]);
    const float2 a2 = a_pi[b], m2 = mu_raw[b], sg2 = sigma[b];
    const float av[2] = {a2.x, a2.y}, mr[2] = {m2.x, m2.y}, sg[2] = {sg2.x, sg2.y};
    const float c = scalars[5] / (float)B;
    float dmu[2], dn[2], dv[2];
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        const bool inside = !(clip_mean > 0.f) || (mr[i] > -clip_mean && mr[i] < clip_mean);
        const float mean = clip_mean > 0.f ? fminf(fmaxf(mr[i], -clip_mean), clip_mean) : mr[i];
        const float g = sde_gauss_arg(av[i]), d = g - mean, t = tanhf(g), omt = 1.f - t * t, is2 = 1.f / (sg[i] * sg[i]);
        const bool clamped = av[i] < -1.f + SDE_ATANH_EPS || av[i] > 1.f - SDE_ATANH_EPS;
        const float dlp_dg = clamped ? 0.f : -d * is2 + 2.f * t * omt / (omt + SAC_SQUASH_EPS);
        const float du = s[i] * (1.f - av[i] * av[i]) + c * dlp_dg;
        dmu[i] = inside ? du + c * d * is2 : 0.f;
        dn[i] = du;
        dv[i] = c * (d * d * is2 / sg[i] - 1.f / sg[i]) / (2.f * sg[i]);
    }
    if (lane == 0) {
        y4[b] = make_float4(dmu[0], dmu[1], dn[0], dn[1]);
        y2[b] = make_float2(dv[0], dv[1]);
    }
    const float *h = h2a + (int64_t)b * H2;
    const float2 *E = reinterpret_cast<const float2 *>(sde), *S2 = E + H2;
    float *o = dz2a + (int64_t)b * H2;
    for (int k = lane; k < H2; k += 32) {
        const float x = h[k];
        const float2 e = E[k], s2 = S2[k];
        float acc = fmaf(dmu[0], W3a[k], dmu[1] * W3a[H2 + k]);
        acc = fmaf(dn[0], e.x, acc), acc = fmaf(dn[1], e.y, acc);
        acc = fmaf(2.f * x, fmaf(dv[0], s2.x, dv[1] * s2.y), acc);
        o[k] = x > 0.f ? acc : 0.f;
    }
}

// head weight gradients over the batch, one CTA per 32 latent units, 8 warps interleaved over rows, fixed-order sums (deterministic):
//   dWmu[j][k] = sum_b y4[b][j] h[b][k];  dlog_std[k][j] = E[k][j] sum_b y4[b][2+j] h[b][k] + 2 std2[k][j] sum_b y2[b][j] h[b][k]^2
//   CTA 0 also writes the bias slot [sum_b dmu_raw_0, sum_b dmu_raw_1, 0, 0]
__global__ void __launch_bounds__(256)
sac_sde_wgrad_kernel(int B, int H2, const float *__restrict__ h2a, const float4 *__restrict__ y4, const float2 *__restrict__ y2, const float *__restrict__ sde,
                     float *__restrict__ gw3, float *__restrict__ gb3) {
    pdl_enter();
    __shared__ float red[8][7][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, k = blockIdx.x * 32 + lane;
    float acc[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // dWmu0, dWmu1, dE0, dE1, dv0, dv1, (bias: dmu sums in lanes 0 / 1)
    float bsum0 = 0.f, bsum1 = 0.f;
    for (int b = warp; b < B; b += 8) {
        const float4 y = y4[b];
        const float2 v = y2[b];
        if (k < H2) {
            const float x = h2a[(int64_t)b * H2 + k], x2 = x * x;
            acc[0] = fmaf(y.x, x, acc[0]), acc[1] = fmaf(y.y, x, acc[1]), acc[2] = fmaf(y.z, x, acc[2]), acc[3] = fmaf(y.w, x, acc[3]);
            acc[4] = fmaf(v.x, x2, acc[4]), acc[5] = fmaf(v.y, x2, acc[5]);
        }
        bsum0 += y.x, bsum1 += y.y;
    }
    acc[6] = lane == 0 ? bsum0 : bsum1;
#pragma unroll
    for (int i = 0; i < 7; ++i) red[warp][i][lane] = acc[i];
    __syncthreads();
    if (warp != 0) return;
    float t[7];
#pragma unroll
    for (int i = 0; i < 7; ++i) {
        t[i] = 0.f;
        for (int w = 0; w < 8; ++w) t[i] += red[w][i][lane];
    }
    if (k < H2) {
        const float2 e = reinterpret_cast<const float2 *>(sde)[k], s2 = reinterpret_cast<const float2 *>(sde)[H2 + k];
        gw3[k] = t[0], gw3[H2 + k] = t[1];
        gw3[2 * H2 + 2 * k] = fmaf(e.x, t[2], 2.f * s2.x * t[4]);
        gw3[2 * H2 + 2 * k + 1] = fmaf(e.y, t[3], 2.f * s2.y * t[5]);
    }
    if (blockIdx.x == 0 && lane < 4) gb3[lane] = lane < 2 ? t[6] : 0.f;
}

// ------------------------------------------------------------------------------------------------------------------
// skinny weight gradients:  out_w[j][i] (or [i][j]) = sum_b X[b][j] * Y[b][i],  out_b = sum_b X[b][j]  (or sum_b Y[b][i])
//   layer 1:  X = dz1 (B,H1), Y = [obs | act]        -> dW1 (H1,in), db1 (H1)
//   layer 2 bias: X = dz2 (B,H2), no Y               -> db2 (H2)
//   layer 3:  X = h2 (B,H2),  Y = dq / dpre (B,out)  -> dW3 (out,H2) [transposed store], db3 = sum_b Y
// One CTA owns 32 columns j and walks the whole batch (fixed order: deterministic), 8 warps interleaved over rows.
// ------------------------------------------------------------------------------------------------------------------
struct SkinnyArgs {
    const float *X;
    int64_t x_z;
    int ldx, H, B;
    const float *Y0;  // (B, n0) shared over z unless y_z != 0
    const float *Y1;  // (B, n1)
    int n0, ld0, n1, ld1;
    int64_t y_z;
    float *part;      // [chunk][z][NY + 1][Hp] partial sums (Hp = H rounded up to 32)
    float *out_w, *out_b;  // out_b: sum_b X (layers 1, 2) or sum_b Y (layer 3)
    int64_t out_z;
    int transposed, chunks, rows_per_chunk;
};
constexpr int SKINNY_ROWS = 64;  // batch rows per CTA

template <int NY, bool YBIAS>
__global__ void __launch_bounds__(256) td3_skinny_wgrad_kernel(SkinnyArgs s) {
    pdl_enter();
    __shared__ float red[8][NY + 1][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, z = blockIdx.z, chunk = blockIdx.y;
    const int j = blockIdx.x * 32 + lane;
    const bool live = j < s.H;
    const float *X = s.X + z * s.x_z + (live ? j : 0);
    const float *Y0 = s.Y0 ? s.Y0 + z * s.y_z : nullptr;
    const int b_lo = chunk * s.rows_per_chunk, b_hi = min(s.B, b_lo + s.rows_per_chunk);
    float acc[NY + 1];
#pragma unroll
    for (int i = 0; i <= NY; ++i) acc[i] = 0.f;
#pragma unroll 4
    for (int b = b_lo + warp; b < b_hi; b += 8) {
        const float x = live ? X[(int64_t)b * s.ldx] : 0.f;
#pragma unroll
        for (int i = 0; i < NY; ++i) {
            const float y = i < s.n0 ? Y0[(int64_t)b * s.ld0 + i] : s.Y1[(int64_t)b * s.ld1 + (i - s.n0)];
            acc[i] = fmaf(x, y, acc[i]);
        }
        if (!YBIAS) acc[NY] += x;  // bias gradient = column sum of X
    }
    if (YBIAS && blockIdx.x == 0 && lane < NY)  // bias gradient = column sum of Y (layer 3): lane i of the first column block
        for (int b = b_lo + warp; b < b_hi; b += 8) acc[NY] += Y0[(int64_t)b * s.ld0 + lane];
#pragma unroll
    for (int i = 0; i <= NY; ++i) red[warp][i][lane] = acc[i];
    __syncthreads();
    const int Hp = gridDim.x * 32;
    float *part = s.part + ((int64_t)chunk * gridDim.z + z) * (NY + 1) * Hp;
    for (int e = threadIdx.x; e < (NY + 1) * 32; e += 256) {
        const int i = e >> 5, l = e & 31;
        float v = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) v += red[w][i][l];
        part[(int64_t)i * Hp + blockIdx.x * 32 + l] = v;
    }
}

// One node instead of four: the second stages of up to three skinny weight gradients and the dW2 slab sum of a backward pass run as
// jobs of ONE launch (blockIdx.z = job).  Fewer graph nodes is what the small-batch update time is made of.
struct FinJob {
    SkinnyArgs s;
    int ny, ybias, hp, Z;
};
struct FinJobs {
    FinJob job[3];
    int n;  // skinny jobs; job index n (if slab_splits > 0) is the slab sum
    int64_t slab_n4, slab_stride4, slab_z4, slab_out_z4;
    int slab_splits, slab_Z;
    const float4 *slabs;
    float4 *slab_out;
};

__global__ void __launch_bounds__(256) td3_finalize_kernel(FinJobs J) {
    pdl_enter();
    const int jb = blockIdx.z, z = blockIdx.y;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (jb == J.n) {  // dW2 = sum of the split-K slabs (fixed order)
        if (z >= J.slab_Z || e >= J.slab_n4) return;
        float4 acc = J.slabs[z * J.slab_z4 + e];
        for (int k = 1; k < J.slab_splits; ++k) {
            const float4 v = J.slabs[k * J.slab_stride4 + z * J.slab_z4 + e];
            acc.x += v.x, acc.y += v.y, acc.z += v.z, acc.w += v.w;
        }
        J.slab_out[z * J.slab_out_z4 + e] = acc;
        return;
    }
    const FinJob &f = J.job[jb];
    const SkinnyArgs &s = f.s;
    const int NY = f.ny, Hp = f.hp;
    if (z >= f.Z || e >= (int64_t)(NY + 1) * Hp) return;
    const int i = (int)(e / Hp), jj = (int)(e % Hp);
    if (i == NY) {
        if (!s.out_b || (f.ybias ? jj >= NY : jj >= s.H)) return;
    } else if (jj >= s.H || !s.out_w) return;
    const int64_t stride = (int64_t)f.Z * (NY + 1) * Hp;
    const float *pp = s.part + (int64_t)z * (NY + 1) * Hp + e;
    float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;  // four loads in flight; the combination order is fixed
    int c = 0;
    for (; c + 4 <= s.chunks; c += 4) {
        a0 += pp[(c + 0) * stride];
        a1 += pp[(c + 1) * stride];
        a2 += pp[(c + 2) * stride];
        a3 += pp[(c + 3) * stride];
    }
    for (; c < s.chunks; ++c) a0 += pp[c * stride];
    const float v = (a0 + a1) + (a2 + a3);
    if (i < NY) {
        if (s.transposed) s.out_w[z * s.out_z + (int64_t)i * s.H + jj] = v;
        else s.out_w[z * s.out_z + (int64_t)jj * NY + i] = v;
    } else {
        s.out_b[z * s.out_z + jj] = v;
    }
}

// graph mode: the per-update scalars (Philox counter of the smoothing noise, Adam bias corrections) cannot be baked into a captured
// launch, so they live on the device.  counters = {n_updates, critic_step, actor_step, sample_draw}; one thread advances them at the
// start of an update and derives scalars = {step_size_c, bc2_sqrt_c, step_size_a, bc2_sqrt_a, bits(n_updates)} (double math as torch).
// lr_c2 / lr_a2 >= 0 (multi-agent: a second critic / actor optimiser with its own rate, which may be 0 as torch's Adam allows): their
// {step_size, bc2_sqrt} pairs go to scalars[8..11]; -1 = no second optimiser.
__global__ void td3_tick_kernel(int64_t *counters, float *scalars, int policy_step, double lr, double beta1, double beta2, double lr_a, double lr_c2,
                                double lr_a2) {
    pdl_enter();
    if (threadIdx.x || blockIdx.x) return;
    const int64_t n = ++counters[0], cs = ++counters[1];
    const int64_t as = policy_step ? ++counters[2] : counters[2];
    counters[3] += 1;
    if (lr_a < 0.0) lr_a = lr;
    scalars[0] = (float)(lr / (1.0 - pow(beta1, (double)cs)));
    scalars[1] = (float)sqrt(1.0 - pow(beta2, (double)cs));
    if (lr_c2 >= 0.0) scalars[8] = (float)(lr_c2 / (1.0 - pow(beta1, (double)cs))), scalars[9] = scalars[1];
    if (as > 0) {
        scalars[2] = (float)(lr_a / (1.0 - pow(beta1, (double)as)));
        scalars[3] = (float)sqrt(1.0 - pow(beta2, (double)as));
        if (lr_a2 >= 0.0) scalars[10] = (float)(lr_a2 / (1.0 - pow(beta1, (double)as))), scalars[11] = scalars[3];
    }
    scalars[4] = __uint_as_float((uint32_t)n);
}

// Adam (torch single-tensor formulas) over a flat range, optionally followed by the polyak update of another flat range;
// block 0 / thread 0 also folds the per-CTA loss partials into the running loss sums.
struct ApplyArgs {
    float *p, *t;
    const float *g;
    float *m, *v;
    int64_t adam_lo, adam_hi;      // Adam on [adam_lo, adam_hi)
    int64_t polyak_lo, polyak_hi;  // polyak on [polyak_lo, polyak_hi) (after Adam where the ranges overlap)
    float beta1, beta2, eps, step_size, bc2_sqrt, tau;
    const float *dev_scalars;  // graph mode: {step_size, bc2_sqrt} written by td3_tick_kernel (NULL: the by-value fields)
    const float *loss_partial;
    int n_loss_partial;
    float loss_scale;
    float *loss_acc;  // [0] += scale * sum(partials), [1] += 1
};

// block 0 of an apply launch: the per-CTA loss partials -> the running loss sums (block-wide tree, fixed order)
__device__ __forceinline__ void fold_loss_partials(const ApplyArgs &a) {
    __shared__ float sl[256];
    float s = 0.f;
    for (int k = threadIdx.x; k < a.n_loss_partial; k += 256) s += a.loss_partial[k];
    sl[threadIdx.x] = s;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) sl[threadIdx.x] += sl[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        a.loss_acc[0] += sl[0] * a.loss_scale;
        a.loss_acc[1] += 1.f;
    }
}

__global__ void __launch_bounds__(256) td3_apply_kernel(ApplyArgs a) {
    pdl_enter();
    const int64_t lo = min(a.adam_lo, a.polyak_lo < a.polyak_hi ? a.polyak_lo : a.adam_lo);
    const int64_t i = lo + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (blockIdx.x == 0 && a.loss_acc) fold_loss_partials(a);
    float p;
    bool have = false;
    const float step_size = a.dev_scalars ? a.dev_scalars[0] : a.step_size, bc2_sqrt = a.dev_scalars ? a.dev_scalars[1] : a.bc2_sqrt;
    if (i >= a.adam_lo && i < a.adam_hi) {
        const float g = a.g[i];
        float m = a.m[i], v = a.v[i];
        m = m + (g - m) * (1.f - a.beta1);           // exp_avg.lerp_(grad, 1 - beta1)
        v = v * a.beta2 + (1.f - a.beta2) * g * g;   // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
        const float denom = sqrtf(v) / bc2_sqrt + a.eps;
        p = a.p[i] - step_size * (m / denom);      // param.addcdiv_(exp_avg, denom, value=-step_size)
        a.p[i] = p, a.m[i] = m, a.v[i] = v;
        have = true;
    }
    if (i >= a.polyak_lo && i < a.polyak_hi) {
        if (!have) p = a.p[i];
        a.t[i] = a.t[i] * (1.f - a.tau) + a.tau * p;  // utils.py:480-481
    }
}


// ------------------------------------------------------------------------------------------------------------------
// data-parallel variant of td3_apply_kernel: the gradient all-reduce is INSIDE the Adam step (include/cstr_b200.h,
// cstr_peer_comm).  Every rank's gradient block is mapped in every process; thread i reads element group i of all `world`
// blocks over NVLink, adds them in rank order (the same order on every rank: bit-identical weights without a broadcast),
// scales by 1/world and continues with exactly the arithmetic of td3_apply_kernel.
// Barrier block of one rank (uint32): [phase 0|1][PEER_MAX_BLOCKS][8 ranks] flags, then {epoch, done-ticket, error, pad}.
// CTA b of rank r: writes `epoch` into slot [phase][b][r] of EVERY rank's block, then spins on its own slots [phase][b][*].
// phase 0 (before the reads): the peer's CTA b has started, hence its stream reached this kernel, hence its backward pass is complete
// and visible (kernel boundary + the release/acquire pair).  phase 1 (after the reads): every peer's CTA b has finished reading
// region b of my block, so the kernels after this one may overwrite it.  The grid never exceeds the resident-CTA capacity, so every
// CTA of every rank is running and the waits cannot deadlock; a dead peer is a bounded wait (error word), not a hang.
// ------------------------------------------------------------------------------------------------------------------
constexpr int PEER_MAX_BLOCKS = 592;  // 148 SMs x 4 CTAs of 256 threads: always co-resident
constexpr int PEER_FLAG_WORDS = 2 * PEER_MAX_BLOCKS * CSTR_PEER_MAX_WORLD;
constexpr int PEER_EPOCH = PEER_FLAG_WORDS, PEER_TICKET = PEER_FLAG_WORDS + 1, PEER_ERROR = PEER_FLAG_WORDS + 2;
constexpr long long PEER_WAIT_CYCLES = 8000000000LL;  // ~4 s at 2 GHz

struct PeerArgs {
    int world, rank;
    const float *g[CSTR_PEER_MAX_WORLD];
    uint32_t *flags[CSTR_PEER_MAX_WORLD];
    float scale;  // 1 / world
};

__device__ __forceinline__ void st_release_sys(uint32_t *p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ float4 ld_peer_f4(const float *p) {  // peer memory written by another GPU: never from this SM's L1
    float4 v;
    asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
    return v;
}

// returns false when a peer never arrived (error word raised)
__device__ __forceinline__ bool peer_barrier(const PeerArgs &pa, int phase, uint32_t epoch) {
    __shared__ int ok_s;
    __syncthreads();
    if (threadIdx.x == 0) ok_s = 1;
    __syncthreads();
    if ((int)threadIdx.x < pa.world) {
        const int slot = (phase * PEER_MAX_BLOCKS + blockIdx.x) * CSTR_PEER_MAX_WORLD;
        st_release_sys(pa.flags[threadIdx.x] + slot + pa.rank, epoch);
        const uint32_t *mine = pa.flags[pa.rank] + slot + threadIdx.x;
        const long long t0 = clock64();
        while ((int32_t)(ld_acquire_sys(mine) - epoch) < 0) {
            if (clock64() - t0 > PEER_WAIT_CYCLES) {
                pa.flags[pa.rank][PEER_ERROR] = 1u + (uint32_t)threadIdx.x;
                ok_s = 0;
                break;
            }
        }
    }
    __syncthreads();
    return ok_s != 0;
}

__global__ void __launch_bounds__(256) td3_apply_peer_kernel(ApplyArgs a, PeerArgs pa) {
    pdl_enter();
    uint32_t *my = pa.flags[pa.rank];
    const uint32_t epoch = *(volatile uint32_t *)(my + PEER_EPOCH) + 1u;
    // once a wait has timed out (a peer died or fell out of step) every later launch skips waiting and updating: the cost of a broken
    // group is ONE bounded wait, after which the host finds the error word (cstr_peer_error) instead of a hung stream
    const bool broken = *(volatile uint32_t *)(my + PEER_ERROR) != 0u;
    const bool alive = !broken && peer_barrier(pa, 0, epoch);
    if (blockIdx.x == 0 && a.loss_acc) fold_loss_partials(a);  // the LOCAL shard's loss
    const float step_size = a.dev_scalars ? a.dev_scalars[0] : a.step_size, bc2_sqrt = a.dev_scalars ? a.dev_scalars[1] : a.bc2_sqrt;
    const int64_t lo = min(a.adam_lo, a.polyak_lo < a.polyak_hi ? a.polyak_lo : a.adam_lo), hi = max(a.adam_hi, a.polyak_hi);
    if (alive)  // every range boundary is a multiple of 4 floats (pad4 layout): one float4 group per thread and trip
        for (int64_t i = lo + 4 * ((int64_t)blockIdx.x * blockDim.x + threadIdx.x); i < hi; i += 4 * (int64_t)gridDim.x * blockDim.x) {
            float p[4];
            bool have = false;
            if (i >= a.adam_lo && i < a.adam_hi) {
                float4 g4 = ld_peer_f4(pa.g[0] + i);
                for (int r = 1; r < pa.world; ++r) {
                    const float4 u = ld_peer_f4(pa.g[r] + i);
                    g4.x += u.x, g4.y += u.y, g4.z += u.z, g4.w += u.w;
                }
                const float g[4] = {g4.x * pa.scale, g4.y * pa.scale, g4.z * pa.scale, g4.w * pa.scale};
                const float4 p4 = *reinterpret_cast<const float4 *>(a.p + i), m4 = *reinterpret_cast<const float4 *>(a.m + i),
                             v4 = *reinterpret_cast<const float4 *>(a.v + i);
                float m[4] = {m4.x, m4.y, m4.z, m4.w}, v[4] = {v4.x, v4.y, v4.z, v4.w};
                p[0] = p4.x, p[1] = p4.y, p[2] = p4.z, p[3] = p4.w;
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    m[c] = m[c] + (g[c] - m[c]) * (1.f - a.beta1);
                    v[c] = v[c] * a.beta2 + (1.f - a.beta2) * g[c] * g[c];
                    const float denom = sqrtf(v[c]) / bc2_sqrt + a.eps;
                    p[c] = p[c] - step_size * (m[c] / denom);
                }
                *reinterpret_cast<float4 *>(a.p + i) = make_float4(p[0], p[1], p[2], p[3]);
                *reinterpret_cast<float4 *>(a.m + i) = make_float4(m[0], m[1], m[2], m[3]);
                *reinterpret_cast<float4 *>(a.v + i) = make_float4(v[0], v[1], v[2], v[3]);
                have = true;
            }
            if (i >= a.polyak_lo && i < a.polyak_hi) {
                if (!have) {
                    const float4 p4 = *reinterpret_cast<const float4 *>(a.p + i);
                    p[0] = p4.x, p[1] = p4.y, p[2] = p4.z, p[3] = p4.w;
                }
                float4 t = *reinterpret_cast<const float4 *>(a.t + i);
                t.x = t.x * (1.f - a.tau) + a.tau * p[0], t.y = t.y * (1.f - a.tau) + a.tau * p[1];
                t.z = t.z * (1.f - a.tau) + a.tau * p[2], t.w = t.w * (1.f - a.tau) + a.tau * p[3];
                *reinterpret_cast<float4 *>(a.t + i) = t;
            }
        }
    if (alive) peer_barrier(pa, 1, epoch);
    __syncthreads();
    if (threadIdx.x == 0) {  // the last CTA to get here publishes the epoch for the next launch (every CTA has read it by now)
        __threadfence();
        if (atomicAdd(my + PEER_TICKET, 1u) == gridDim.x - 1) {
            my[PEER_TICKET] = 0u;
            *(volatile uint32_t *)(my + PEER_EPOCH) = epoch;
        }
    }
}

}  // namespace cstr

#include "cstr_mlp.cuh"
#include "cstr_bcq_kernels.cuh"

using namespace cstr;

// ------------------------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------------------------
namespace {

constexpr int MAX_SPLITS = 16;

// split-K factor of the dW2 GEMM: minimise (CTA rounds per SM) x (k-iterations per CTA) over the 148 SMs
int choose_splits(int B, int H1, int H2, int Z, int tc) {
    const int64_t tiles = tc ? (int64_t)((H2 + TC_BM - 1) / TC_BM) * tc_tile(H1).n_tiles * Z : (int64_t)((H2 + BM - 1) / BM) * ((H1 + BN - 1) / BN) * Z;
    const int sms = sm_count();
    int best = 1;
    int64_t best_cost = INT64_MAX;
    for (int s = 1; s <= MAX_SPLITS && s * 32 <= B + 31; ++s) {
        const int64_t rounds = (tiles * s + sms - 1) / sms, iters = ((B + s - 1) / s + BK - 1) / BK;
        const int64_t cost = rounds * iters + 2 * s;  // + the slab-sum traffic
        if (cost < best_cost) best_cost = cost, best = s;
    }
    return best;
}

int check_cfg(const cstr_td3_config *c) {
    if (!c) return fail_arg(CSTR_EINVAL, "td3: null config");
    if (c->h1 < 4 || c->h2 < 4 || (c->h1 & 3) || (c->h2 & 3) || c->h1 > 4096 || c->h2 > 4096)
        return fail_arg(CSTR_EINVAL, "td3: hidden sizes must be multiples of 4 in [4, 4096]");
    if (c->batch < 1 || c->batch > (1 << 22)) return fail_arg(CSTR_EINVAL, "td3: batch must be in [1, 4194304]");
    if (c->policy_delay < 1) return fail_arg(CSTR_EINVAL, "td3: policy_delay must be >= 1");
    if (c->n_critics < 0 || c->n_critics > 2) return fail_arg(CSTR_EINVAL, "td3: n_critics must be 1 or 2 (0 = 2)");
    if (c->gemm_mode < CSTR_TD3_GEMM_FP32 || c->gemm_mode > CSTR_TD3_GEMM_BF16) return fail_arg(CSTR_EINVAL, "td3: gemm_mode must be 0 (fp32 FFMA), 1 (bf16x3 tensor) or 2 (bf16 tensor)");
    return 0;
}

template <int NY, bool YBIAS>
int launch_skinny(SkinnyArgs s, int Z, float *part, cudaStream_t st, const char *what, FinJobs &J) {
    s.part = part;
    s.rows_per_chunk = SKINNY_ROWS;
    s.chunks = (s.B + SKINNY_ROWS - 1) / SKINNY_ROWS;
    const int cols = (s.H + 31) / 32;
    launch_k(td3_skinny_wgrad_kernel<NY, YBIAS>, dim3(cols, s.chunks, Z), 256, 0, st, s);
    if (int rc = check_launch(what)) return rc;
    FinJob &f = J.job[J.n++];  // the second stage runs as a job of the backward pass's finalize launch
    f.s = s, f.ny = NY, f.ybias = YBIAS ? 1 : 0, f.hp = cols * 32, f.Z = Z;
    return 0;
}

int launch_finalize(const FinJobs &J, cudaStream_t st) {
    int64_t elems = J.slab_splits > 0 ? J.slab_n4 : 0;
    int Z = J.slab_splits > 0 ? J.slab_Z : 1;
    for (int k = 0; k < J.n; ++k) {
        const int64_t e = (int64_t)(J.job[k].ny + 1) * J.job[k].hp;
        if (e > elems) elems = e;
        if (J.job[k].Z > Z) Z = J.job[k].Z;
    }
    const int jobs = J.n + (J.slab_splits > 0 ? 1 : 0);
    if (jobs == 0) return 0;
    launch_k(td3_finalize_kernel, dim3((unsigned)((elems + 255) / 256), Z, jobs), 256, 0, st, J);
    return check_launch("td3_finalize_kernel");
}

template <int MODE>
int launch_gemm(const GemmArgs &g, int Z, int tensor, cudaStream_t st, const char *what) {  // tensor: 0 FFMA, 1 bf16x3 split, 2 plain bf16
    if (tensor) {
        const TcTile t = tc_tile(g.N);
        static bool attr_set[3] = {false, false, false};
        if (!attr_set[MODE]) {
            if (int rc = check_cuda(cudaFuncSetAttribute(td3_gemm_tc_kernel<MODE, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024), "td3_gemm_tc smem attr"))
                return rc;
            if (int rc = check_cuda(cudaFuncSetAttribute(td3_gemm_tc_kernel<MODE, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024), "td3_gemm_tc smem attr"))
                return rc;
            attr_set[MODE] = true;
        }
        dim3 grid(t.n_tiles, (g.M + TC_BM - 1) / TC_BM, Z * g.splits);
        if (tensor == CSTR_TD3_GEMM_BF16) launch_k(td3_gemm_tc_kernel<MODE, 1>, grid, TC_GEMM_THREADS, t.smem_bytes, st, g, t.n_tile, t.tmem_cols);
        else launch_k(td3_gemm_tc_kernel<MODE, 3>, grid, TC_GEMM_THREADS, t.smem_bytes, st, g, t.n_tile, t.tmem_cols);
        return check_launch(what);
    }
    if constexpr (MODE != G_WGRAD) if (g.split_buf) {  // small batch: too few tiles for 148 SMs and a 25-iteration serial K loop -> split K
        const int64_t tiles = (int64_t)((g.N + BN - 1) / BN) * ((g.M + BM - 1) / BM) * Z, sms = sm_count();
        int s = (int)(2 * sms / tiles);  // two CTAs are resident per SM
        const int64_t per = (int64_t)Z * g.M * g.N;
        if (s > 8) s = 8;
        if (s > g.K / (2 * BK)) s = g.K / (2 * BK);
        if (per > 0 && s > g.split_cap / per) s = (int)(g.split_cap / per);
        if (s >= 2) {
            const int kps = (((g.K + s - 1) / s) + BK - 1) / BK * BK;
            s = (g.K + kps - 1) / kps;
            GemmArgs q = g;
            q.raw_partials = 1, q.splits = s, q.k_per_split = kps, q.C = g.split_buf, q.c_z = (int64_t)g.M * g.N, q.c_split = per, q.ldc = g.N;
            dim3 grid((g.N + BN - 1) / BN, (g.M + BM - 1) / BM, Z * s);
            launch_k(td3_gemm_kernel<MODE, true>, grid, 256, 0, st, q);
            if (int rc = check_launch(what)) return rc;
            const int64_t n = (int64_t)g.M * (g.N / 4);
            launch_k(td3_splitk_finish_kernel<MODE>, dim3((unsigned)((n + 255) / 256), Z), 256, 0, st, g, g.split_buf, s, per, g.C);
            return check_launch("td3_splitk_finish_kernel");
        }
    }
    dim3 grid((g.N + BN - 1) / BN, (g.M + BM - 1) / BM, Z * g.splits);
    launch_k(td3_gemm_kernel<MODE>, grid, 256, 0, st, g);
    return check_launch(what);
}

// Adam (+ polyak) over flat ranges; with a peer communicator the gradient is averaged over the ranks inside the kernel
int launch_apply(const ApplyArgs &a, const cstr_peer_comm *peer, const float *local_grads, cudaStream_t st, const char *what) {
    const int64_t lo = std::min(a.adam_lo, a.polyak_lo < a.polyak_hi ? a.polyak_lo : a.adam_lo), hi = std::max(a.adam_hi, a.polyak_hi);
    if (!peer) {
        launch_k(td3_apply_kernel, (unsigned)((hi - lo + 255) / 256), 256, 0, st, a);
        return check_launch(what);
    }
    if (peer->world < 1 || peer->world > CSTR_PEER_MAX_WORLD || peer->rank < 0 || peer->rank >= peer->world)
        return fail_arg(CSTR_EINVAL, "peer comm: world must be in [1, 8] and rank in [0, world)");
    if (peer->grads[peer->rank] != local_grads) return fail_arg(CSTR_EINVAL, "peer comm: state.grads must be peer->grads[rank]");
    if ((lo | hi | a.adam_lo | a.adam_hi | a.polyak_lo | a.polyak_hi) & 3) return fail_arg(CSTR_EINVAL, "peer apply: ranges must be multiples of 4 floats");
    PeerArgs pa{};
    pa.world = peer->world, pa.rank = peer->rank, pa.scale = 1.f / (float)peer->world;
    for (int r = 0; r < peer->world; ++r) {
        if (!peer->grads[r] || !peer->flags[r] || !aligned(peer->grads[r], 16)) return fail_arg(CSTR_EINVAL, "peer comm: null or misaligned peer pointer");
        pa.g[r] = peer->grads[r], pa.flags[r] = peer->flags[r];
    }
    int64_t blocks = ((hi - lo) / 4 + 255) / 256;
    if (blocks > PEER_MAX_BLOCKS) blocks = PEER_MAX_BLOCKS;
    if (blocks < 1) blocks = 1;
    launch_k(td3_apply_peer_kernel, (unsigned)blocks, 256, 0, st, a, pa);
    return check_launch(what);
}

struct Net {  // pointers of one net (or the first of a z-batched pair) inside a flat block
    float *w1, *b1, *w2, *b2, *w3, *b3;
};
Net net_at(float *base, int64_t off, const NetLayout &L) { return Net{base + off + L.w1, base + off + L.b1, base + off + L.w2, base + off + L.b2, base + off + L.w3, base + off + L.b3}; }

inline Src td3_src(const float *obs, const float *act, int in) {  // [obs (4) | act (in - 4)]
    Src s{};
    s.x0 = obs, s.n0 = OBS, s.ld0 = OBS, s.x0_rows = 0, s.x1 = in > OBS ? act : nullptr, s.n1 = in - OBS, s.ld1 = ACT;
    return s;
}

#include "cstr_mlp_host.cuh"

struct Workspace {  // carved out of the caller's workspace buffer (floats)
    float *h1[2], *h2[2];    // forward activations, [z] slabs contiguous: h1[0] + B*H1 == h1[1]
    float *dz1, *dz2;        // 2 slabs each
    float *t_h1, *t_h2;      // target-critic activations (2 slabs)
    float *a_h1, *a_h2;      // actor / actor-target activations
    float *next_act, *a_pi, *target, *dq, *dpre, *loss_partial, *scalars;
    float *logp, *next_logp, *std_eps, *raw_log_std, *dpre4, *lp_partial;  // SAC
    float *sde;                                                            // SAC gSDE: E (H2,2), std^2 (H2,2)
    MlpScratch sc;
    int n_row_blocks;
    int64_t floats;
};

Workspace carve(float *base, int B, int H1, int H2, bool sde = false) {
    Workspace w;
    Bump b(base);
    const int64_t bh1 = (int64_t)B * H1, bh2 = (int64_t)B * H2;
    w.h1[0] = b.take(2 * bh1), w.h1[1] = w.h1[0] ? w.h1[0] + bh1 : nullptr;
    w.h2[0] = b.take(2 * bh2), w.h2[1] = w.h2[0] ? w.h2[0] + bh2 : nullptr;
    w.dz1 = b.take(2 * bh1), w.dz2 = b.take(2 * bh2);
    w.t_h1 = b.take(2 * bh1), w.t_h2 = b.take(2 * bh2);
    w.a_h1 = b.take(bh1), w.a_h2 = b.take(bh2);
    w.next_act = b.take(2 * (int64_t)B), w.a_pi = b.take(2 * (int64_t)B), w.target = b.take(B), w.dq = b.take(2 * (int64_t)B), w.dpre = b.take(2 * (int64_t)B);
    w.n_row_blocks = (B + 7) / 8;
    w.loss_partial = b.take(2 * (int64_t)w.n_row_blocks);
    w.sc.slab_cap = (int64_t)MAX_SPLITS * 2 * pad4((int64_t)H1 * H2);  // the dW2 slabs of two H2 x H1 critics
    w.sc.slabs = b.take(w.sc.slab_cap);
    const int64_t hp = ((int64_t)(H1 > H2 ? H1 : H2) + 31) / 32 * 32;
    w.sc.skinny_region = (int64_t)((B + SKINNY_ROWS - 1) / SKINNY_ROWS) * 2 * (OBS + ACT + 1) * hp;
    w.sc.skinny = b.take(3 * w.sc.skinny_region);
    w.sc.tensor = 0;
    w.scalars = b.take(8);
    w.logp = b.take(B), w.next_logp = b.take(B), w.std_eps = b.take(2 * (int64_t)B), w.raw_log_std = b.take(2 * (int64_t)B), w.dpre4 = b.take(4 * (int64_t)B);
    w.lp_partial = b.take(w.n_row_blocks);
    w.sde = sde ? b.take(4 * (int64_t)H2) : nullptr;  // last, so that the other configurations keep their workspace size
    w.floats = b.o;
    return w;
}

}  // namespace

extern "C" {

int64_t cstr_td3_param_count(int32_t h1, int32_t h2) {
    if (h1 < 4 || h2 < 4 || (h1 & 3) || (h2 & 3)) return -1;
    return td3_layout(h1, h2).total;
}

int cstr_td3_layout(int32_t h1, int32_t h2, int64_t *offsets) {
    if (!offsets || h1 < 4 || h2 < 4 || (h1 & 3) || (h2 & 3)) return fail_arg(CSTR_EINVAL, "td3_layout: bad sizes or null output");
    const Td3Layout T = td3_layout(h1, h2);
    put_offsets(offsets, 0, T.actor_off, T.actor);
    for (int n = 1; n < 3; ++n) put_offsets(offsets, n, T.critic_off[n - 1], T.critic);
    offsets[18] = T.total;
    return 0;
}

int64_t cstr_td3_workspace_bytes(const cstr_td3_config *cfg) {
    if (check_cfg(cfg)) return -1;
    return carve(nullptr, cfg->batch, cfg->h1, cfg->h2).floats * (int64_t)sizeof(float);
}

int cstr_td3_update(const cstr_td3_config *cfg, const cstr_td3_state *stt, const float *obs, const float *actions, const float *next_obs,
                    const float *dones, const float *rewards, const float *noise, int64_t n_updates, int64_t critic_step, int64_t actor_step,
                    int32_t phases, void *stream) {
    if (int rc = check_cfg(cfg)) return rc;
    if (int rc = check_update("td3", stt, cstr_td3_workspace_bytes(cfg), obs, actions, next_obs, dones, rewards, n_updates, critic_step, actor_step)) return rc;
    if (noise && !aligned(noise, 8)) return fail_arg(CSTR_EALIGN, "td3_update: noise needs 8 B alignment");
    const int B = cfg->batch, H1 = cfg->h1, H2 = cfg->h2;
    Workspace w = carve(stt->workspace, B, H1, H2);
    w.sc.tensor = cfg->gemm_mode;
    const Td3Layout T = td3_layout(H1, H2);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t cz = T.critic.size;
    const Net actor = net_at(stt->params, T.actor_off, T.actor), actor_t = net_at(stt->targets, T.actor_off, T.actor);
    const Net critic = net_at(stt->params, T.critic_off[0], T.critic), critic_t = net_at(stt->targets, T.critic_off[0], T.critic);
    const Net g_actor = net_at(stt->grads, T.actor_off, T.actor), g_critic = net_at(stt->grads, T.critic_off[0], T.critic);
    const int rb = w.n_row_blocks;
    const bool policy_step = (n_updates % cfg->policy_delay) == 0;
    const int ZC = cfg->n_critics == 1 ? 1 : 2;  // DDPG = TD3 with one critic (core/ddpg/ddpg.py:100-109); its block 1 stays unused
    const float *dev_sc = stt->counters ? w.scalars : nullptr;  // graph mode (see td3_tick_kernel)
    if (stt->counters && (phases & CSTR_TD3_CRITIC_GRAD))
        if (int rc = launch_tick(stt, w.scalars, policy_step, cfg->lr, cfg->beta1, cfg->beta2, -1.0, -1.0, -1.0, st)) return rc;

    if (phases & CSTR_TD3_CRITIC_GRAD) {
        // ---- target (td3.py:166-175) ----
        if (int rc = forward_hidden(B, H1, H2, OBS, next_obs, nullptr, actor_t, 0, 1, w.a_h1, w.a_h2, w.sc, st)) return rc;
        launch_k(td3_actor_head_kernel, rb, 256, 0, st, B, H2, w.a_h2, actor_t.w3, actor_t.b3, 1, (const float2 *)noise, cfg->target_policy_noise,
                                                 cfg->target_noise_clip, cfg->seed, (uint32_t)n_updates, dev_sc, (float2 *)w.next_act);
        if (int rc = check_launch("td3_actor_head_kernel")) return rc;
        if (int rc = forward_hidden(B, H1, H2, OBS + ACT, next_obs, w.next_act, critic_t, cz, ZC, w.t_h1, w.t_h2, w.sc, st)) return rc;
        launch_k(td3_target_head_kernel, rb, 256, 0, st, B, H2, w.t_h2, (int64_t)B * H2, critic_t.w3, critic_t.b3, cz, rewards, dones, cfg->gamma, ZC, w.target);
        if (int rc = check_launch("td3_target_head_kernel")) return rc;
        // ---- current Q, loss, backward (td3.py:178-186) ----
        if (int rc = forward_hidden(B, H1, H2, OBS + ACT, obs, actions, critic, cz, ZC, w.h1[0], w.h2[0], w.sc, st)) return rc;
        if (int rc = critic_loss_backward(B, H1, H2, td3_src(obs, actions, OBS + ACT), critic, g_critic, cz, ZC, w.h1[0], w.h2[0], w.target, 2.f / (float)B, w.dq,
                                          w.dz2, w.dz1, w.loss_partial, w.sc, st))
            return rc;
    }
    if (phases & CSTR_TD3_CRITIC_APPLY) {
        ApplyArgs a = adam_args(stt, cfg->lr, cfg->beta1, cfg->beta2, cfg->eps, cfg->tau, critic_step, dev_sc, 0);
        a.adam_lo = T.critic_off[0], a.adam_hi = T.critic_off[0] + ZC * cz, a.polyak_lo = a.polyak_hi = 0;
        a.loss_partial = w.loss_partial, a.n_loss_partial = ZC * rb, a.loss_scale = 1.f / (float)B, a.loss_acc = stt->losses;
        if (int rc = launch_apply(a, stt->peer, stt->grads, st, "td3_apply_kernel<critic>")) return rc;
    }
    if (policy_step && (phases & CSTR_TD3_ACTOR_GRAD)) {
        // ---- actor loss = -Q1(s, pi(s)).mean() and its backward (td3.py:189-196) ----
        if (int rc = forward_hidden(B, H1, H2, OBS, obs, nullptr, actor, 0, 1, w.a_h1, w.a_h2, w.sc, st)) return rc;
        launch_k(td3_actor_head_kernel, rb, 256, 0, st, B, H2, w.a_h2, actor.w3, actor.b3, 0, nullptr, 0.f, 0.f, 0, 0, nullptr, (float2 *)w.a_pi);
        if (int rc = check_launch("td3_actor_head_kernel<pi>")) return rc;
        if (int rc = forward_hidden(B, H1, H2, OBS + ACT, obs, w.a_pi, critic, cz, 1, w.h1[0], w.h2[0], w.sc, st)) return rc;
        if (int rc = policy_critic_backward(B, H1, H2, critic, cz, w.h1[0], w.h2[0], w.dq, w.dz2, w.dz1, w.loss_partial, w.sc, st)) return rc;
        // through the critic's input layer and the tanh into the actor; dz2 of the actor reuses slab 1 of the dz2 buffer
        float *dz2a = w.dz2 + (int64_t)B * H2, *dz1a = w.dz1 + (int64_t)B * H1;
        launch_k(td3_actor_bwd_head_kernel, rb, 256, 0, st, B, H1, H2, w.dz1, critic.w1, (const float2 *)w.a_pi, actor.w3, w.a_h2, (float2 *)w.dpre, dz2a);
        if (int rc = check_launch("td3_actor_bwd_head_kernel")) return rc;
        SkinnyArgs s{};  // dW3a = dpre^T @ h2a, db3a = sum dpre
        s.X = w.a_h2, s.x_z = 0, s.ldx = H2, s.H = H2, s.B = B;
        s.Y0 = w.dpre, s.n0 = ACT, s.ld0 = ACT, s.Y1 = nullptr, s.n1 = 0, s.ld1 = 0, s.y_z = 0;
        s.out_w = g_actor.w3, s.out_b = g_actor.b3, s.out_z = 0, s.transposed = 1;
        FinJobs J{};
        if (int rc = launch_skinny<ACT, true>(s, 1, w.sc.skinny + 2 * w.sc.skinny_region, st, "td3_skinny_wgrad_kernel<actor w3>", J)) return rc;
        if (int rc = backward_hidden(B, H1, H2, td3_src(obs, nullptr, OBS), nullptr, actor, g_actor, 0, 1, w.a_h1, dz2a, dz1a, w.sc, J, st)) return rc;
    }
    if (policy_step && (phases & CSTR_TD3_ACTOR_APPLY)) {
        if (actor_step < 1) return fail_arg(CSTR_EINVAL, "td3_update: actor_step must be >= 1 on a policy step");
        ApplyArgs a = adam_args(stt, cfg->lr, cfg->beta1, cfg->beta2, cfg->eps, cfg->tau, actor_step, dev_sc, 2);
        a.adam_lo = T.actor_off, a.adam_hi = T.actor_off + T.actor.size, a.polyak_lo = 0, a.polyak_hi = T.total;
        a.loss_partial = w.loss_partial, a.n_loss_partial = rb, a.loss_scale = -1.f / (float)B, a.loss_acc = stt->losses ? stt->losses + 2 : nullptr;
        if (int rc = launch_apply(a, stt->peer, stt->grads, st, "td3_apply_kernel<actor+polyak>")) return rc;
    }
    return 0;
}


// ---- SAC (core/sac/sac.py:199-296) --------------------------------------------------------------------------------
static int check_sac_cfg(const cstr_sac_config *c) {
    if (!c) return fail_arg(CSTR_EINVAL, "sac: null config");
    if (c->h1 < 4 || c->h2 < 4 || (c->h1 & 3) || (c->h2 & 3) || c->h1 > 4096 || c->h2 > 4096)
        return fail_arg(CSTR_EINVAL, "sac: hidden sizes must be multiples of 4 in [4, 4096]");
    if (c->batch < 1 || c->batch > (1 << 22)) return fail_arg(CSTR_EINVAL, "sac: batch must be in [1, 4194304]");
    if (c->target_update_interval < 1) return fail_arg(CSTR_EINVAL, "sac: target_update_interval must be >= 1");
    if (c->local_step < 0) return fail_arg(CSTR_EINVAL, "sac: local_step must be >= 0 (0 = use the global update counter)");
    if (c->gemm_mode < CSTR_TD3_GEMM_FP32 || c->gemm_mode > CSTR_TD3_GEMM_BF16) return fail_arg(CSTR_EINVAL, "sac: gemm_mode must be 0, 1 or 2");
    if (c->sde != 0 && c->sde != 1) return fail_arg(CSTR_EINVAL, "sac: sde must be 0 or 1");
    if (!(c->clip_mean == c->clip_mean)) return fail_arg(CSTR_EINVAL, "sac: clip_mean is NaN");
    return 0;
}

int64_t cstr_sac_param_count(int32_t h1, int32_t h2) {
    if (h1 < 4 || h2 < 4 || (h1 & 3) || (h2 & 3)) return -1;
    return td3_layout(h1, h2, 2 * ACT).total + 4;  // + the entropy-coefficient slot (log_ent_coef, padded to 4 floats)
}

int cstr_sac_layout(int32_t h1, int32_t h2, int64_t *offsets) {
    if (!offsets || h1 < 4 || h2 < 4 || (h1 & 3) || (h2 & 3)) return fail_arg(CSTR_EINVAL, "sac_layout: bad sizes or null output");
    const Td3Layout T = td3_layout(h1, h2, 2 * ACT);
    put_offsets(offsets, 0, T.actor_off, T.actor);
    for (int n = 1; n < 3; ++n) put_offsets(offsets, n, T.critic_off[n - 1], T.critic);
    offsets[18] = T.total;      // log_ent_coef
    offsets[19] = T.total + 4;  // block size
    return 0;
}

int64_t cstr_sac_workspace_bytes(const cstr_sac_config *cfg) {
    if (check_sac_cfg(cfg)) return -1;
    return carve(nullptr, cfg->batch, cfg->h1, cfg->h2, cfg->sde != 0).floats * (int64_t)sizeof(float);
}

int cstr_sac_update(const cstr_sac_config *cfg, const cstr_td3_state *stt, const float *obs, const float *actions, const float *next_obs,
                    const float *dones, const float *rewards, const float *eps_pi, const float *eps_next, int64_t n_updates, int64_t adam_step,
                    int32_t phases, void *stream) {
    if (int rc = check_sac_cfg(cfg)) return rc;
    if (!(phases & CSTR_TD3_ALL) || (phases & ~CSTR_TD3_ALL)) return fail_arg(CSTR_EINVAL, "sac_update: phases must be a non-empty subset of CSTR_TD3_ALL");
    if (int rc = check_update("sac", stt, cstr_sac_workspace_bytes(cfg), obs, actions, next_obs, dones, rewards, n_updates, adam_step, 0)) return rc;
    if ((eps_pi && !aligned(eps_pi, 8)) || (eps_next && !aligned(eps_next, 8))) return fail_arg(CSTR_EALIGN, "sac_update: eps_pi / eps_next need 8 B alignment");
    if (cfg->sde && eps_next) return fail_arg(CSTR_EINVAL, "sac_update: in gSDE mode eps_pi carries the (h2,2) exploration eps and eps_next must be NULL");
    const bool sde = cfg->sde != 0;
    const int B = cfg->batch, H1 = cfg->h1, H2 = cfg->h2;
    Workspace w = carve(stt->workspace, B, H1, H2, cfg->sde != 0);
    w.sc.tensor = cfg->gemm_mode;
    const Td3Layout T = td3_layout(H1, H2, 2 * ACT);
    cudaStream_t st = (cudaStream_t)stream;
    const int64_t cz = T.critic.size, ent = T.total;
    const Net actor = net_at(stt->params, T.actor_off, T.actor), critic = net_at(stt->params, T.critic_off[0], T.critic);
    const Net critic_t = net_at(stt->targets, T.critic_off[0], T.critic);
    const Net g_actor = net_at(stt->grads, T.actor_off, T.actor), g_critic = net_at(stt->grads, T.critic_off[0], T.critic);
    const int rb = w.n_row_blocks;

    const float *dev_sc = stt->counters ? w.scalars : nullptr;  // graph mode: per-update scalars live on the device (td3_tick_kernel)
    const ApplyArgs adam = adam_args(stt, cfg->lr, cfg->beta1, cfg->beta2, cfg->eps, cfg->tau, adam_step, dev_sc, 0);  // one step for all three optimisers
    // log_ent_coef: gradient and Adam step in one launch when nothing sits between them; gradient only when the caller all-reduces
    // between the phases, or when a peer communicator averages it inside the critic apply (its slot joins that Adam range)
    const bool fused_ent = !stt->peer && (phases & (CSTR_TD3_CRITIC_GRAD | CSTR_TD3_CRITIC_APPLY)) == (CSTR_TD3_CRITIC_GRAD | CSTR_TD3_CRITIC_APPLY);
    auto ent_coef = [&](int mode) {
        launch_k(sac_ent_coef_kernel, 1, 256, 0, st, B, rb, w.lp_partial, cfg->target_entropy, stt->params + ent, stt->grads + ent, stt->adam_m + ent,
                                              stt->adam_v + ent, cfg->beta1, cfg->beta2, cfg->eps, adam.step_size, adam.bc2_sqrt, dev_sc ? 1 : 0, w.scalars,
                                              stt->losses, mode);
        return check_launch("sac_ent_coef_kernel");
    };
    if (stt->counters && (phases & CSTR_TD3_CRITIC_GRAD))
        if (int rc = launch_tick(stt, w.scalars, true, cfg->lr, cfg->beta1, cfg->beta2, -1.0, -1.0, -1.0, st)) return rc;
    if (phases & CSTR_TD3_CRITIC_GRAD) {
    if (sde) {  // actor.reset_noise() at the top of the loop body (sac.py): one E for the whole update, the same on every rank
        launch_k(sac_sde_draw_kernel, (unsigned)((H2 + 255) / 256), 256, 0, st, H2, (const float *)(actor.w3 + 2 * H2), (const float2 *)eps_pi, cfg->sde_seed,
                 (uint32_t)n_updates, dev_sc, w.sde);
        if (int rc = check_launch("sac_sde_draw_kernel")) return rc;
    }
    // ---- actions_pi, log_prob of the current actor (sac.py:222-223) and the entropy-coefficient step (:226-243) ----
    if (int rc = forward_hidden(B, H1, H2, OBS, obs, nullptr, actor, 0, 1, w.a_h1, w.a_h2, w.sc, st)) return rc;
    if (sde) launch_k(sac_sde_head_kernel, rb, 256, 0, st, B, H2, w.a_h2, actor.w3, actor.b3, w.sde, cfg->clip_mean, (float2 *)w.a_pi, w.logp,
                      (float2 *)w.raw_log_std, (float2 *)w.std_eps, w.lp_partial);
    else launch_k(sac_actor_head_kernel, rb, 256, 0, st, B, H2, w.a_h2, actor.w3, actor.b3, (const float2 *)eps_pi, cfg->seed, (uint32_t)n_updates, dev_sc, 0u, (float2 *)w.a_pi,
                                             w.logp, (float2 *)w.std_eps, (float2 *)w.raw_log_std, w.lp_partial);
    if (int rc = check_launch("sac_actor_head_kernel")) return rc;
    // one launch when nothing sits between gradient and step; split around the caller's all-reduce of grads[critics .. log_ent_coef] otherwise
    if (int rc = ent_coef(fused_ent ? 3 : 1)) return rc;
    // ---- target (sac.py:245-254): next action from the CURRENT actor (scratch: the dz slabs are free here) ----
    if (int rc = forward_hidden(B, H1, H2, OBS, next_obs, nullptr, actor, 0, 1, w.dz1, w.dz2, w.sc, st)) return rc;
    if (sde) launch_k(sac_sde_head_kernel, rb, 256, 0, st, B, H2, w.dz2, actor.w3, actor.b3, w.sde, cfg->clip_mean, (float2 *)w.next_act, w.next_logp,
                      nullptr, nullptr, nullptr);
    else launch_k(sac_actor_head_kernel, rb, 256, 0, st, B, H2, w.dz2, actor.w3, actor.b3, (const float2 *)eps_next, cfg->seed, (uint32_t)n_updates, dev_sc, 1u,
                                             (float2 *)w.next_act, w.next_logp, nullptr, nullptr, nullptr);
    if (int rc = check_launch("sac_actor_head_kernel<next>")) return rc;
    if (int rc = forward_hidden(B, H1, H2, OBS + ACT, next_obs, w.next_act, critic_t, cz, 2, w.t_h1, w.t_h2, w.sc, st)) return rc;
    launch_k(sac_target_head_kernel, rb, 256, 0, st, B, H2, w.t_h2, (int64_t)B * H2, critic_t.w3, critic_t.b3, cz, rewards, dones, w.next_logp, w.scalars,
                                              cfg->gamma, w.target);
    if (int rc = check_launch("sac_target_head_kernel")) return rc;
    // ---- critics (sac.py:256-268): loss = 0.5 * sum_i mse ----
    if (int rc = forward_hidden(B, H1, H2, OBS + ACT, obs, actions, critic, cz, 2, w.h1[0], w.h2[0], w.sc, st)) return rc;
    if (int rc = critic_loss_backward(B, H1, H2, td3_src(obs, actions, OBS + ACT), critic, g_critic, cz, 2, w.h1[0], w.h2[0], w.target, 1.f / (float)B, w.dq, w.dz2,
                                      w.dz1, w.loss_partial, w.sc, st))
        return rc;
    }  // CRITIC_GRAD
    if (phases & CSTR_TD3_CRITIC_APPLY) {
        if (!fused_ent && !stt->peer)
            if (int rc = ent_coef(2)) return rc;
        ApplyArgs a = adam;
        a.adam_lo = T.critic_off[0], a.adam_hi = T.total, a.polyak_lo = a.polyak_hi = 0;
        a.loss_partial = w.loss_partial, a.n_loss_partial = 2 * rb, a.loss_scale = 0.5f / (float)B, a.loss_acc = stt->losses;
        if (stt->peer) a.adam_hi = T.total + 4;  // the log_ent_coef slot rides in the same averaged Adam range (same formulas, same step size)
        if (int rc = launch_apply(a, stt->peer, stt->grads, st, "td3_apply_kernel<sac critic>")) return rc;
    }
    if (phases & CSTR_TD3_ACTOR_GRAD) {
    // ---- actor (sac.py:270-281): (ent_coef * log_prob - min_i Q_i(s, a_pi)).mean() with the updated critics ----
    if (int rc = forward_hidden(B, H1, H2, OBS + ACT, obs, w.a_pi, critic, cz, 2, w.h1[0], w.h2[0], w.sc, st)) return rc;
    launch_k(sac_qmin_head_kernel, rb, 256, 0, st, B, H2, w.h2[0], (int64_t)B * H2, critic.w3, critic.b3, cz, w.logp, w.scalars, w.dz2, w.loss_partial);
    if (int rc = check_launch("sac_qmin_head_kernel")) return rc;
    if (int rc = backward_dz1(B, H1, H2, critic, cz, 2, w.h1[0], w.dz2, w.dz1, w.sc, st)) return rc;
    // the actor's dz2 / dz1 live in the target-activation slabs (free since the target was formed)
    FinJobs J{};
    if (sde) {
        launch_k(sac_sde_bwd_head_kernel, rb, 256, 0, st, B, H1, H2, w.dz1, (int64_t)B * H1, critic.w1, cz, (const float2 *)w.a_pi,
                 (const float2 *)w.raw_log_std, (const float2 *)w.std_eps, w.scalars, actor.w3, w.sde, cfg->clip_mean, w.a_h2, (float4 *)w.dpre4,
                 (float2 *)w.dpre, w.t_h2);
        if (int rc = check_launch("sac_sde_bwd_head_kernel")) return rc;
        launch_k(sac_sde_wgrad_kernel, (unsigned)((H2 + 31) / 32), 256, 0, st, B, H2, w.a_h2, (const float4 *)w.dpre4, (const float2 *)w.dpre, w.sde,
                 g_actor.w3, g_actor.b3);
        if (int rc = check_launch("sac_sde_wgrad_kernel")) return rc;
    } else {
    launch_k(sac_actor_bwd_head_kernel, rb, 256, 0, st, B, H1, H2, w.dz1, (int64_t)B * H1, critic.w1, cz, (const float2 *)w.a_pi, (const float2 *)w.std_eps,
                                                 (const float2 *)w.raw_log_std, w.scalars, actor.w3, w.a_h2, (float4 *)w.dpre4, w.t_h2);
    if (int rc = check_launch("sac_actor_bwd_head_kernel")) return rc;
    SkinnyArgs s{};  // d[mu; log_std] head = dpre4^T @ h2a, bias = sum dpre4
    s.X = w.a_h2, s.x_z = 0, s.ldx = H2, s.H = H2, s.B = B;
    s.Y0 = w.dpre4, s.n0 = 2 * ACT, s.ld0 = 2 * ACT, s.Y1 = nullptr, s.n1 = 0, s.ld1 = 0, s.y_z = 0;
    s.out_w = g_actor.w3, s.out_b = g_actor.b3, s.out_z = 0, s.transposed = 1;
    if (int rc = launch_skinny<2 * ACT, true>(s, 1, w.sc.skinny + 2 * w.sc.skinny_region, st, "td3_skinny_wgrad_kernel<sac head>", J)) return rc;
    }
    if (int rc = backward_hidden(B, H1, H2, td3_src(obs, nullptr, OBS), nullptr, actor, g_actor, 0, 1, w.a_h1, w.t_h2, w.t_h1, w.sc, J, st)) return rc;
    }  // ACTOR_GRAD
    if (phases & CSTR_TD3_ACTOR_APPLY) {
        ApplyArgs a = adam;
        a.adam_lo = T.actor_off, a.adam_hi = T.actor_off + T.actor.size;
        // `gradient_step % target_update_interval == 0` (:284) with gradient_step the index inside the current train() call
        const int64_t loop_index = cfg->local_step > 0 ? (int64_t)cfg->local_step - 1 : n_updates - 1;
        const bool sync_targets = (loop_index % cfg->target_update_interval) == 0;
        a.polyak_lo = sync_targets ? T.critic_off[0] : 0, a.polyak_hi = sync_targets ? T.total : 0;
        a.loss_partial = w.loss_partial, a.n_loss_partial = rb, a.loss_scale = 1.f / (float)B, a.loss_acc = stt->losses ? stt->losses + 2 : nullptr;
        if (int rc = launch_apply(a, stt->peer, stt->grads, st, "td3_apply_kernel<sac actor+polyak>")) return rc;
    }
    return 0;
}

}  // extern "C"
#include "cstr_bcq.cuh"
#include "cstr_ma.cuh"
extern "C" {

// ---- peer memory for the fused gradient all-reduce (include/cstr_b200.h, cstr_peer_comm) ---------------------------------
int64_t cstr_peer_flag_bytes(void) { return (int64_t)(PEER_FLAG_WORDS + 4) * (int64_t)sizeof(uint32_t); }

int cstr_peer_alloc(int64_t bytes, void **ptr, void *handle64) {
    if (bytes <= 0 || !ptr || !handle64) return fail_arg(CSTR_EINVAL, "peer_alloc: bad arguments");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    void *p = nullptr;
    if (int rc = check_cuda(cudaMalloc(&p, (size_t)bytes), "peer_alloc: cudaMalloc")) return rc;
    if (int rc = check_cuda(cudaMemset(p, 0, (size_t)bytes), "peer_alloc: cudaMemset")) return rc;
    cudaIpcMemHandle_t h;
    if (int rc = check_cuda(cudaIpcGetMemHandle(&h, p), "peer_alloc: cudaIpcGetMemHandle")) {
        cudaFree(p);
        return rc;
    }
    if (int rc = check_cuda(cudaDeviceSynchronize(), "peer_alloc: sync")) return rc;
    memcpy(handle64, &h, 64);
    *ptr = p;
    return 0;
}

int cstr_peer_open(const void *handle64, void **ptr) {
    if (!handle64 || !ptr) return fail_arg(CSTR_EINVAL, "peer_open: bad arguments");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    return check_cuda(cudaIpcOpenMemHandle(ptr, h, cudaIpcMemLazyEnablePeerAccess), "peer_open: cudaIpcOpenMemHandle");
}

int cstr_peer_close(void *ptr) { return ptr ? check_cuda(cudaIpcCloseMemHandle(ptr), "peer_close") : 0; }

int cstr_peer_free(void *ptr) { return ptr ? check_cuda(cudaFree(ptr), "peer_free") : 0; }

int cstr_peer_error(const cstr_peer_comm *comm, uint32_t *error, void *stream) {
    if (!comm || !error || comm->rank < 0 || comm->rank >= CSTR_PEER_MAX_WORLD || !comm->flags[comm->rank]) return fail_arg(CSTR_EINVAL, "peer_error: bad arguments");
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = check_cuda(cudaMemcpyAsync(error, comm->flags[comm->rank] + PEER_ERROR, sizeof(uint32_t), cudaMemcpyDeviceToHost, st), "peer_error: copy")) return rc;
    return check_cuda(cudaStreamSynchronize(st), "peer_error: sync");
}

}  // extern "C"
