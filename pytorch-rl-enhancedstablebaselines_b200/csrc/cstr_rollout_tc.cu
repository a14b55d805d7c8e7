// K2, tensor-core path — fused rollout with the actor's hidden layer on tcgen05 (sm_100a only).
//
//   obs (4) --W1,b1,relu--> h1 (H1) ==W2 on tcgen05.mma, bf16 x bf16 -> fp32 in TMEM==> (H2) --b2,relu,W3,b3,tanh--> mu (2)
//   -> exploration noise -> action maps -> CSTR step -> reward/done -> replay record        (same tail as the fp32 path)
//
// One CTA owns a tile of 128 reactors for the K steps of the launch; the reactor state never leaves
// registers.  Warp roles (10 warps):
//   warps 0-7  "env" warps: thread t serves reactor m = t % 128, half h = t / 128.  Each step they
//              (a) compute layer 1 in fp32 on the CUDA cores, K-chunk by K-chunk, and write it as bf16 straight
//                  into the UMMA A-operand image in shared memory (no-swizzle K-major: 16-byte st.shared,
//                  conflict-free), (b) read the accumulator row of their reactor out of TMEM (tcgen05.ld),
//                  apply b2/relu and contract with W3 (half of the columns per thread), (c) run the env step.
//   warp 8     W2 loader: streams the pre-packed bf16 K-chunks of W2 (L2-resident, 243 KB) into a 3-deep
//              shared-memory ring with cp.async.bulk + mbarrier complete_tx (TMA bulk engine).
//   warp 9     MMA issuer: one elected thread issues tcgen05.mma (M=128, N=160+144, K=16) accumulating over the
//              K-chunks in TMEM, and tcgen05.commit's to the mbarriers that free the operand buffers.
// Layer-1 compute of chunk c+1 overlaps the MMAs of chunk c (A is double-buffered); the accumulators
// (128 lanes x N_pad fp32 columns) live in TMEM and are only read once per step.
//
// Reference replaced: same as cstr_rollout.cu (off_policy_algorithm.py:364-411,445-508,564; td3/policies.py:75-78;
// policies.py:331-413; buffers.py:247-283).  bf16 operands => the action differs from the fp32 actor by
// ~1e-2 relative in the pre-activation (documented tolerance, tests/test_gpu_rollout.py); everything
// after the actor (maps, step, reward, record) is the strict fp32 arithmetic.
#include <cuda_bf16.h>

#include "cstr_abi.cuh"
#include "cstr_device.cuh"
#include "cstr_rollout_common.cuh"

namespace cstr {

constexpr int TC_M = 128;             // reactors per CTA = UMMA M
#ifndef TC_PER_
#define TC_PER_ 2
#endif
constexpr int TC_PER = TC_PER_;                 // env threads per reactor (2 or 4): they split the accumulator columns
constexpr int TC_ENV_THREADS = TC_M * TC_PER;
constexpr int TC_ENV_WARPS = TC_ENV_THREADS / 32;
constexpr int TC_THREADS = TC_ENV_THREADS + 96;  // + loader warp + two MMA-issuer warps
constexpr int TC_WSTAGES = 3;
constexpr int TC_ASTAGES = 2;

struct TcGeometry {
    int H1, H2;      // actor hidden sizes
    int KC;          // K-chunk (multiple of 16, divides H1)
    int NKC;         // H1 / KC
    int NP;          // H2 padded to a multiple of 16
    int N0, N1;      // MMA instruction widths: N0 + N1 == NP, each a multiple of 16 and <= 256 (N1 may be 0)
    int tmem_cols;   // power of two >= NP
    uint32_t a_chunk_bytes, w_chunk_bytes;
    uint32_t off_w1, off_a1, off_ep, off_part, off_a, off_w, smem_bytes;
    int d1_col;      // first TMEM column of the two layer-1 accumulator buffers (KC columns each)
};

static bool make_geometry(int H1, int H2, TcGeometry &g) {
    g.H1 = H1; g.H2 = H2;
    if (H1 <= 0 || H2 <= 0 || (H1 % 16) || H1 > 1024) return false;
    g.NP = (H2 + 15) & ~15;
    if (g.NP > 512) return false;
    const int cands[] = {80, 64, 48, 32, 16};
    g.KC = 0;
    for (int c : cands)
        if (H1 % c == 0) { g.KC = c; break; }
    if (!g.KC) return false;
    g.NKC = H1 / g.KC;
    if (g.NP <= 256) { g.N0 = g.NP; g.N1 = 0; }
    else { g.N0 = ((g.NP / 2) + 15) & ~15; g.N1 = g.NP - g.N0; }
    g.d1_col = g.NP;
    if (g.NP + 2 * g.KC > 512) return false;  // layer-2 accumulator + two layer-1 chunk accumulators must fit in TMEM
    g.tmem_cols = 32;
    while (g.tmem_cols < g.NP + 2 * g.KC) g.tmem_cols <<= 1;
    auto up = [](uint32_t x) { return (x + 127u) & ~127u; };
    g.a_chunk_bytes = (uint32_t)(g.KC / 8) * TC_M * 16;
    g.w_chunk_bytes = (uint32_t)(g.KC / 8) * g.NP * 16;
    g.off_w1 = 256;                                             // [0,256): mbarriers + tmem base
    g.off_a1 = up(g.off_w1 + 2u * H1 * 16);                     // W1 split-bf16 UMMA image [2][H1][8 x bf16]
    g.off_ep = up(g.off_a1 + 2u * TC_M * 16);                   // layer-1 A operand [2][128][8 x bf16]
    g.off_part = up(g.off_ep + 5u * g.NP * 4);                  // b2 and up to four W3 rows (zero padded)
    g.off_a = up(g.off_part + 2 * TC_PER * TC_M * 4 * 4);            // layer-3 partial sums [step parity][half][m] x float4
    g.off_w = up(g.off_a + TC_ASTAGES * g.a_chunk_bytes);
    g.smem_bytes = up(g.off_w + TC_WSTAGES * g.w_chunk_bytes);
    return g.smem_bytes <= 227u * 1024u;
}

// ---- PTX wrappers ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}\n" ::"r"(bar), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// 8 consecutive fp32 columns of this thread's TMEM lane
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float v[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 8 hidden units of the layer-2/3 epilogue: h = relu(acc + b2); o[r] += W3[r] * h for the NOUT head rows.
// sep = [1 + NOUT][NP] floats (b2, then the W3 rows), col = first of the 8 columns (multiple of 8: 32-byte aligned).
template <int NOUT>
__device__ __forceinline__ void epi8(const float v[8], const float *sep, int NP, int col, float o[4]) {
    const float4 *bv = reinterpret_cast<const float4 *>(sep + col);
    const float4 ba = bv[0], bb = bv[1];
    const float b[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
    float h[8];
#pragma unroll
    for (int q = 0; q < 8; ++q) h[q] = fmaxf(v[q] + b[q], 0.0f);
#pragma unroll
    for (int r = 0; r < NOUT; ++r) {
        const float4 *wv = reinterpret_cast<const float4 *>(sep + (size_t)(1 + r) * NP + col);
        const float4 wa = wv[0], wb = wv[1];
        const float w[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
        for (int q = 0; q < 8; ++q) o[r] = fmaf(w[q], h[q], o[r]);
    }
}

// UMMA shared-memory descriptor, K-major, SWIZZLE_NONE (cute::UMMA::SmemDescriptor, version 1):
// canonical layout ((8,n),2):((16 B, SBO), LBO) — 8x16-byte core matrices, SBO between 8-row groups,
// LBO between the two 8-element K halves of one K=16 instruction.
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;  // descriptor version (Blackwell)
    return d;                // base_offset 0, lbo_mode 0, layout_type 0 (no swizzle)
}
// cute::UMMA::InstrDescriptor for kind::f16: D=f32, A=B=bf16, both K-major, dense
__host__ __device__ inline uint32_t umma_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// barrier slots inside the first 256 bytes of shared memory
enum { BAR_W_FULL = 0, BAR_W_EMPTY = 3, BAR_A_FULL = 6, BAR_A_EMPTY = 8, BAR_D_FULL = 10, BAR_A1_FULL = 11, BAR_D1_FULL = 12, BAR_D1_EMPTY = 14, BAR_ORDER = 16, BAR_COUNT = 18 };

// NORM (cstr_rollout_fused_norm, K == 1): layer 1 reads the normalised observation, done rows keep their raw terminal observation until
// the statistics that include this step exist, and the CTA's moment sums go to norm_merge.
template <int MODE, int KIND, bool NORM>
__global__ void __launch_bounds__(TC_THREADS, 1)
rollout_tc_kernel(cstr_env_params p, int64_t n, int64_t K, ActorNet actor, const uint8_t *__restrict__ packed_w2, TcGeometry g,
                  float sigma, const float2 *__restrict__ noise, uint32_t t_base, float4 *__restrict__ state,
                  int32_t *__restrict__ step_count, int32_t *__restrict__ episode, double *static_base, int64_t rows, int64_t pos0,
                  float4 *__restrict__ records, double *reward_sum, cstr_episode_stats stats, int has_stats, NormLaunch nl) {
    extern __shared__ __align__(128) uint8_t smem[];
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bars = smem_base;  // BAR_COUNT x 8 bytes
    volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem + 128);
    constexpr int NOUT = KIND == CSTR_ACTOR_GAUSSIAN ? 4 : 2;
    float *sep = reinterpret_cast<float *>(smem + g.off_ep);     // [1 + NOUT][NP]: b2, then the W3 rows
    float4 *spart = reinterpret_cast<float4 *>(smem + g.off_part);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int H1 = g.H1, NP = g.NP;

    // ---- one-time setup ---------------------------------------------------------------------------------
    if (tid == 0) {
        for (int b = 0; b < TC_WSTAGES; ++b) { mbar_init(bars + 8 * (BAR_W_FULL + b), 1); mbar_init(bars + 8 * (BAR_W_EMPTY + b), 1); }
        for (int b = 0; b < TC_ASTAGES; ++b) { mbar_init(bars + 8 * (BAR_A_FULL + b), TC_ENV_THREADS); mbar_init(bars + 8 * (BAR_A_EMPTY + b), 1); }
        mbar_init(bars + 8 * BAR_D_FULL, 1);
        mbar_init(bars + 8 * BAR_A1_FULL, TC_ENV_THREADS);
        for (int b = 0; b < 2; ++b) mbar_init(bars + 8 * (BAR_ORDER + b), 1);
        for (int b = 0; b < 2; ++b) { mbar_init(bars + 8 * (BAR_D1_FULL + b), 1); mbar_init(bars + 8 * (BAR_D1_EMPTY + b), TC_ENV_THREADS); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == TC_ENV_WARPS + 1) {  // TMEM allocation is warp-collective; the same warp frees it at the end
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void *)tmem_slot)),
                     "r"((uint32_t)g.tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // Layer 1 (K=4 + bias) as ONE K=16 bf16 MMA with fp32-grade accuracy: x = x_hi + x_lo (two bf16 each), and
    //   W.s + b ~= W_hi.s_hi + W_hi.s_lo + W_lo.s_hi + b_hi + b_lo          (the dropped W_lo.s_lo term is ~2^-18 relative)
    // B1 row j = [W_hi(4) | W_hi(4)] [W_lo(4) | b_hi b_lo 0 0]   against   A1 row m = [s_hi(4) | s_lo(4)] [s_hi(4) | 1 1 0 0]
    for (int j = tid; j < H1; j += TC_THREADS) {
        const float4 w = __ldg(reinterpret_cast<const float4 *>(actor.W1) + j);
        const float b = __ldg(actor.b1 + j);
        const float wf[4] = {w.x, w.y, w.z, w.w};
        __nv_bfloat16 hi[4], lo[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) { hi[q] = __float2bfloat16_rn(wf[q]); lo[q] = __float2bfloat16_rn(wf[q] - __bfloat162float(hi[q])); }
        const __nv_bfloat16 bhi = __float2bfloat16_rn(b), blo = __float2bfloat16_rn(b - __bfloat162float(bhi)), z = __float2bfloat16_rn(0.0f);
        __nv_bfloat16 *g0 = reinterpret_cast<__nv_bfloat16 *>(smem + g.off_w1 + (size_t)j * 16);
        __nv_bfloat16 *g1 = reinterpret_cast<__nv_bfloat16 *>(smem + g.off_w1 + (size_t)(H1 + j) * 16);
#pragma unroll
        for (int q = 0; q < 4; ++q) { g0[q] = hi[q]; g0[4 + q] = hi[q]; g1[q] = lo[q]; }
        g1[4] = bhi; g1[5] = blo; g1[6] = z; g1[7] = z;
    }
    for (int j = tid; j < NP; j += TC_THREADS) {
        const bool in = j < g.H2;
        sep[0 * NP + j] = in ? __ldg(actor.b2 + j) : 0.0f;
#pragma unroll
        for (int r = 0; r < NOUT; ++r) sep[(1 + r) * NP + j] = in ? __ldg(actor.W3 + (size_t)r * g.H2 + j) : 0.0f;
    }
    fence_proxy_async();  // the W1 image above is read by the tensor core (async proxy)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int kgroups = g.KC / 8;  // 16-byte K groups per chunk
    double nacc[NORM_SUMS];
    if constexpr (NORM) {
#pragma unroll
        for (int j = 0; j < NORM_SUMS; ++j) nacc[j] = 0.0;
    }

    if (warp < TC_ENV_WARPS) {
        // =========================== env warps ===========================================================
        const int m = tid & (TC_M - 1), half = tid >> 7;
        const int64_t i = (int64_t)blockIdx.x * TC_M + m;
        const bool live = i < n;
        float4 s = live ? state[i] : make_float4(0.f, 0.f, 0.f, 0.f);
        int sc = live ? step_count[i] : 0, ep = live ? episode[i] : 0;
        const uint64_t env = (uint64_t)(p.env_offset + i);
        float b3[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int r = 0; r < NOUT; ++r) b3[r] = __ldg(actor.b3 + r);
        double acc_r = 0.0;
        double ep_ret = (has_stats && live && half == 0) ? stats.ep_return[i] : 0.0;
        double sb[4] = {0.0, 0.0, 0.0, 0.0};
        if (static_base && live) {
#pragma unroll
            for (int q = 0; q < 4; ++q) sb[q] = static_base[4 * i + q];
        }
        uint32_t gchunk = 0;
        const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
        if constexpr (NORM) {
            if (live && half == 0) norm_fix_pending(nl, i, n, records);
        }

#ifdef CSTR_TC_TIMING
        long long T0 = 0, T1 = 0, T2 = 0, T3 = 0, T4 = 0;
#define CSTR_TICK(x) x = clock64()
#else
#define CSTR_TICK(x)
#endif
        for (int64_t k = 0; k < K; ++k) {
            CSTR_TICK(T0);
            // ---- (a) layer 1 on the tensor core: publish this step's split-bf16 observation row (A1) ... -------------
            const uint32_t gstep = t_base + (uint32_t)k;
            {
                float4 sa = s;
                if constexpr (NORM) {
                    if (nl.norm_obs) sa = norm_obs4(s, nl);
                }
                const float sf[4] = {sa.x, sa.y, sa.z, sa.w};
                __nv_bfloat16 hi[4], lo[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) { hi[q] = __float2bfloat16_rn(sf[q]); lo[q] = __float2bfloat16_rn(sf[q] - __bfloat162float(hi[q])); }
                const __nv_bfloat16 one = __float2bfloat16_rn(1.0f), z = __float2bfloat16_rn(0.0f);
                __nv_bfloat162 p0 = __halves2bfloat162(hi[0], hi[1]), p1 = __halves2bfloat162(hi[2], hi[3]);
                __nv_bfloat162 p2 = half == 0 ? __halves2bfloat162(lo[0], lo[1]) : __halves2bfloat162(one, one);
                __nv_bfloat162 p3 = half == 0 ? __halves2bfloat162(lo[2], lo[3]) : __halves2bfloat162(z, z);
                if (half < 2) {  // the layer-1 A operand has two K groups: parts 0 and 1 publish them
                uint4 pk;
                pk.x = *reinterpret_cast<uint32_t *>(&p0); pk.y = *reinterpret_cast<uint32_t *>(&p1);
                pk.z = *reinterpret_cast<uint32_t *>(&p2); pk.w = *reinterpret_cast<uint32_t *>(&p3);
                *reinterpret_cast<uint4 *>(smem + g.off_a1 + (size_t)half * (TC_M * 16) + m * 16) = pk;  // K group = half
                }
                fence_proxy_async();
                mbar_arrive(bars + 8 * BAR_A1_FULL);
            }
            float2 nz;  // exploration noise does not depend on the actor: drawn here, while the first MMAs are in flight
            if (noise) nz = live ? noise[k * n + i] : make_float2(0.f, 0.f);
            else if (KIND == CSTR_ACTOR_GAUSSIAN) nz = philox_normal2(p.seed, env, gstep);  // eps ~ N(0,1) of the squashed Gaussian
            else if (sigma != 0.0f) { nz = philox_normal2(p.seed, env, gstep); nz.x *= sigma; nz.y *= sigma; }
            else nz = make_float2(0.f, 0.f);
            // ---- ... then turn each layer-1 accumulator chunk (TMEM) into the bf16 A operand of layer 2 (relu + pack) ---
            for (int kc = 0; kc < g.NKC; ++kc, ++gchunk) {
                const uint32_t ab = gchunk & 1u;
                const uint32_t db = (uint32_t)kc & 1u, duse = (uint32_t)(k * ((g.NKC + 1 - (int)db) / 2) + (kc >> 1));
                mbar_wait(bars + 8 * (BAR_D1_FULL + db), duse & 1u);
                tc_fence_after();
                const uint32_t d1 = tmem_base + lane_base + (uint32_t)(g.d1_col + (int)db * g.KC);
                constexpr int KGT = (10 + TC_PER - 1) / TC_PER;  // K-groups per thread and chunk (KC <= 80); static indices only
                float v[KGT][8];
#pragma unroll
                for (int c5 = 0; c5 < KGT; ++c5) {
                    const int kg = half + TC_PER * c5;
                    if (kg < kgroups) tmem_ld8(d1 + (uint32_t)(kg * 8), v[c5]);
                }
                tmem_ld_wait();
                tc_fence_before();
                mbar_arrive(bars + 8 * (BAR_D1_EMPTY + db));  // this chunk's layer-1 accumulator may be overwritten
                // No "A buffer empty" barrier: the layer-1 MMA of THIS chunk was issued after the layer-2 MMAs that last read
                // this A buffer (chunk g-2) on the same in-order tensor pipe, and its commit (D1_FULL, waited above) tracks
                // completion of everything issued before it — so the buffer is already free.
                uint8_t *abuf = smem + g.off_a + ab * g.a_chunk_bytes;
#pragma unroll
                for (int c5 = 0; c5 < KGT; ++c5) {
                    const int kg = half + TC_PER * c5;
                    if (kg < kgroups) {
                        __nv_bfloat162 h01 = __floats2bfloat162_rn(fmaxf(v[c5][0], 0.f), fmaxf(v[c5][1], 0.f));
                        __nv_bfloat162 h23 = __floats2bfloat162_rn(fmaxf(v[c5][2], 0.f), fmaxf(v[c5][3], 0.f));
                        __nv_bfloat162 h45 = __floats2bfloat162_rn(fmaxf(v[c5][4], 0.f), fmaxf(v[c5][5], 0.f));
                        __nv_bfloat162 h67 = __floats2bfloat162_rn(fmaxf(v[c5][6], 0.f), fmaxf(v[c5][7], 0.f));
                        uint4 pk;
                        pk.x = *reinterpret_cast<uint32_t *>(&h01); pk.y = *reinterpret_cast<uint32_t *>(&h23);
                        pk.z = *reinterpret_cast<uint32_t *>(&h45); pk.w = *reinterpret_cast<uint32_t *>(&h67);
                        *reinterpret_cast<uint4 *>(abuf + (size_t)kg * (TC_M * 16) + m * 16) = pk;  // [kg][m][8 x bf16]
                    }
                }
                fence_proxy_async();  // generic-proxy smem writes -> visible to the tensor core (async proxy)
                mbar_arrive(bars + 8 * (BAR_A_FULL + ab));
            }
            CSTR_TICK(T1);
            // ---- (b) epilogue: TMEM row -> b2, relu, W3 --------------------------------------------------
            mbar_wait(bars + 8 * BAR_D_FULL, (uint32_t)(k & 1));
            CSTR_TICK(T2);
            tc_fence_after();
            float o[4] = {0.f, 0.f, 0.f, 0.f};
            // the NP/8 eight-column groups of the row are dealt round-robin to the reactor's threads: group index = half + TC_PER * j
            const uint32_t d2 = tmem_base + lane_base;
            const int my_groups = (NP / 8 - half + TC_PER - 1) / TC_PER;
            float va[8], vb[8];
            if (my_groups > 0) tmem_ld8(d2 + (uint32_t)(half * 8), va);
            for (int j = 0; j < my_groups; j += 2) {  // two groups per trip, loads one group ahead of the math
                const int c0 = (half + TC_PER * j) * 8, c1 = c0 + TC_PER * 8, c2 = c1 + TC_PER * 8;
                tmem_ld_wait();
                if (j + 1 < my_groups) tmem_ld8(d2 + (uint32_t)c1, vb);
                // constants come as 16-byte broadcast loads (scalar LDS made the epilogue shared-memory-issue bound)
                epi8<NOUT>(va, sep, NP, c0, o);
                if (j + 1 < my_groups) {
                    tmem_ld_wait();
                    if (j + 2 < my_groups) tmem_ld8(d2 + (uint32_t)c2, va);
                    epi8<NOUT>(vb, sep, NP, c1, o);
                }
            }
            CSTR_TICK(T3);
            tc_fence_before();  // TMEM reads are complete before anybody re-arms the accumulator
            float4 *sp = spart + (size_t)(k & 1) * (TC_PER * TC_M);  // double-buffered by step parity: one barrier per step
            sp[half * TC_M + m] = make_float4(o[0], o[1], o[2], o[3]);
            asm volatile("bar.sync 1, %0;" ::"n"(TC_ENV_THREADS) : "memory");
            float4 ps = sp[m];
#pragma unroll
            for (int q = 1; q < TC_PER; ++q) {  // same order in every thread of the reactor
                const float4 pq = sp[q * TC_M + m];
                ps.x += pq.x, ps.y += pq.y, ps.z += pq.z, ps.w += pq.w;
            }
            const float head[4] = {ps.x + b3[0], ps.y + b3[1], ps.z + b3[2], ps.w + b3[3]};
            float mu0, mu1;
            float2 add;
            actor_head<KIND>(head, nz, mu0, mu1, add);
            // ---- (c) noise, action maps, env step, record (both threads of a pair compute, half 0 stores) ---
            float2 env_a, buf_a;
            action_maps(mu0, add.x, env_a.x, buf_a.x);
            action_maps(mu1, add.y, env_a.y, buf_a.y);
            const float4 obs = s;
            const StepResult r = (MODE == CSTR_MATH_STRICT) ? step_strict_f32(s, env_a, sc, (float)p.target_c2, p.max_steps)
                                                            : step_fast_f32(s, env_a, sc, (float)p.target_c2, p.max_steps);
            if (live && half == 0) {
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
#ifdef CSTR_TC_TIMING
            CSTR_TICK(T4);
            if (blockIdx.x == 0 && tid == 0 && (k == 6 || k == 7))
                printf("tc-timing k=%d chunks=%lld drain=%lld epilogue=%lld tail=%lld total=%lld cycles\n", (int)k, T1 - T0, T2 - T1, T3 - T2, T4 - T3, T4 - T0);
#endif
            if (r.truncated) {
                // both threads of a pair draw the same reset from the same Philox counter; in static mode each keeps its own
                // copy of the drifting base state (Q2) and only half 0 writes it back at the end of the launch
                s = reset_f32_call(p.seed, env, (uint32_t)ep, p.init_mode, static_base ? sb : nullptr);
                ep += 1;
                sc = 0;
            }
            if constexpr (NORM) {
                if (live && half == 0) norm_account(nl, i, s, r.reward, r.truncated, nacc);
            }
        }
        if (live && half == 0) {
            state[i] = s;
            step_count[i] = sc;
            episode[i] = ep;
            if (has_stats) stats.ep_return[i] = ep_ret;
            if (static_base) {
#pragma unroll
                for (int q = 0; q < 4; ++q) static_base[4 * i + q] = sb[q];
            }
        }
        if (reward_sum) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) acc_r += __shfl_down_sync(0xffffffffu, acc_r, o);
            if (lane == 0 && half == 0) atomicAdd(reward_sum, acc_r);
        }
    } else if (warp == TC_ENV_WARPS) {
        // =========================== W2 loader ===========================================================
        if (lane == 0) {
            const uint32_t total = (uint32_t)(K * g.NKC);
            for (uint32_t gc = 0; gc < total; ++gc) {
                const uint32_t wb = gc % TC_WSTAGES, use = gc / TC_WSTAGES;
                mbar_wait(bars + 8 * (BAR_W_EMPTY + wb), (use & 1u) ^ 1u);
                mbar_expect_tx(bars + 8 * (BAR_W_FULL + wb), g.w_chunk_bytes);
                bulk_g2s(smem_base + g.off_w + wb * g.w_chunk_bytes, packed_w2 + (size_t)(gc % g.NKC) * g.w_chunk_bytes, g.w_chunk_bytes,
                         bars + 8 * (BAR_W_FULL + wb));
            }
        }
    } else {
        // =========================== MMA issuers (warps 9 and 10) ==========================================
        // Two issuing threads take alternate chunks.  tcgen05.mma issue is effectively synchronous (the thread blocks
        // ~76 cycles per MMA while the pipe is busy) and every tcgen05.commit / mbarrier wait costs the issuing thread
        // another 75-130 cycles: with one issuer a chunk cost ~1,450 cycles for 760 cycles of tensor time.  With two, one
        // thread's commits, waits and layer-1 MMA overlap the other thread's layer-2 MMAs.  Pipe order between the two
        // threads is the ORDER token (tcgen05.fence::before_thread_sync + mbarrier arrive / wait + fence::after).
        if (lane == 0) {
            const uint32_t me = (uint32_t)(warp - (TC_ENV_WARPS + 1));  // chunk gc is issued by thread (gc & 1)
            const uint32_t idesc0 = umma_idesc_bf16(TC_M, g.N0), idesc1 = g.N1 ? umma_idesc_bf16(TC_M, g.N1) : 0;
            const uint32_t lbo_a = TC_M * 16, lbo_b = (uint32_t)NP * 16, sbo = 128;
            const uint64_t a_step = (uint64_t)((2u * lbo_a) >> 4), b_step = (uint64_t)((2u * lbo_b) >> 4);  // one K=16 step, in 16-byte units
            const uint64_t n1_off = (uint64_t)(((uint32_t)g.N0 * 16u) >> 4);
            uint64_t a_desc0[TC_ASTAGES], b_desc0[TC_WSTAGES];
#pragma unroll
            for (int b2 = 0; b2 < TC_ASTAGES; ++b2) a_desc0[b2] = umma_desc(smem_base + g.off_a + b2 * g.a_chunk_bytes, lbo_a, sbo);
#pragma unroll
            for (int b2 = 0; b2 < TC_WSTAGES; ++b2) b_desc0[b2] = umma_desc(smem_base + g.off_w + b2 * g.w_chunk_bytes, lbo_b, sbo);
            const int ksteps = g.KC / 16;
            // layer 1: one K=16 MMA per chunk, A1 = split-bf16 observation rows, B1 = this chunk's rows of the W1 image
            const uint32_t idesc_l1 = umma_idesc_bf16(TC_M, g.KC);
            const uint64_t da1 = umma_desc(smem_base + g.off_a1, TC_M * 16, sbo);
            const uint64_t dw1_0 = umma_desc(smem_base + g.off_w1, (uint32_t)H1 * 16, sbo);
            const uint64_t w1_step = (uint64_t)(((uint32_t)g.KC * 16u) >> 4);
            const uint32_t d1_per_step[2] = {(uint32_t)((g.NKC + 1) / 2), (uint32_t)(g.NKC / 2)};  // uses of each layer-1 buffer per step
            auto issue_l1 = [&](int64_t k, int kc) {
                const uint32_t db = (uint32_t)kc & 1u;
                const uint32_t uses = (uint32_t)k * (db ? d1_per_step[1] : d1_per_step[0]) + (uint32_t)(kc >> 1);  // uses before this one
                mbar_wait(bars + 8 * (BAR_D1_EMPTY + db), (uses & 1u) ^ 1u);  // env threads drained the previous use
                tc_fence_after();
                tc_mma_bf16(tmem_base + (uint32_t)(g.d1_col + (int)db * g.KC), da1, dw1_0 + (uint64_t)kc * w1_step, idesc_l1, 0u);
                tc_commit(bars + 8 * (BAR_D1_FULL + db));
            };
            uint32_t order_waits = 0;  // completed waits on my ORDER token
            uint32_t gc = 0;
            for (int64_t k = 0; k < K; ++k) {
                // the first two layer-1 MMAs of the step go to the threads that own chunks 0 and 1
                const uint32_t own0 = gc & 1u, own1 = own0 ^ 1u;
                bool ordered = false;  // this thread already holds the ORDER token for its first chunk of the step
                if (me == own0 || (g.NKC > 1 && me == own1)) {
                    if (g.NKC == 1 && gc > 0) {
                        // One chunk per step: the threads take alternate steps, so this one skipped the previous step's A1_FULL phase,
                        // and parity k&1 also matches the phase two steps back, which has completed long ago.  Waiting first for
                        // the other thread's chunk gc-1 (issued after it waited for the previous phase) leaves only this step's phase.
                        mbar_wait(bars + 8 * (BAR_ORDER + me), order_waits & 1u);
                        order_waits += 1;
                        ordered = true;
                    }
                    mbar_wait(bars + 8 * BAR_A1_FULL, (uint32_t)(k & 1));  // this step's observation rows are in shared memory
                    tc_fence_after();
                    if (me == own0) issue_l1(k, 0);
                    if (g.NKC > 1 && me == own1) issue_l1(k, 1);
                }
                for (int kc = 0; kc < g.NKC; ++kc, ++gc) {
                    if ((gc & 1u) != me) continue;
                    const uint32_t wb = gc % TC_WSTAGES, wuse = gc / TC_WSTAGES, ab = gc & 1u, ause = gc >> 1;  // A_FULL phase = use count of the A buffer
                    mbar_wait(bars + 8 * (BAR_W_FULL + wb), wuse & 1u);
                    mbar_wait(bars + 8 * (BAR_A_FULL + ab), ause & 1u);
                    if (gc > 0 && !ordered) {  // the other thread has issued chunk gc-1: keeps the accumulation order (chunk 0 overwrites)
                        mbar_wait(bars + 8 * (BAR_ORDER + me), order_waits & 1u);
                        order_waits += 1;
                    }
                    tc_fence_after();
                    uint64_t da = ab == 0 ? a_desc0[0] : a_desc0[1];
                    uint64_t dbw = wb == 0 ? b_desc0[0] : (wb == 1 ? b_desc0[1] : b_desc0[2]);
                    uint32_t acc = kc > 0 ? 1u : 0u;
                    for (int j = 0; j < ksteps; ++j) {
                        tc_mma_bf16(tmem_base, da, dbw, idesc0, acc);
                        if (g.N1) tc_mma_bf16(tmem_base + (uint32_t)g.N0, da, dbw + n1_off, idesc1, acc);
                        da += a_step;
                        dbw += b_step;
                        acc = 1u;
                    }
                    tc_fence_before();
                    mbar_arrive(bars + 8 * (BAR_ORDER + (me ^ 1u)));  // hand the pipe to the other issuer
                    tc_commit(bars + 8 * (BAR_W_EMPTY + wb));  // operand buffers are free once these MMAs retire
                    if (kc == g.NKC - 1) tc_commit(bars + 8 * BAR_D_FULL);  // in-order pipe: the last chunk retires after all others
                    if (kc + 2 < g.NKC) issue_l1(k, kc + 2);  // its accumulator buffer was drained before A chunk kc was published
                }
            }
        }
    }
    // ---- teardown ---------------------------------------------------------------------------------------------
    tc_fence_before();
    __syncthreads();
    if (warp == TC_ENV_WARPS + 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)g.tmem_cols) : "memory");
    }
    if constexpr (NORM) {  // the odd-step half of the layer-3 partials is never written when K == 1: it holds the sums
        if (nl.training) norm_merge<TC_THREADS>(nl, n, nacc, reinterpret_cast<double *>(spart + TC_PER * TC_M));
    }
}

// W2 (H2,H1) fp32 -> bf16 UMMA image: [kc][kg][n (NP, zero padded)][8 x bf16], one contiguous chunk per kc
__global__ void pack_w2_kernel(const float *__restrict__ W2, int H1, int H2, int KC, int NP, __nv_bfloat16 *__restrict__ out) {
    const int64_t total = (int64_t)(H1 / 8) * NP * 8;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x) {
        const int e = (int)(idx & 7);
        const int64_t t = idx >> 3;
        const int nrow = (int)(t % NP);
        const int kgg = (int)(t / NP);  // global K group = kc * (KC/8) + kg
        const int kcol = kgg * 8 + e;
        out[idx] = __float2bfloat16_rn(nrow < H2 ? W2[(size_t)nrow * H1 + kcol] : 0.0f);
    }
    (void)KC;
}

}  // namespace cstr

using namespace cstr;

int cstr_rollout_tc_launch(const cstr_env_params *p, int64_t n, int64_t K, int math_mode, const cstr_actor_f32 *actor,
                           const void *packed_bf16, float sigma, const float *noise, int warmup, uint32_t t_base, float *state,
                           int32_t *step_count, int32_t *episode, double *static_base, int64_t rows, int64_t pos0, float *records,
                           double *reward_sum, const cstr_episode_stats *stats, const NormLaunch *nl, void *stream) {
    (void)warmup;
    TcGeometry g;
    if (!make_geometry(actor->H1, actor->H2, g)) return fail_arg(CSTR_EINVAL, "rollout(tc): H1 must be a multiple of 16 (<=1024), H2 rounded up to 16 plus two layer-1 K-chunks must fit 512 TMEM columns (H2 <= 480), and the operands must fit in shared memory");
    if (!packed_bf16) return fail_arg(CSTR_EINVAL, "rollout(tc): packed bf16 weights missing (cstr_actor_pack_bf16)");
    if (!aligned(packed_bf16, 16)) return fail_arg(CSTR_EALIGN, "rollout(tc): packed weights must be 16-byte aligned");
    if ((int64_t)K * g.NKC >= (int64_t)1 << 31) return fail_arg(CSTR_EINVAL, "rollout(tc): K too large");
    const int grid = (int)((n + TC_M - 1) / TC_M);
    cudaStream_t st = (cudaStream_t)stream;
    int rc = 0;
#define CSTR_LAUNCH_TC(MODE, KIND)                                                                                                          \
    do {                                                                                                                                    \
        rc = check_cuda(cudaFuncSetAttribute(rollout_tc_kernel<MODE, KIND, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem_bytes), "smem attr"); \
        if (!rc)                                                                                                                            \
            rollout_tc_kernel<MODE, KIND, false><<<grid, TC_THREADS, g.smem_bytes, st>>>(*p, n, K, net, (const uint8_t *)packed_bf16, g, sigma, (const float2 *)noise, \
                                                                                  t_base, (float4 *)state, step_count, episode, static_base, rows, pos0,   \
                                                                                  (float4 *)records, reward_sum, st_copy, has_stats, NormLaunch{}); \
    } while (0)
    cstr_episode_stats st_copy = {};
    const int has_stats = stats != nullptr;
    if (stats) st_copy = *stats;
#define CSTR_LAUNCH_TC_NORM(MODE, KIND)                                                                                                     \
    do {                                                                                                                                    \
        rc = check_cuda(cudaFuncSetAttribute(rollout_tc_kernel<MODE, KIND, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem_bytes), "smem attr"); \
        if (!rc)                                                                                                                            \
            rollout_tc_kernel<MODE, KIND, true><<<grid, TC_THREADS, g.smem_bytes, st>>>(*p, n, K, net, (const uint8_t *)packed_bf16, g, sigma,         \
                                                                                       (const float2 *)noise, t_base, (float4 *)state, step_count,   \
                                                                                       episode, static_base, rows, pos0, (float4 *)records,          \
                                                                                       reward_sum, st_copy, has_stats, *nl);                         \
    } while (0)
    const ActorNet net = actor_net(*actor);
    const bool gauss = actor->kind == CSTR_ACTOR_GAUSSIAN;
    if (nl) {
        if (K != 1) return fail_arg(CSTR_EINVAL, "rollout(tc): the VecNormalize variant runs one step per launch");
        if (math_mode == CSTR_MATH_STRICT) { if (gauss) CSTR_LAUNCH_TC_NORM(CSTR_MATH_STRICT, CSTR_ACTOR_GAUSSIAN); else CSTR_LAUNCH_TC_NORM(CSTR_MATH_STRICT, CSTR_ACTOR_TANH); }
        else { if (gauss) CSTR_LAUNCH_TC_NORM(CSTR_MATH_FAST, CSTR_ACTOR_GAUSSIAN); else CSTR_LAUNCH_TC_NORM(CSTR_MATH_FAST, CSTR_ACTOR_TANH); }
    } else if (math_mode == CSTR_MATH_STRICT) { if (gauss) CSTR_LAUNCH_TC(CSTR_MATH_STRICT, CSTR_ACTOR_GAUSSIAN); else CSTR_LAUNCH_TC(CSTR_MATH_STRICT, CSTR_ACTOR_TANH); }
    else { if (gauss) CSTR_LAUNCH_TC(CSTR_MATH_FAST, CSTR_ACTOR_GAUSSIAN); else CSTR_LAUNCH_TC(CSTR_MATH_FAST, CSTR_ACTOR_TANH); }
#undef CSTR_LAUNCH_TC
#undef CSTR_LAUNCH_TC_NORM
    if (rc) return rc;
    return check_launch("rollout_tc_kernel");
}

extern "C" int64_t cstr_actor_pack_bf16(const cstr_actor_f32 *actor, void *dst, void *stream) {
    if (!actor || !actor->W2) { fail_arg(CSTR_EINVAL, "actor_pack_bf16: null actor"); return -1; }
    TcGeometry g;
    if (!make_geometry(actor->H1, actor->H2, g)) { fail_arg(CSTR_EINVAL, "actor_pack_bf16: unsupported actor shape"); return -1; }
    const int64_t bytes = (int64_t)g.NKC * g.w_chunk_bytes;
    if (!dst) return bytes;
    if (!aligned(dst, 16)) { fail_arg(CSTR_EALIGN, "actor_pack_bf16: dst must be 16-byte aligned"); return -2; }
    pack_w2_kernel<<<256, 256, 0, (cudaStream_t)stream>>>(actor->W2, g.H1, g.H2, g.KC, g.NP, (__nv_bfloat16 *)dst);
    if (check_launch("pack_w2_kernel")) return -3;
    return bytes;
}
