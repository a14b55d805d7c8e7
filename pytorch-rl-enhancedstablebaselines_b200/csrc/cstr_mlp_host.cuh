// Host-side chaining of the update kernels (the GEMM / skinny / finalize / apply kernels of cstr_td3.cu and the generic MLP kernels of
// cstr_mlp.cuh): the forward and backward passes and the step pieces the TD3, SAC, BCQ and MADDPG / IDDPG updates are built from.
// Included inside cstr_td3.cu's anonymous namespace, after the launch helpers.
#pragma once

// bump allocator over the caller's workspace (base == nullptr: size query)
struct Bump {
    float *base;
    int64_t o = 0;
    explicit Bump(float *b) : base(b) {}
    float *take(int64_t n) {
        float *p = base ? base + o : nullptr;
        o += pad4(n);
        return p;
    }
};

// scratch the shared backward kernels need: split-K / dW2 slabs and one skinny partial-sum region per deferred job of a backward pass
struct MlpScratch {
    float *slabs, *skinny;
    int64_t slab_cap, skinny_region;  // floats
    int tensor;  // cfg->gemm_mode: 0 FFMA, 1 tcgen05 bf16x3 split, 2 tcgen05 plain bf16
};

// sized for hidden widths up to HM and Z nets per call
inline MlpScratch mlp_scratch(Bump &b, int rows, int HM, int Z, int max_skinny_ny) {
    MlpScratch s;
    s.slab_cap = (int64_t)MAX_SPLITS * Z * pad4((int64_t)HM * HM);
    s.slabs = b.take(s.slab_cap);
    const int64_t hp = ((int64_t)HM + 31) / 32 * 32;
    s.skinny_region = (int64_t)((rows + SKINNY_ROWS - 1) / SKINNY_ROWS) * Z * (max_skinny_ny + 1) * hp;
    s.skinny = b.take(3 * s.skinny_region);
    s.tensor = 0;
    return s;
}

template <bool YBIAS>
int launch_skinny_ny(int ny, SkinnyArgs s, int Z, float *part, cudaStream_t st, const char *what, FinJobs &J) {
    switch (ny) {
        case 0: return launch_skinny<0, false>(s, Z, part, st, what, J);
        case 1: return launch_skinny<1, YBIAS>(s, Z, part, st, what, J);
        case 2: return launch_skinny<2, YBIAS>(s, Z, part, st, what, J);
        case 3: return launch_skinny<3, YBIAS>(s, Z, part, st, what, J);
        case 4: return launch_skinny<4, YBIAS>(s, Z, part, st, what, J);
        case 6: return launch_skinny<6, YBIAS>(s, Z, part, st, what, J);
        default: return fail_arg(CSTR_EINVAL, "mlp: skinny weight gradient supports widths 0-4 and 6");
    }
}

// plain FFMA C (M,N) = A^T-role GEMM over the batch, written straight into the gradient tensor (one split: fixed summation order)
int wgrad_gemm_direct(int M, int N, int K, const float *A, int lda, const float *Bm, int ldb, float *C, int ldc, cudaStream_t st, const char *what) {
    if ((M & 3) || (N & 3) || (lda & 3) || (ldb & 3) || (ldc & 3)) return fail_arg(CSTR_EINVAL, "mlp: wide weight gradients need widths that are multiples of 4");
    GemmArgs q{};
    q.A = A, q.Bm = Bm, q.aux = nullptr, q.C = C;
    q.M = M, q.N = N, q.K = K, q.lda = lda, q.ldb = ldb, q.ldc = ldc, q.ldaux = 0;
    q.splits = 1, q.k_per_split = K, q.c_split = 0;
    return launch_gemm<G_WGRAD>(q, 1, 0, st, what);
}

// h2 = relu(L2(h1)) for Z nets `z_stride` floats apart (activations: Z slabs of B rows)
int forward_layer2(int B, int H1, int H2, const Net &n, int64_t z_stride, int Z, float *h1, float *h2, const MlpScratch &sc, cudaStream_t st) {
    GemmArgs g{};
    g.A = h1, g.Bm = n.w2, g.aux = n.b2, g.C = h2;
    g.M = B, g.N = H2, g.K = H1, g.lda = H1, g.ldb = H1, g.ldc = H2, g.ldaux = 0;
    g.a_z = (int64_t)B * H1, g.b_z = z_stride, g.c_z = (int64_t)B * H2, g.aux_z = z_stride;
    g.splits = 1, g.k_per_split = H1, g.c_split = 0;
    g.split_buf = sc.slabs, g.split_cap = sc.slab_cap;
    return launch_gemm<G_FWD>(g, Z, sc.tensor, st, "td3_gemm_kernel<fwd>");
}

// h1 = relu(L1([obs | act])) through td3_layer1_kernel (in = 4: obs only, 6: obs and act), then layer 2
int forward_hidden(int B, int H1, int H2, int in, const float *obs, const float *act, const Net &n, int64_t z_stride, int Z, float *h1, float *h2,
                   const MlpScratch &sc, cudaStream_t st) {
    const int64_t threads = (int64_t)((B + L1_ROWS - 1) / L1_ROWS) * (H1 / 4);
    dim3 grid((unsigned)((threads + 255) / 256), Z);
    if (in == OBS)
        launch_k(td3_layer1_kernel<OBS>, grid, 256, 0, st, B, H1, (const float4 *)obs, nullptr, n.w1, n.b1, z_stride, h1, (int64_t)B * H1);
    else
        launch_k(td3_layer1_kernel<OBS + ACT>, grid, 256, 0, st, B, H1, (const float4 *)obs, (const float2 *)act, n.w1, n.b1, z_stride, h1, (int64_t)B * H1);
    if (int rc = check_launch("td3_layer1_kernel")) return rc;
    return forward_layer2(B, H1, H2, n, z_stride, Z, h1, h2, sc, st);
}

// h1 = relu(L1(x)) over any layer-1 source through mlp_layer1_kernel, then layer 2
int forward_hidden_g(int B, const NetLayout &L, const Src &s, const Net &n, int64_t z_stride, int Z, float *h1, float *h2, const MlpScratch &sc,
                     cudaStream_t st) {
    if (s.n0 + s.n1 != L.in) return fail_arg(CSTR_EINVAL, "mlp: source widths do not add up to the net's input width");
    const int64_t threads = (int64_t)((B + L1G_ROWS - 1) / L1G_ROWS) * (L.h1 / 4);
    launch_k(mlp_layer1_kernel, dim3((unsigned)((threads + 255) / 256), Z), 256, 0, st, B, L.h1, s, (const float *)n.w1, (const float *)n.b1, z_stride, h1,
             (int64_t)B * L.h1);
    if (int rc = check_launch("mlp_layer1_kernel")) return rc;
    return forward_layer2(B, L.h1, L.h2, n, z_stride, Z, h1, h2, sc, st);
}

// ... followed by the linear head: y (Z, B, out), tanh when squash
int forward_mlp(int B, const NetLayout &L, const Src &s, const Net &n, int64_t z_stride, int Z, float *h1, float *h2, float *y, bool squash,
                const MlpScratch &sc, cudaStream_t st) {
    if (int rc = forward_hidden_g(B, L, s, n, z_stride, Z, h1, h2, sc, st)) return rc;
    launch_k(mlp_head_fwd_kernel, dim3((B + 7) / 8, Z), 256, 0, st, B, L.h2, L.out, (const float *)h2, (int64_t)B * L.h2, (const float *)n.w3, (const float *)n.b3,
             z_stride, y, squash ? 1 : 0);
    return check_launch("mlp_head_fwd_kernel");
}

// dz1 = (dz2 @ W2) * (h1 > 0) for Z nets
int backward_dz1(int B, int H1, int H2, const Net &n, int64_t z_stride, int Z, const float *h1, const float *dz2, float *dz1, const MlpScratch &sc,
                 cudaStream_t st) {
    GemmArgs g{};
    g.A = dz2, g.Bm = n.w2, g.aux = h1, g.C = dz1;
    g.M = B, g.N = H1, g.K = H2, g.lda = H2, g.ldb = H1, g.ldc = H1, g.ldaux = H1;
    g.a_z = (int64_t)B * H2, g.b_z = z_stride, g.c_z = (int64_t)B * H1, g.aux_z = (int64_t)B * H1;
    g.splits = 1, g.k_per_split = H2, g.c_split = 0;
    g.split_buf = sc.slabs, g.split_cap = sc.slab_cap;
    return launch_gemm<G_DGRAD>(g, Z, sc.tensor, st, "td3_gemm_kernel<dgrad>");
}

// Given dz2 (and h1, the layer-1 source): dz1, then every weight gradient of layers 1 and 2 into `gn`.  The second stages run as jobs of
// one finalize launch, together with the jobs the caller already queued in J (its layer-3 gradient, region 2 of the skinny scratch).
// x_wide: the contiguous (B, in) input, needed (instead of the skinny kernel) for dW1 when in > 6 or in == 5.
int backward_hidden(int B, int H1, int H2, const Src &src, const float *x_wide, const Net &n, const Net &gn, int64_t z_stride, int Z, const float *h1,
                    const float *dz2, float *dz1, const MlpScratch &sc, FinJobs &J, cudaStream_t st) {
    if (int rc = backward_dz1(B, H1, H2, n, z_stride, Z, h1, dz2, dz1, sc, st)) return rc;
    // dW2 = dz2^T @ h1, split over the batch into slabs, then summed in order by the finalize launch
    const int64_t w2n = pad4((int64_t)H1 * H2);
    GemmArgs q{};
    q.A = dz2, q.Bm = h1, q.aux = nullptr, q.C = sc.slabs;
    q.M = H2, q.N = H1, q.K = B, q.lda = H2, q.ldb = H1, q.ldc = H1, q.ldaux = 0;
    q.a_z = (int64_t)B * H2, q.b_z = (int64_t)B * H1, q.c_z = w2n, q.aux_z = 0;
    const int splits = choose_splits(B, H1, H2, Z, sc.tensor);
    q.splits = splits, q.k_per_split = (B + splits - 1) / splits, q.c_split = 2 * w2n;
    if (int rc = launch_gemm<G_WGRAD>(q, Z, sc.tensor, st, "td3_gemm_kernel<wgrad>")) return rc;
    J.slab_n4 = (int64_t)H1 * H2 / 4, J.slab_splits = splits, J.slabs = (const float4 *)sc.slabs, J.slab_stride4 = 2 * w2n / 4, J.slab_z4 = w2n / 4;
    J.slab_out = (float4 *)gn.w2, J.slab_out_z4 = z_stride / 4, J.slab_Z = Z;
    // db2 = colsum(dz2)
    SkinnyArgs s{};
    s.X = dz2, s.x_z = (int64_t)B * H2, s.ldx = H2, s.H = H2, s.B = B;
    s.out_w = nullptr, s.out_b = gn.b2, s.out_z = z_stride;
    if (int rc = launch_skinny<0, false>(s, Z, sc.skinny, st, "td3_skinny_wgrad_kernel<b2>", J)) return rc;
    const int in = src.n0 + src.n1;
    SkinnyArgs t{};
    t.X = dz1, t.x_z = (int64_t)B * H1, t.ldx = H1, t.H = H1, t.B = B;
    t.out_b = gn.b1, t.out_z = z_stride;
    if (in <= 6 && in != 5) {  // dW1 = dz1^T @ [x0 | x1] (TD3: [obs | act]), db1 = colsum(dz1)
        if (src.x0_rows) return fail_arg(CSTR_EINVAL, "mlp: weight gradients over a repeated source are not supported");
        t.Y0 = src.x0, t.n0 = src.n0, t.ld0 = src.ld0, t.Y1 = src.x1, t.n1 = src.n1, t.ld1 = src.ld1, t.y_z = 0;
        t.out_w = gn.w1;
        if (int rc = launch_skinny_ny<false>(in, t, Z, sc.skinny + sc.skinny_region, st, "td3_skinny_wgrad_kernel<w1>", J)) return rc;
    } else {  // a wide input (the VAE decoder's [obs | z]): GEMM over the batch, and db1 alone through the skinny kernel
        if (!x_wide) return fail_arg(CSTR_EINVAL, "mlp: a layer-1 input wider than 6 needs its contiguous copy for the weight gradient");
        if (int rc = wgrad_gemm_direct(H1, in, B, dz1, H1, x_wide, in, gn.w1, in, st, "td3_gemm_kernel<wgrad layer1>")) return rc;
        t.out_w = nullptr;
        if (int rc = launch_skinny<0, false>(t, Z, sc.skinny + sc.skinny_region, st, "td3_skinny_wgrad_kernel<b1>", J)) return rc;
    }
    return launch_finalize(J, st);
}

// Given dy (B, out; tanh' already applied by the caller) and the forward activations: every weight gradient of ONE net into `gn`, and dz1 left in
// `dz1` for a following mlp_dx_kernel.
int backward_mlp(int B, const NetLayout &L, const Src &s, const float *x_wide, const Net &n, const Net &gn, const float *h1, const float *h2,
                 const float *dy, float *dz2, float *dz1, const MlpScratch &sc, cudaStream_t st) {
    const int H2 = L.h2, OUT = L.out;
    launch_k(mlp_head_bwd_kernel, (B + 7) / 8, 256, 0, st, B, H2, OUT, dy, (const float *)n.w3, h2, dz2);
    if (int rc = check_launch("mlp_head_bwd_kernel")) return rc;
    FinJobs J{};
    if (OUT <= 4) {  // dW3 = dy^T @ h2, db3 = sum_b dy
        SkinnyArgs k{};
        k.X = h2, k.x_z = 0, k.ldx = H2, k.H = H2, k.B = B;
        k.Y0 = dy, k.n0 = OUT, k.ld0 = OUT, k.Y1 = nullptr, k.n1 = 0, k.ld1 = 0, k.y_z = 0;
        k.out_w = gn.w3, k.out_b = gn.b3, k.out_z = 0, k.transposed = 1;
        if (int rc = launch_skinny_ny<true>(OUT, k, 1, sc.skinny + 2 * sc.skinny_region, st, "td3_skinny_wgrad_kernel<w3>", J)) return rc;
    } else {  // a wide head (the VAE's [mean; log_std]): GEMM over the batch + a column sum for the bias
        if (int rc = wgrad_gemm_direct(OUT, H2, B, dy, OUT, h2, H2, gn.w3, H2, st, "td3_gemm_kernel<wgrad head>")) return rc;
        SkinnyArgs k{};
        k.X = dy, k.x_z = 0, k.ldx = OUT, k.H = OUT, k.B = B;
        k.out_w = nullptr, k.out_b = gn.b3, k.out_z = 0;
        if (int rc = launch_skinny<0, false>(k, 1, sc.skinny + 2 * sc.skinny_region, st, "td3_skinny_wgrad_kernel<b3>", J)) return rc;
    }
    return backward_hidden(B, L.h1, H2, s, x_wide, n, gn, 0, 1, h1, dz2, dz1, sc, J, st);
}

// The critic step's backward for ZC critics `cz` floats apart, from their forward activations: the squared-error head (dq = scale (q - target),
// dz2 and the per-CTA loss partials), dW3 / db3 as a deferred skinny job, then the hidden layers' gradients.
int critic_loss_backward(int B, int H1, int H2, const Src &src, const Net &critic, const Net &g_critic, int64_t cz, int ZC, const float *h1,
                         const float *h2, const float *target, float scale, float *dq, float *dz2, float *dz1, float *loss_partial, const MlpScratch &sc,
                         cudaStream_t st) {
    launch_k(td3_critic_head_kernel<false>, dim3((B + 7) / 8, ZC), 256, 0, st, B, H2, h2, (int64_t)B * H2, (const float *)critic.w3, (const float *)critic.b3, cz,
             target, scale, dq, dz2, loss_partial);
    if (int rc = check_launch("td3_critic_head_kernel")) return rc;
    SkinnyArgs s{};  // dW3 = dq^T @ h2, db3 = sum dq
    s.X = h2, s.x_z = (int64_t)B * H2, s.ldx = H2, s.H = H2, s.B = B;
    s.Y0 = dq, s.n0 = 1, s.ld0 = 1, s.Y1 = nullptr, s.n1 = 0, s.ld1 = 0, s.y_z = B;
    s.out_w = g_critic.w3, s.out_b = g_critic.b3, s.out_z = cz, s.transposed = 1;
    FinJobs J{};
    if (int rc = launch_skinny<1, true>(s, ZC, sc.skinny + 2 * sc.skinny_region, st, "td3_skinny_wgrad_kernel<w3>", J)) return rc;
    return backward_hidden(B, H1, H2, src, nullptr, critic, g_critic, cz, ZC, h1, dz2, dz1, sc, J, st);
}

// The policy loss -Q1(s, pi(s)).mean() through critic 0, from its forward activations on the policy's actions: the head (dq = -1/B, dz2, loss
// partials), then dz1 for the gradient with respect to the critic's input.  No critic weight gradients.
int policy_critic_backward(int B, int H1, int H2, const Net &critic, int64_t cz, const float *h1, const float *h2, float *dq, float *dz2, float *dz1,
                           float *loss_partial, const MlpScratch &sc, cudaStream_t st) {
    launch_k(td3_critic_head_kernel<true>, dim3((B + 7) / 8, 1), 256, 0, st, B, H2, h2, (int64_t)B * H2, (const float *)critic.w3, (const float *)critic.b3, cz,
             (const float *)nullptr, 0.f, dq, dz2, loss_partial);
    if (int rc = check_launch("td3_critic_head_kernel<policy>")) return rc;
    return backward_dz1(B, H1, H2, critic, cz, 1, h1, dz2, dz1, sc, st);
}

// One optimiser's Adam step `step` (1-based) over the state blocks: torch's bias corrections in double.  Graph mode (dev_sc != NULL) reads
// {step_size, bc2_sqrt} from dev_sc[slot..] instead, where td3_tick_kernel wrote them.  The caller sets the ranges and the loss fold.
ApplyArgs adam_args(const cstr_td3_state *stt, double lr, float beta1, float beta2, float eps, float tau, int64_t step, const float *dev_sc, int slot) {
    ApplyArgs a{};
    a.p = stt->params, a.t = stt->targets, a.g = stt->grads, a.m = stt->adam_m, a.v = stt->adam_v;
    const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
    a.beta1 = beta1, a.beta2 = beta2, a.eps = eps, a.step_size = (float)(lr / bc1), a.bc2_sqrt = (float)sqrt(bc2), a.tau = tau;
    a.dev_scalars = dev_sc ? dev_sc + slot : nullptr;
    return a;
}

// What every update entry point checks before its first launch (after its config): state and batch pointers, their alignment, the
// workspace size and the 1-based counters.  `name` prefixes the message ("td3" -> "td3_update: ...").
int check_update(const char *name, const cstr_td3_state *stt, int64_t workspace_bytes, const float *obs, const float *actions, const float *next_obs,
                 const float *dones, const float *rewards, int64_t n_updates, int64_t critic_step, int64_t actor_step) {
    char msg[160];
    auto fail = [&](int code, const char *what) {
        snprintf(msg, sizeof msg, "%s_update: %s", name, what);
        return fail_arg(code, msg);
    };
    if (!stt || !stt->params || !stt->targets || !stt->grads || !stt->adam_m || !stt->adam_v || !stt->workspace) return fail(CSTR_EINVAL, "null state pointer");
    if (!obs || !actions || !next_obs || !dones || !rewards) return fail(CSTR_EINVAL, "null batch pointer");
    if (!aligned(obs, 16) || !aligned(next_obs, 16) || !aligned(actions, 8) || !aligned(stt->params, 16) || !aligned(stt->targets, 16) ||
        !aligned(stt->grads, 16) || !aligned(stt->adam_m, 16) || !aligned(stt->adam_v, 16) || !aligned(stt->workspace, 16))
        return fail(CSTR_EALIGN, "16 B (obs, params, workspace) / 8 B (actions) alignment");
    if (stt->workspace_bytes < workspace_bytes) {
        char what[96];
        snprintf(what, sizeof what, "workspace too small (cstr_%s_workspace_bytes)", name);
        return fail(CSTR_EINVAL, what);
    }
    if (n_updates < 1 || critic_step < 1 || actor_step < 0) return fail(CSTR_EINVAL, "counters are 1-based (value after this update)");
    return 0;
}

// graph mode: advance the device counters and derive the update's scalars (td3_tick_kernel); lr_a / lr_c2 / lr_a2 = -1: not used
int launch_tick(const cstr_td3_state *stt, float *scalars, bool policy_step, double lr, float beta1, float beta2, double lr_a, double lr_c2, double lr_a2,
                cudaStream_t st) {
    launch_k(td3_tick_kernel, 1, 32, 0, st, stt->counters, scalars, policy_step ? 1 : 0, lr, (double)beta1, (double)beta2, lr_a, lr_c2, lr_a2);
    return check_launch("td3_tick_kernel");
}

// the `*_layout` exports: net n's six tensor offsets (W1 b1 W2 b2 W3 b3) at offsets[6n .. 6n+5]
void put_offsets(int64_t *offsets, int n, int64_t base, const NetLayout &L) {
    const int64_t o[6] = {L.w1, L.b1, L.w2, L.b2, L.w3, L.b3};
    for (int k = 0; k < 6; ++k) offsets[n * 6 + k] = base + o[k];
}
