// BCQ gradient step on the device: cstr_bcq_update (include/cstr_b200.h).  Replaces the loop body of BCQ.train
// (core/bcq/bcq.py:137-205); restated from oracle/td3_oracle.py::BCQUpdateOracle, which is pinned against the reference.
// Included at the end of cstr_td3.cu (shares its kernels and host helpers).
#pragma once

namespace {

struct BcqLayout {
    NetLayout enc, dec, pert, critic;
    int64_t enc_off, dec_off, pert_off, critic_off[2], total;
};

inline BcqLayout bcq_layout(const cstr_bcq_config *c) {
    BcqLayout T;
    T.enc = net_layout(OBS + ACT, 2 * c->latent, c->vae_hidden, c->vae_hidden);
    T.dec = net_layout(OBS + c->latent, ACT, c->vae_hidden, c->vae_hidden);
    T.pert = net_layout(OBS + ACT, ACT, c->pert_hidden, c->pert_hidden);
    T.critic = net_layout(OBS + ACT, 1, c->h1, c->h2);
    T.enc_off = 0;
    T.dec_off = T.enc.size;
    T.pert_off = T.dec_off + T.dec.size;
    T.critic_off[0] = T.pert_off + T.pert.size;
    T.critic_off[1] = T.critic_off[0] + T.critic.size;
    T.total = T.critic_off[1] + T.critic.size;
    return T;
}

int check_bcq_cfg(const cstr_bcq_config *c) {
    if (!c) return fail_arg(CSTR_EINVAL, "bcq: null config");
    auto bad = [](int h) { return h < 4 || (h & 3) || h > 4096; };
    if (c->latent < 4 || (c->latent & 3) || c->latent > 64) return fail_arg(CSTR_EINVAL, "bcq: latent must be a multiple of 4 in [4, 64]");
    if (bad(c->vae_hidden) || bad(c->pert_hidden) || bad(c->h1) || bad(c->h2)) return fail_arg(CSTR_EINVAL, "bcq: hidden sizes must be multiples of 4 in [4, 4096]");
    if (c->batch < 1 || c->batch > (1 << 20)) return fail_arg(CSTR_EINVAL, "bcq: batch must be in [1, 1048576]");
    if (c->actor_delay < 1) return fail_arg(CSTR_EINVAL, "bcq: actor_delay must be >= 1");
    if (c->n_candidates < 1 || c->n_candidates > 64) return fail_arg(CSTR_EINVAL, "bcq: n_candidates must be in [1, 64]");
    if (c->gemm_mode < CSTR_TD3_GEMM_FP32 || c->gemm_mode > CSTR_TD3_GEMM_BF16) return fail_arg(CSTR_EINVAL, "bcq: gemm_mode must be 0, 1 or 2");
    return 0;
}

struct BcqWorkspace {
    // VAE pass (B rows)
    float *e_h1, *e_h2, *e_y, *std, *eps, *xdec, *d_h1, *d_h2, *recon, *d_dy, *v_dz2, *v_dz1, *dzl, *e_dy;
    // candidates (R = n_candidates * B rows)
    float *zc, *c_h1, *c_h2, *cand, *p_h1, *p_h2, *xi, *cand_p, *t_h1, *t_h2, *t_q;
    // critics (TD3 shapes) and the perturbation step
    float *h1, *h2, *dz1, *dz2, *target, *dq, *loss_partial, *za, *a0, *a, *pre, *da, *p_dy, *p_dz2, *p_dz1, *scalars;
    MlpScratch sc;
    int n_row_blocks;
    int64_t floats;
};

BcqWorkspace bcq_carve(float *base, const cstr_bcq_config *c) {
    BcqWorkspace w{};
    Bump b(base);
    const int64_t B = c->batch, R = B * c->n_candidates, L = c->latent, Hv = c->vae_hidden, Hp = c->pert_hidden, H1 = c->h1, H2 = c->h2;
    w.e_h1 = b.take(B * Hv), w.e_h2 = b.take(B * Hv), w.e_y = b.take(B * 2 * L), w.std = b.take(B * L), w.eps = b.take(B * L), w.xdec = b.take(B * (4 + L));
    w.d_h1 = b.take(B * Hv), w.d_h2 = b.take(B * Hv), w.recon = b.take(B * 2), w.d_dy = b.take(B * 2), w.v_dz2 = b.take(B * Hv), w.v_dz1 = b.take(B * Hv);
    w.dzl = b.take(B * L), w.e_dy = b.take(B * 2 * L);
    w.zc = b.take(R * L), w.c_h1 = b.take(R * Hv), w.c_h2 = b.take(R * Hv), w.cand = b.take(R * 2), w.p_h1 = b.take(R * Hp), w.p_h2 = b.take(R * Hp);
    w.xi = b.take(R * 2), w.cand_p = b.take(R * 2), w.t_h1 = b.take(2 * R * H1), w.t_h2 = b.take(2 * R * H2), w.t_q = b.take(2 * R);
    w.h1 = b.take(2 * B * H1), w.h2 = b.take(2 * B * H2), w.dz1 = b.take(2 * B * H1), w.dz2 = b.take(2 * B * H2), w.target = b.take(B), w.dq = b.take(2 * B);
    w.n_row_blocks = (int)((B + 7) / 8);
    w.loss_partial = b.take(2 * (int64_t)w.n_row_blocks);
    w.za = b.take(B * L), w.a0 = b.take(B * 2), w.a = b.take(B * 2), w.pre = b.take(B * 2), w.da = b.take(B * 2), w.p_dy = b.take(B * 2);
    w.p_dz2 = b.take(B * Hp), w.p_dz1 = b.take(B * Hp), w.scalars = b.take(8);
    int hm = (int)std::max(std::max(Hv, Hp), std::max(std::max(H1, H2), 2 * L));
    w.sc = mlp_scratch(b, (int)R, hm, 2, OBS + ACT);
    w.floats = b.o;
    return w;
}

}  // namespace

extern "C" {

int64_t cstr_bcq_param_count(const cstr_bcq_config *cfg) { return check_bcq_cfg(cfg) ? -1 : bcq_layout(cfg).total; }

int cstr_bcq_layout(const cstr_bcq_config *cfg, int64_t *offsets) {
    if (int rc = check_bcq_cfg(cfg)) return rc;
    if (!offsets) return fail_arg(CSTR_EINVAL, "bcq_layout: null output");
    const BcqLayout T = bcq_layout(cfg);
    put_offsets(offsets, 0, T.enc_off, T.enc);
    put_offsets(offsets, 1, T.dec_off, T.dec);
    put_offsets(offsets, 2, T.pert_off, T.pert);
    for (int n = 3; n < 5; ++n) put_offsets(offsets, n, T.critic_off[n - 3], T.critic);
    offsets[30] = T.total;
    return 0;
}

int64_t cstr_bcq_workspace_bytes(const cstr_bcq_config *cfg) {
    if (check_bcq_cfg(cfg)) return -1;
    return bcq_carve(nullptr, cfg).floats * (int64_t)sizeof(float);
}

int cstr_bcq_update(const cstr_bcq_config *cfg, const cstr_td3_state *stt, const float *obs, const float *actions, const float *next_obs,
                    const float *dones, const float *rewards, const float *eps_vae, const float *z_next, const float *z_actor, int64_t n_updates,
                    int64_t critic_step, int64_t actor_step, void *stream) {
    if (int rc = check_bcq_cfg(cfg)) return rc;
    if (int rc = check_update("bcq", stt, cstr_bcq_workspace_bytes(cfg), obs, actions, next_obs, dones, rewards, n_updates, critic_step, actor_step)) return rc;
    if ((eps_vae && !aligned(eps_vae, 16)) || (z_next && !aligned(z_next, 16)) || (z_actor && !aligned(z_actor, 16)))
        return fail_arg(CSTR_EALIGN, "bcq_update: latent draws need 16 B alignment");
    BcqWorkspace w = bcq_carve(stt->workspace, cfg);
    w.sc.tensor = cfg->gemm_mode;
    const BcqLayout T = bcq_layout(cfg);
    cudaStream_t st = (cudaStream_t)stream;
    const int B = cfg->batch, L = cfg->latent, K = cfg->n_candidates, H1 = cfg->h1, H2 = cfg->h2;
    const int64_t R = (int64_t)B * K, cz = T.critic.size;
    const int rb = w.n_row_blocks, tb = (B + 255) / 256;
    const bool actor_step_now = (n_updates % cfg->actor_delay) == 0;
    const Net enc = net_at(stt->params, T.enc_off, T.enc), dec = net_at(stt->params, T.dec_off, T.dec), pert = net_at(stt->params, T.pert_off, T.pert);
    const Net pert_t = net_at(stt->targets, T.pert_off, T.pert);
    const Net critic = net_at(stt->params, T.critic_off[0], T.critic), critic_t = net_at(stt->targets, T.critic_off[0], T.critic);
    const Net g_enc = net_at(stt->grads, T.enc_off, T.enc), g_dec = net_at(stt->grads, T.dec_off, T.dec), g_pert = net_at(stt->grads, T.pert_off, T.pert);
    const Net g_critic = net_at(stt->grads, T.critic_off[0], T.critic);
    const float *dev_sc = stt->counters ? w.scalars : nullptr;
    if (stt->counters)
        if (int rc = launch_tick(stt, w.scalars, actor_step_now, cfg->lr, cfg->beta1, cfg->beta2, -1.0, -1.0, -1.0, st)) return rc;

    // ---- VAE (bcq.py:142-155) ----
    Src s_enc{};
    s_enc.x0 = obs, s_enc.n0 = OBS, s_enc.ld0 = OBS, s_enc.x1 = actions, s_enc.n1 = ACT, s_enc.ld1 = ACT;
    if (int rc = forward_mlp(B, T.enc, s_enc, enc, 0, 1, w.e_h1, w.e_h2, w.e_y, false, w.sc, st)) return rc;
    launch_k(bcq_latent_kernel, (unsigned)(((int64_t)B * (L / 4) + 255) / 256), 256, 0, st, B, L, (const float *)w.e_y, eps_vae, cfg->seed, (uint32_t)n_updates, dev_sc,
             (const float4 *)obs, w.std, w.eps, w.xdec);
    if (int rc = check_launch("bcq_latent_kernel")) return rc;
    Src s_dec{};
    s_dec.x0 = w.xdec, s_dec.n0 = OBS + L, s_dec.ld0 = OBS + L;
    if (int rc = forward_mlp(B, T.dec, s_dec, dec, 0, 1, w.d_h1, w.d_h2, w.recon, true, w.sc, st)) return rc;
    launch_k(bcq_vae_loss_kernel, tb, 256, 0, st, B, L, (const float2 *)w.recon, (const float2 *)actions, (const float *)w.e_y, (const float *)w.std, (float2 *)w.d_dy,
             w.loss_partial);
    if (int rc = check_launch("bcq_vae_loss_kernel")) return rc;
    if (int rc = backward_mlp(B, T.dec, s_dec, w.xdec, dec, g_dec, w.d_h1, w.d_h2, w.d_dy, w.v_dz2, w.v_dz1, w.sc, st)) return rc;
    launch_k(mlp_dx_kernel, rb, 256, 0, st, B, T.dec.h1, OBS + L, (const float *)w.v_dz1, (const float *)dec.w1, OBS, L, w.dzl);
    if (int rc = check_launch("mlp_dx_kernel<latent>")) return rc;
    launch_k(bcq_enc_grad_kernel, (unsigned)(((int64_t)B * L + 255) / 256), 256, 0, st, B, L, (const float *)w.dzl, (const float *)w.e_y, (const float *)w.std,
             (const float *)w.eps, w.e_dy);
    if (int rc = check_launch("bcq_enc_grad_kernel")) return rc;
    if (int rc = backward_mlp(B, T.enc, s_enc, nullptr, enc, g_enc, w.e_h1, w.e_h2, w.e_dy, w.v_dz2, w.v_dz1, w.sc, st)) return rc;
    {
        ApplyArgs a = adam_args(stt, cfg->lr, cfg->beta1, cfg->beta2, cfg->eps, cfg->tau, critic_step, dev_sc, 0);
        a.adam_lo = T.enc_off, a.adam_hi = T.pert_off, a.polyak_lo = a.polyak_hi = 0;
        a.loss_partial = w.loss_partial, a.n_loss_partial = tb, a.loss_scale = 1.f, a.loss_acc = stt->losses;
        if (int rc = launch_apply(a, stt->peer, stt->grads, st, "td3_apply_kernel<bcq vae>")) return rc;
    }

    // ---- target (bcq.py:157-172): candidates from the refreshed (= current) VAE and the TARGET perturbation net ----
    launch_k(bcq_clip_latent_kernel, (unsigned)((R * (L / 4) + 255) / 256), 256, 0, st, R, L, z_next, cfg->seed, (uint32_t)n_updates, dev_sc, (uint32_t)STREAM_BCQ_NEXT, w.zc);
    if (int rc = check_launch("bcq_clip_latent_kernel<next>")) return rc;
    Src s_cdec{};
    s_cdec.x0 = next_obs, s_cdec.n0 = OBS, s_cdec.ld0 = OBS, s_cdec.x0_rows = B, s_cdec.x1 = w.zc, s_cdec.n1 = L, s_cdec.ld1 = L;
    if (int rc = forward_mlp((int)R, T.dec, s_cdec, dec, 0, 1, w.c_h1, w.c_h2, w.cand, true, w.sc, st)) return rc;
    Src s_cpert{};
    s_cpert.x0 = next_obs, s_cpert.n0 = OBS, s_cpert.ld0 = OBS, s_cpert.x0_rows = B, s_cpert.x1 = w.cand, s_cpert.n1 = ACT, s_cpert.ld1 = ACT;
    if (int rc = forward_mlp((int)R, T.pert, s_cpert, pert_t, 0, 1, w.p_h1, w.p_h2, w.xi, true, w.sc, st)) return rc;
    launch_k(bcq_perturb_kernel, (unsigned)((R + 255) / 256), 256, 0, st, R, (const float2 *)w.cand, (const float2 *)w.xi, cfg->max_perturbation, (float2 *)w.cand_p,
             (float2 *)nullptr);
    if (int rc = check_launch("bcq_perturb_kernel<target>")) return rc;
    Src s_cq = s_cpert;
    s_cq.x1 = w.cand_p;
    if (int rc = forward_mlp((int)R, T.critic, s_cq, critic_t, cz, 2, w.t_h1, w.t_h2, w.t_q, false, w.sc, st)) return rc;
    launch_k(bcq_target_kernel, tb, 256, 0, st, B, K, 2, (const float *)w.t_q, rewards, dones, cfg->gamma, w.target);
    if (int rc = check_launch("bcq_target_kernel")) return rc;

    // ---- critics (bcq.py:174-186): TD3's twin-critic step ----
    if (int rc = forward_hidden(B, H1, H2, OBS + ACT, obs, actions, critic, cz, 2, w.h1, w.h2, w.sc, st)) return rc;
    if (int rc = critic_loss_backward(B, H1, H2, td3_src(obs, actions, OBS + ACT), critic, g_critic, cz, 2, w.h1, w.h2, w.target, 2.f / (float)B, w.dq, w.dz2, w.dz1,
                                      w.loss_partial, w.sc, st))
        return rc;
    {
        ApplyArgs a = adam_args(stt, cfg->lr, cfg->beta1, cfg->beta2, cfg->eps, cfg->tau, critic_step, dev_sc, 0);
        a.adam_lo = T.critic_off[0], a.adam_hi = T.total, a.polyak_lo = a.polyak_hi = 0;
        a.loss_partial = w.loss_partial, a.n_loss_partial = 2 * rb, a.loss_scale = 1.f / (float)B, a.loss_acc = stt->losses ? stt->losses + 2 : nullptr;
        if (int rc = launch_apply(a, stt->peer, stt->grads, st, "td3_apply_kernel<bcq critic>")) return rc;
    }
    if (!actor_step_now) return 0;

    // ---- delayed perturbation step (bcq.py:188-203): -Q1(s, pert(s, dec(s, z))).mean(), only the perturbation optimiser steps ----
    if (actor_step < 1) return fail_arg(CSTR_EINVAL, "bcq_update: actor_step must be >= 1 on an actor step");
    launch_k(bcq_clip_latent_kernel, (unsigned)(((int64_t)B * (L / 4) + 255) / 256), 256, 0, st, (int64_t)B, L, z_actor, cfg->seed, (uint32_t)n_updates, dev_sc,
             (uint32_t)STREAM_BCQ_ACTOR, w.za);
    if (int rc = check_launch("bcq_clip_latent_kernel<actor>")) return rc;
    Src s_adec{};
    s_adec.x0 = obs, s_adec.n0 = OBS, s_adec.ld0 = OBS, s_adec.x1 = w.za, s_adec.n1 = L, s_adec.ld1 = L;
    if (int rc = forward_mlp(B, T.dec, s_adec, dec, 0, 1, w.d_h1, w.d_h2, w.a0, true, w.sc, st)) return rc;
    Src s_apert{};
    s_apert.x0 = obs, s_apert.n0 = OBS, s_apert.ld0 = OBS, s_apert.x1 = w.a0, s_apert.n1 = ACT, s_apert.ld1 = ACT;
    if (int rc = forward_mlp(B, T.pert, s_apert, pert, 0, 1, w.p_h1, w.p_h2, w.xi, true, w.sc, st)) return rc;
    launch_k(bcq_perturb_kernel, tb, 256, 0, st, (int64_t)B, (const float2 *)w.a0, (const float2 *)w.xi, cfg->max_perturbation, (float2 *)w.a, (float2 *)w.pre);
    if (int rc = check_launch("bcq_perturb_kernel<actor>")) return rc;
    if (int rc = forward_hidden(B, H1, H2, OBS + ACT, obs, w.a, critic, cz, 1, w.h1, w.h2, w.sc, st)) return rc;
    if (int rc = policy_critic_backward(B, H1, H2, critic, cz, w.h1, w.h2, w.dq, w.dz2, w.dz1, w.loss_partial, w.sc, st)) return rc;
    launch_k(mlp_dx_kernel, rb, 256, 0, st, B, H1, OBS + ACT, (const float *)w.dz1, (const float *)critic.w1, OBS, ACT, w.da);
    if (int rc = check_launch("mlp_dx_kernel<action>")) return rc;
    launch_k(bcq_pert_grad_kernel, tb, 256, 0, st, B, (const float2 *)w.da, (const float2 *)w.pre, (const float2 *)w.xi, cfg->max_perturbation, (float2 *)w.p_dy);
    if (int rc = check_launch("bcq_pert_grad_kernel")) return rc;
    if (int rc = backward_mlp(B, T.pert, s_apert, nullptr, pert, g_pert, w.p_h1, w.p_h2, w.p_dy, w.p_dz2, w.p_dz1, w.sc, st)) return rc;
    ApplyArgs a = adam_args(stt, cfg->lr, cfg->beta1, cfg->beta2, cfg->eps, cfg->tau, actor_step, dev_sc, 2);
    a.adam_lo = T.pert_off, a.adam_hi = T.critic_off[0], a.polyak_lo = T.pert_off, a.polyak_hi = T.total;  // pert + both critics: one contiguous range
    a.loss_partial = w.loss_partial, a.n_loss_partial = rb, a.loss_scale = -1.f / (float)B, a.loss_acc = stt->losses ? stt->losses + 4 : nullptr;
    return launch_apply(a, stt->peer, stt->grads, st, "td3_apply_kernel<bcq pert+polyak>");
}

}  // extern "C"
