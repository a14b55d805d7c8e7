// MADDPG / IDDPG gradient step on the device: cstr_ma_update (include/cstr_b200.h).  Replaces the loop body shared by
// MADDPG.train (core/maddpg/maddpg.py:127-185) and IDDPG.train (core/iddpg/iddpg.py:127-185) for the two-reactor agents;
// restated from oracle/td3_oracle.py::MultiAgentDDPGOracle, which is pinned against the reference (including its in-loop polyak, the
// agent-i observation fed to every actor, and the learning-rate pairing).  Included at the end of cstr_td3.cu.
#pragma once

namespace {

constexpr int MA_AGENTS = 2, MA_OBS = 2, MA_ACT = 1;  // per agent: observation_splits [[0,1],[2,3]], action_splits [[0],[1]]

struct MaLayout {
    NetLayout actor, critic;
    int n_critics;
    int64_t actor_off[MA_AGENTS], critic_off[MA_AGENTS], total;  // critic_off[i]: first q-network of agent i (its n_critics are contiguous)
};

inline MaLayout ma_layout(const cstr_ma_config *c) {
    MaLayout T;
    T.n_critics = c->n_critics;
    T.actor = net_layout(MA_OBS, MA_ACT, c->h1, c->h2);
    T.critic = net_layout(c->centralised ? OBS + ACT : MA_OBS + MA_ACT, 1, c->h1, c->h2);
    int64_t o = 0;
    for (int i = 0; i < MA_AGENTS; ++i) T.actor_off[i] = o, o += T.actor.size;
    for (int i = 0; i < MA_AGENTS; ++i) T.critic_off[i] = o, o += (int64_t)c->n_critics * T.critic.size;
    T.total = o;
    return T;
}

int check_ma_cfg(const cstr_ma_config *c) {
    if (!c) return fail_arg(CSTR_EINVAL, "ma: null config");
    if (c->h1 < 4 || c->h2 < 4 || (c->h1 & 3) || (c->h2 & 3) || c->h1 > 4096 || c->h2 > 4096) return fail_arg(CSTR_EINVAL, "ma: hidden sizes must be multiples of 4 in [4, 4096]");
    if (c->batch < 1 || c->batch > (1 << 22)) return fail_arg(CSTR_EINVAL, "ma: batch must be in [1, 4194304]");
    if (c->policy_delay < 1) return fail_arg(CSTR_EINVAL, "ma: policy_delay must be >= 1");
    if (c->n_critics < 1 || c->n_critics > 2) return fail_arg(CSTR_EINVAL, "ma: n_critics must be 1 or 2");
    if (c->centralised != 0 && c->centralised != 1) return fail_arg(CSTR_EINVAL, "ma: centralised must be 0 (IDDPG) or 1 (MADDPG)");
    if (c->gemm_mode < CSTR_TD3_GEMM_FP32 || c->gemm_mode > CSTR_TD3_GEMM_BF16) return fail_arg(CSTR_EINVAL, "ma: gemm_mode must be 0, 1 or 2");
    return 0;
}

struct MaWorkspace {
    float *a_h1, *a_h2, *a_y, *next_act, *t_h1, *t_h2, *target, *h1, *h2, *dz1, *dz2, *dq, *loss_partial, *joint, *da, *a_dy, *a_dz2, *a_dz1, *scalars;
    MlpScratch sc;
    int n_row_blocks;
    int64_t floats;
};

MaWorkspace ma_carve(float *base, const cstr_ma_config *c) {
    MaWorkspace w{};
    Bump b(base);
    const int64_t B = c->batch, H1 = c->h1, H2 = c->h2;
    w.a_h1 = b.take(MA_AGENTS * B * H1), w.a_h2 = b.take(MA_AGENTS * B * H2), w.a_y = b.take(MA_AGENTS * B), w.next_act = b.take(B * MA_AGENTS);
    w.t_h1 = b.take(2 * B * H1), w.t_h2 = b.take(2 * B * H2), w.target = b.take(B);
    w.h1 = b.take(2 * B * H1), w.h2 = b.take(2 * B * H2), w.dz1 = b.take(2 * B * H1), w.dz2 = b.take(2 * B * H2), w.dq = b.take(2 * B);
    w.n_row_blocks = (int)((B + 7) / 8);
    w.loss_partial = b.take(2 * (int64_t)w.n_row_blocks);
    w.joint = b.take(B * MA_AGENTS), w.da = b.take(B), w.a_dy = b.take(B), w.a_dz2 = b.take(B * H2), w.a_dz1 = b.take(B * H1), w.scalars = b.take(16);
    w.sc = mlp_scratch(b, (int)B, (int)std::max(H1, H2), 2, OBS + ACT);
    w.floats = b.o;
    return w;
}

}  // namespace

extern "C" {

int64_t cstr_ma_param_count(const cstr_ma_config *cfg) { return check_ma_cfg(cfg) ? -1 : ma_layout(cfg).total; }

int cstr_ma_layout(const cstr_ma_config *cfg, int64_t *offsets) {
    if (int rc = check_ma_cfg(cfg)) return rc;
    if (!offsets) return fail_arg(CSTR_EINVAL, "ma_layout: null output");
    const MaLayout T = ma_layout(cfg);
    int n = 0;
    for (int i = 0; i < MA_AGENTS; ++i) put_offsets(offsets, n++, T.actor_off[i], T.actor);
    for (int i = 0; i < MA_AGENTS; ++i)
        for (int k = 0; k < T.n_critics; ++k) put_offsets(offsets, n++, T.critic_off[i] + k * T.critic.size, T.critic);
    offsets[n * 6] = T.total;
    return 0;
}

int64_t cstr_ma_workspace_bytes(const cstr_ma_config *cfg) {
    if (check_ma_cfg(cfg)) return -1;
    return ma_carve(nullptr, cfg).floats * (int64_t)sizeof(float);
}

int cstr_ma_update(const cstr_ma_config *cfg, const cstr_td3_state *stt, const float *obs, const float *actions, const float *next_obs,
                   const float *dones, const float *rewards, const float *noise, int64_t n_updates, int64_t critic_step, int64_t actor_step,
                   void *stream) {
    if (int rc = check_ma_cfg(cfg)) return rc;
    if (int rc = check_update("ma", stt, cstr_ma_workspace_bytes(cfg), obs, actions, next_obs, dones, rewards, n_updates, critic_step, actor_step)) return rc;
    MaWorkspace w = ma_carve(stt->workspace, cfg);
    w.sc.tensor = cfg->gemm_mode;
    const MaLayout T = ma_layout(cfg);
    cudaStream_t st = (cudaStream_t)stream;
    const int B = cfg->batch, H1 = cfg->h1, H2 = cfg->h2, ZC = cfg->n_critics, CI = T.critic.in;
    const int64_t cz = T.critic.size, az = T.actor.size;
    const int rb = w.n_row_blocks, tb = (B + 255) / 256;
    const bool policy_step = (n_updates % cfg->policy_delay) == 0;
    if (policy_step && actor_step < 1) return fail_arg(CSTR_EINVAL, "ma_update: actor_step must be >= 1 on a policy step");
    const float *dev_sc = stt->counters ? w.scalars : nullptr;
    if (stt->counters)  // one {step_size, bc2_sqrt} pair per optimiser: critic 0, actor 0 at scalars[0..3], critic 1, actor 1 at scalars[8..11]
        if (int rc = launch_tick(stt, w.scalars, policy_step, cfg->critic_lr[0], cfg->beta1, cfg->beta2, cfg->actor_lr[0], cfg->critic_lr[1], cfg->actor_lr[1], st))
            return rc;
    for (int i = 0; i < MA_AGENTS; ++i)
        if (!(cfg->actor_lr[i] >= 0.f) || !(cfg->critic_lr[i] >= 0.f)) return fail_arg(CSTR_EINVAL, "ma_update: learning rates must be >= 0");
    // critic input of agent i over (observations X, actions A): all of both (MADDPG) or the agent's own slices (IDDPG)
    auto critic_src = [&](int i, const float *X, const float *A) {
        Src s{};
        if (cfg->centralised) s.x0 = X, s.n0 = OBS, s.ld0 = OBS, s.x1 = A, s.n1 = ACT, s.ld1 = ACT;
        else s.x0 = X + i * MA_OBS, s.n0 = MA_OBS, s.ld0 = OBS, s.x1 = A + i * MA_ACT, s.n1 = MA_ACT, s.ld1 = ACT;
        return s;
    };

    // ---- target actions of every agent, once, from the actor targets as they are now (maddpg.py:132-144) ----
    {
        Src s{};
        s.x0 = next_obs, s.n0 = MA_OBS, s.ld0 = OBS, s.x0_z = MA_OBS;  // actor target z reads observation slice z
        const Net at = net_at(stt->targets, T.actor_off[0], T.actor);
        if (int rc = forward_mlp(B, T.actor, s, at, az, MA_AGENTS, w.a_h1, w.a_h2, w.a_y, true, w.sc, st)) return rc;
        launch_k(ma_next_action_kernel, tb, 256, 0, st, B, MA_AGENTS, (const float *)w.a_y, noise, cfg->target_policy_noise, cfg->target_noise_clip, cfg->seed,
                 (uint32_t)n_updates, dev_sc, w.next_act);
        if (int rc = check_launch("ma_next_action_kernel")) return rc;
    }
    for (int i = 0; i < MA_AGENTS; ++i) {
        const Net critic = net_at(stt->params, T.critic_off[i], T.critic), critic_t = net_at(stt->targets, T.critic_off[i], T.critic);
        const Net g_critic = net_at(stt->grads, T.critic_off[i], T.critic);
        // ---- target and critic step of agent i (:146-163) ----
        if (int rc = forward_hidden_g(B, T.critic, critic_src(i, next_obs, w.next_act), critic_t, cz, ZC, w.t_h1, w.t_h2, w.sc, st)) return rc;
        launch_k(td3_target_head_kernel, rb, 256, 0, st, B, H2, (const float *)w.t_h2, (int64_t)B * H2, (const float *)critic_t.w3, (const float *)critic_t.b3, cz, rewards,
                 dones, cfg->gamma, ZC, w.target);
        if (int rc = check_launch("td3_target_head_kernel<ma>")) return rc;
        const Src s_cur = critic_src(i, obs, actions);
        if (int rc = forward_hidden_g(B, T.critic, s_cur, critic, cz, ZC, w.h1, w.h2, w.sc, st)) return rc;
        if (int rc = critic_loss_backward(B, H1, H2, s_cur, critic, g_critic, cz, ZC, w.h1, w.h2, w.target, 2.f / (float)B, w.dq, w.dz2, w.dz1, w.loss_partial, w.sc, st))
            return rc;
        {
            ApplyArgs a = adam_args(stt, cfg->critic_lr[i], cfg->beta1, cfg->beta2, cfg->eps, cfg->tau, critic_step, dev_sc, i ? 8 : 0);
            a.adam_lo = T.critic_off[i], a.adam_hi = T.critic_off[i] + ZC * cz, a.polyak_lo = a.polyak_hi = 0;
            a.loss_partial = w.loss_partial, a.n_loss_partial = ZC * rb, a.loss_scale = 1.f / (float)B, a.loss_acc = stt->losses ? stt->losses + 4 * i : nullptr;
            if (int rc = launch_apply(a, stt->peer, stt->grads, st, "td3_apply_kernel<ma critic>")) return rc;
        }
        if (!policy_step) continue;
        // ---- actor step of agent i (:166-179): every actor evaluated on agent i's observation slice ----
        Src s_act{};
        s_act.x0 = obs + i * MA_OBS, s_act.n0 = MA_OBS, s_act.ld0 = OBS;  // x0_z = 0: the same slice for every actor
        const Net actors = net_at(stt->params, T.actor_off[0], T.actor);
        if (int rc = forward_mlp(B, T.actor, s_act, actors, az, MA_AGENTS, w.a_h1, w.a_h2, w.a_y, true, w.sc, st)) return rc;
        launch_k(ma_joint_kernel, tb, 256, 0, st, B, MA_AGENTS, (const float *)w.a_y, w.joint);
        if (int rc = check_launch("ma_joint_kernel")) return rc;
        const Src s_pi = critic_src(i, obs, w.joint);
        if (int rc = forward_hidden_g(B, T.critic, s_pi, critic, cz, 1, w.h1, w.h2, w.sc, st)) return rc;
        if (int rc = policy_critic_backward(B, H1, H2, critic, cz, w.h1, w.h2, w.dq, w.dz2, w.dz1, w.loss_partial, w.sc, st)) return rc;
        const int col = cfg->centralised ? OBS + i * MA_ACT : MA_OBS;  // where agent i's action sits in its critic's input
        launch_k(mlp_dx_kernel, rb, 256, 0, st, B, H1, CI, (const float *)w.dz1, (const float *)critic.w1, col, MA_ACT, w.da);
        if (int rc = check_launch("mlp_dx_kernel<ma action>")) return rc;
        launch_k(ma_actor_grad_kernel, tb, 256, 0, st, B, (const float *)w.da, (const float *)(w.a_y + (int64_t)i * B), w.a_dy);
        if (int rc = check_launch("ma_actor_grad_kernel")) return rc;
        const Net actor_i = net_at(stt->params, T.actor_off[i], T.actor), g_actor_i = net_at(stt->grads, T.actor_off[i], T.actor);
        if (int rc = backward_mlp(B, T.actor, s_act, nullptr, actor_i, g_actor_i, w.a_h1 + (int64_t)i * B * H1, w.a_h2 + (int64_t)i * B * H2, w.a_dy, w.a_dz2, w.a_dz1,
                                  w.sc, st))
            return rc;
        ApplyArgs a = adam_args(stt, cfg->actor_lr[i], cfg->beta1, cfg->beta2, cfg->eps, cfg->tau, actor_step, dev_sc, (i ? 8 : 0) + 2);
        a.adam_lo = T.actor_off[i], a.adam_hi = T.actor_off[i] + az, a.polyak_lo = 0, a.polyak_hi = T.total;  // polyak of ALL nets, inside the agent loop (:181-182)
        a.loss_partial = w.loss_partial, a.n_loss_partial = rb, a.loss_scale = -1.f / (float)B, a.loss_acc = stt->losses ? stt->losses + 4 * i + 2 : nullptr;
        if (int rc = launch_apply(a, stt->peer, stt->grads, st, "td3_apply_kernel<ma actor+polyak>")) return rc;
    }
    return 0;
}

}  // extern "C"
