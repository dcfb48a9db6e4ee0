// ppo_common.cuh -- what the two PPO minibatch steps share: the SIMT step of learner.cu (pime_ppo_step) and the tcgen05
// step of learner_tc.cu (pime_ppo_grad_tc -> pime_ppo_apply_grad -> pime_ppo_close_step) implement the same update, so
// theta's layout, the state block, the objectives and the Adam arithmetic are defined here once.
#pragma once

#include "pime_common.cuh"
#include "tc_mlp.cuh"

namespace pime {
namespace ppo {

// ------------------------------------------------------------------------------------------------ theta and the nets
struct Net {                  // one net of the step, as tc::make_pack_layout lays out its parameters
    int kind, S, H, So;       // So: inputs of the modular actor's other branch (S otherwise)
    int theta_off;            // first parameter of this net in theta
    int src[12];              // offsets of the state_dict tensors inside the net's parameters
};

// parameter count of the net, or -1 for dimensions make_pack_layout rejects
inline int fill_net(const pime_actor_config &c, int theta_off, Net &d) {
    tc::PackLayout L;
    if (!tc::make_pack_layout(c, L)) return -1;
    d.kind = c.kind; d.S = c.state_dim; d.H = c.mid_dim; d.theta_off = theta_off;
    d.So = c.kind == PIME_ACTOR_MODULAR ? c.state_dim - c.integrator_dim : c.state_dim;
    for (int j = 0; j < 12; ++j) d.src[j] = L.src[j];
    return L.param_count;
}

// theta = [actor parameters | pad | critic parameters | a_std_log]; the critic is CriticAdv with the actor's S and H and
// starts on a 16-byte boundary (learner.cu streams its hidden-layer matrices with cp.async.bulk).  n_theta counts all of it.
inline bool theta_layout(const pime_actor_config &actor, Net &act, Net &cri, int &n_theta) {
    const int pa = fill_net(actor, 0, act);
    if (pa < 0) return false;
    const pime_actor_config cc{PIME_CRITIC_ADV, actor.state_dim, actor.mid_dim, 0};
    const int pc = fill_net(cc, (pa + 3) & ~3, cri);
    if (pc < 0) return false;
    n_theta = cri.theta_off + pc + 1;
    return true;
}

// ------------------------------------------------------------------------------------------------ the state block
// pime_ppo_args::state (int32[1024], zero-initialised, owned by the library between steps).  The first three words and the
// output-layer accumulators belong to learner.cu's weight-gradient kernel, which resets them when it closes the step.
struct State {
    enum { kStep = 0, kTicket = 1, kAstd = 2, kAdamC = 8, kGOut = 16 };   // word offsets
    int *step;            // Adam steps taken so far (the step being taken is *step + 1)
    unsigned *ticket;     // weight-gradient CTAs of this step that have finished
    float *g_astd;        // accumulated gradient of a_std_log
    float *adam_c;        // [2]: lr / bias_correction1 and 1 / sqrt(bias_correction2) of the step being taken
    float *g_out;         // accumulated gradients of the two output layers Linear(H -> 1)

    State() = default;
    explicit State(int32_t *s)
        : step(s + kStep), ticket((unsigned *)(s + kTicket)), g_astd((float *)(s + kAstd)), adam_c((float *)(s + kAdamC)),
          g_out((float *)(s + kGOut)) {}
};

// The argument checks both steps need.  Each entry adds its own: theta_t, work and the Adam moments for pime_ppo_step,
// work_tc, grad and the supported shapes for pime_ppo_grad_tc.  No device is needed, so they run before require_device().
inline int validate_ppo_args(const pime_ppo_args *a) {
    PIME_REQUIRE(a && a->actor, "null ppo args / actor config");
    PIME_REQUIRE(a->theta && a->state, "null theta / state");
    PIME_REQUIRE(a->buf_state && a->buf_action && a->buf_r_sum && a->buf_logprob && a->buf_advantage && a->idx, "null replay tensor");
    PIME_REQUIRE(a->batch >= 2 && a->batch <= (1 << 20), "batch must be in [2, 2^20]");
    PIME_REQUIRE(a->loss_ring && a->ring_len >= 2, "loss ring");
    return PIME_OK;
}

// ------------------------------------------------------------------------------------------------ objectives (agent.py:635-652)
struct RowObj {
    float d_out;                        // d united / d (net output) of the row
    float o_act, o_cri, o_ent, g_asl;   // the row's share of obj_actor, obj_critic, obj_entropy and of d united / d a_std_log
};

// One minibatch row of the actor (net 0) or the critic (net 1): out = the net's output; action, r_sum, old logprob and
// advantage come from the replay; inv_cs = 1 / (r_sum.std() + 1e-5).  Rows past the batch (live false) contribute zeros.
__device__ __forceinline__ RowObj row_objectives(int net, float out, float action, float r_sum, float logprob, float adv,
                                                 float a_std_log, float inv_cs, float ratio_clip, float lambda_entropy,
                                                 float invB, bool live) {
    RowObj r{0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    if (net == 0) {
        const float std = expf(a_std_log);
        const float dd = (out - action) / std;
        const float lp = -(a_std_log + 0.9189385332046727f + dd * dd * 0.5f);   // compute_logprob (net_residual.py:62-66)
        const float ratio = expf(lp - logprob);
        const float s1 = adv * ratio;
        const float s2 = adv * fminf(fmaxf(ratio, 1.0f - ratio_clip), 1.0f + ratio_clip);
        const float sur = fminf(s1, s2);
        const float elp = expf(lp);
        const float ent = elp * lp;
        const float g_lp = (-(s1 <= s2 ? s1 : 0.0f) + lambda_entropy * (ent + elp)) * invB;   // d united / d new_logprob
        if (live) { r.d_out = g_lp * (-dd / std); r.o_act = (-sur + lambda_entropy * ent) * invB; r.o_ent = ent * invB; r.g_asl = g_lp * (dd * dd - 1.0f); }
    } else {
        const float e = out - r_sum;
        const float ae = fabsf(e);
        const float l1 = ae < 1.0f ? 0.5f * e * e : ae - 0.5f;                     // SmoothL1Loss, beta = 1
        if (live) { r.d_out = fminf(fmaxf(e, -1.0f), 1.0f) * invB * inv_cs; r.o_cri = l1 * invB; }
    }
    return r;
}

// ------------------------------------------------------------------------------------------------ Adam and the step count
// torch.optim.Adam (fused implementation's arithmetic): exp_avg = lerp(exp_avg, g, 1-b1); exp_avg_sq = b2 v + (1-b2) g^2;
// p -= (lr / bc1) * exp_avg / (sqrt(exp_avg_sq) / sqrt(bc2) + eps)
struct AdamCoef {
    float lr_bc1, inv_sqrt_bc2, one_m_b1, b2, one_m_b2, eps;
};
// the two step-dependent coefficients (double-precision pow), computed once per step by one thread into adam_c
__device__ __forceinline__ void adam_prepare(const int *step, float lr, float beta1, float beta2, float *adam_c) {
    const int t = *step + 1;
    const double bc1 = 1.0 - pow((double)beta1, (double)t), bc2 = 1.0 - pow((double)beta2, (double)t);
    adam_c[0] = (float)((double)lr / bc1);
    adam_c[1] = (float)(1.0 / sqrt(bc2));
}
__device__ __forceinline__ AdamCoef adam_coef(const float *adam_c, float beta1, float beta2, float eps) {
    AdamCoef c;
    c.lr_bc1 = adam_c[0];
    c.inv_sqrt_bc2 = adam_c[1];
    c.one_m_b1 = 1.0f - beta1; c.b2 = beta2; c.one_m_b2 = 1.0f - beta2; c.eps = eps;
    return c;
}
// every operation is spelled out (no compiler-chosen FMA contraction): the fused weight-gradient epilogue and the
// stand-alone Adam kernel of the data-parallel and tensor-core paths must produce bit-identical parameters and moments
__device__ __forceinline__ float adam_update(const AdamCoef &c, float g, float theta, float &m, float &v) {
    m = __fmaf_rn(c.one_m_b1, __fsub_rn(g, m), m);                              // lerp(exp_avg, grad, 1 - beta1)
    v = __fmaf_rn(__fmul_rn(c.one_m_b2, g), g, __fmul_rn(c.b2, v));             // beta2 v + (1 - beta2) g g
    const float den = __fmaf_rn(sqrtf(v), c.inv_sqrt_bc2, c.eps);
    return __fsub_rn(theta, __fdiv_rn(__fmul_rn(c.lr_bc1, m), den));
}

// the end of a step: clear the loss-ring row of the next step, then count this one
__device__ __forceinline__ void close_step(int *step, float *loss_ring, int ring_len) {
    const int t = *step + 1;
    float *nxt = loss_ring + (size_t)(t % ring_len) * 4;
    nxt[0] = nxt[1] = nxt[2] = nxt[3] = 0.0f;
    *step = t;
}

}  // namespace ppo
}  // namespace pime
