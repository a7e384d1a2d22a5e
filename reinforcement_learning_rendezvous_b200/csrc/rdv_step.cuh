// rdv_step.cuh -- one RendezvousEnv.step (rendezvous_env.py:160-221) on register-resident state, as the
// building blocks shared by the thread-per-env step kernel and the fused multi-step rollout kernel:
//   ingest_action_*  :168-173, :201-202, :333   action -> impulses, fuel term, delta-v / delta-w totals
//   env_advance      :172-184                   CW translation + both attitude propagations
//   env_evaluate     :186-211                   latch, time, bubble, observation, done, reward
#pragma once
#include "rdv_env.cuh"

namespace rdv {

__constant__ double c_zero3[3] = {0.0, 0.0, 0.0};     // the target carries no torque (rendezvous_env.py:585)

// Per-env quantities that live next to the 20 state numbers.
struct EnvCounters {
    double tdv, tdw, ep_ret;          // total_delta_v, total_delta_w, running episode return
    int step, success, collided, episode;
};

struct ActionTerms { double dvb[3], dw[3], fuel; };

RDV_DEV void ingest_action_f64(const RdvParams &P, const double (&a)[6], EnvCounters &c, ActionTerms &t)
{
    t.dvb[0] = a[0] * P.max_delta_v; t.dvb[1] = a[1] * P.max_delta_v; t.dvb[2] = a[2] * P.max_delta_v;
    t.dw[0] = a[3] * P.max_delta_w; t.dw[1] = a[4] * P.max_delta_w; t.dw[2] = a[5] * P.max_delta_w;
    const double sv = fabs(a[0]) + fabs(a[1]) + fabs(a[2]);
    const double sw = fabs(a[3]) + fabs(a[4]) + fabs(a[5]);
    c.tdv += sv * P.max_delta_v;
    c.tdw += sw * P.max_delta_w;
    t.fuel = P.fuel_scale * sv;
}

// float32 actions follow NumPy-2 promotion (SURVEY.md 8a row a2): delta_v, total_delta_v and the fuel term are
// rounded in fp32; delta_w and total_delta_w are fp64.
RDV_DEV void ingest_action_f32(const RdvParams &P, const float (&a)[6], EnvCounters &c, ActionTerms &t)
{
    t.dvb[0] = (double)__fmul_rn(a[0], P.max_delta_v_f32);
    t.dvb[1] = (double)__fmul_rn(a[1], P.max_delta_v_f32);
    t.dvb[2] = (double)__fmul_rn(a[2], P.max_delta_v_f32);
    t.dw[0] = (double)a[3] * P.max_delta_w; t.dw[1] = (double)a[4] * P.max_delta_w; t.dw[2] = (double)a[5] * P.max_delta_w;
    const float sv = __fadd_rn(__fadd_rn(fabsf(a[0]), fabsf(a[1])), fabsf(a[2]));
    const float sw = __fadd_rn(__fadd_rn(fabsf(a[3]), fabsf(a[4])), fabsf(a[5]));
    c.tdv = (double)__fadd_rn((float)c.tdv, __fmul_rn(sv, P.max_delta_v_f32));
    c.tdw += (double)sw * P.max_delta_w;
    t.fuel = (double)__fdiv_rn(__fmul_rn(P.fuel_num_f32, sv), P.fuel_den_f32);
}

// Translation (impulse rotated by the OLD chaser attitude, then the CW transition; dynamics.py:24-55) and the
// two attitude propagations (:552-604).  LOCKSTEP: the two isotropic solves advance interleaved stage by stage
// (rk45_iso_plane_pair, 2x ILP) -- the right choice with <= 2 warps per SM sub-partition; otherwise one solve after
// the other through a single copy of the solver (rk45_iso_plane, 128 registers), which wins once 3-4 warps per
// sub-partition hide the latency instead.  This still holds with the closed-form attempt: the pair fits 128 registers
// at 448 and 512 threads and is 4-16 % slower there (DESIGN 4.3, profiles/r08_lockstep_timing.txt).
// first half of env_advance: the impulse rotated by the OLD chaser attitude, then the CW transition
RDV_DEV void env_translate(const RdvParams &P, EnvRegs &e, const ActionTerms &t)
{
    double dv[3];
    const Rot Rc_old = rot_from_quat(e.qc);
    rot_apply(Rc_old, t.dvb, dv);
    const double r0 = e.rc[0], r1 = e.rc[1], r2 = e.rc[2];
    const double v0 = e.vc[0] + dv[0], v1 = e.vc[1] + dv[1], v2 = e.vc[2] + dv[2];
    const double *c = P.cw;
    e.rc[0] = fma(c[2], v1, fma(c[1], v0, c[0] * r0));
    e.rc[1] = fma(c[6], v1, fma(c[5], v0, fma(c[3], r0, c[4] * r1)));
    e.rc[2] = fma(c[8], v2, c[7] * r2);
    e.vc[0] = fma(c[11], v1, fma(c[10], v0, c[9] * r0));
    e.vc[1] = fma(c[14], v1, fma(c[13], v0, c[12] * r0));
    e.vc[2] = fma(c[16], v2, c[15] * r2);
}

// second half: the two attitude propagations (rendezvous_env.py:180-184, :552-604)
template <bool ISO, bool CLOSED, bool LOCKSTEP>
RDV_DEV void env_attitude(const RdvParams &P, EnvRegs &e, const ActionTerms &t, int &rk_acc, int &rk_rej, int &fail)
{
    double y[7] = {e.qc[0], e.qc[1], e.qc[2], e.qc[3], e.wc[0] + t.dw[0], e.wc[1] + t.dw[1], e.wc[2] + t.dw[2]};
    double z[7] = {e.qt[0], e.qt[1], e.qt[2], e.qt[3], e.wt[0], e.wt[1], e.wt[2]};
    if (CLOSED) {
        closed_form_attitude(y, P.dt);
        closed_form_attitude(z, P.dt);
    } else {
        BodyConst bc, bt;
        bc.I = P.inertia_c; bc.Iinv = P.inv_inertia_c; bc.tau = P.torque_c;
        bt.I = P.inertia_t; bt.Iinv = P.inv_inertia_t; bt.tau = c_zero3;
        if (ISO && LOCKSTEP) {
            const int k = rk45_iso_plane_pair(y, z, P.dt, rk_rej);
            if (k < 0) { fail = 1; rk_acc += -1 - k; } else rk_acc += k;
        } else if (ISO) {
            // one solve after the other through a single copy of the solver code (bounded registers)
#pragma unroll 1
            for (int body = 0; body < 2; ++body) {
                const int k = rk45_iso_plane(y, P.dt, rk_rej);
                if (k < 0) fail = 1; else rk_acc += k;
#pragma unroll
                for (int j = 0; j < 7; ++j) { const double tmp = y[j]; y[j] = z[j]; z[j] = tmp; }
            }
        } else {
            const int kc = rk45_attitude<false>(y, P.dt, bc, rk_rej);
            const int kt = rk45_attitude<false>(z, P.dt, bt, rk_rej);
            if (kc < 0) fail = 1; else rk_acc += kc;
            if (kt < 0) fail = 1; else rk_acc += kt;
        }
    }
    const double ry = fast_rsqrt(dot4(y, y)), rz = fast_rsqrt(dot4(z, z));       // q / |q|  (:574-575, :601-602)
#pragma unroll
    for (int k = 0; k < 4; ++k) { e.qc[k] = y[k] * ry; e.qt[k] = z[k] * rz; }
#pragma unroll
    for (int k = 0; k < 3; ++k) { e.wc[k] = y[4 + k]; e.wt[k] = z[4 + k]; }
}

template <bool ISO, bool CLOSED, bool LOCKSTEP>
RDV_DEV void env_advance(const RdvParams &P, EnvRegs &e, const ActionTerms &t, int &rk_acc, int &rk_rej, int &fail)
{
    env_translate(P, e, t);
    env_attitude<ISO, CLOSED, LOCKSTEP>(P, e, t, rk_acc, rk_rej, fail);
}

struct StepResult { double rew; int done, reason; };

// gym 0.21 Box.contains on the float32 observation (rendezvous_env.py:367) WITHOUT forming the observation: a double
// x rounds to a float in [-1, 1] iff |x| <= 1 + 2^-24.  Fast path on the high words of the raw state: a scaled entry
// with |x| < hi (1 - 1e-6) maps to |o| < 1 whatever the rounding of normalize_value, and a quaternion component with
// |q| < 1 is in the box; P.box_hi_* are the high words of those thresholds (rdv_params_derive).  Everything else --
// a component at exactly +-1, a state near the edge of the box, NaN -- takes the exact path through make_obs.
RDV_DEV bool obs_in_box_state(const RdvParams &P, const EnvRegs &e)
{
    auto hi = [](double x) { return __double2hiint(x) & 0x7fffffff; };
    const int mr = max(max(hi(e.rc[0]), hi(e.rc[1])), hi(e.rc[2]));
    const int mv = max(max(hi(e.vc[0]), hi(e.vc[1])), hi(e.vc[2]));
    const int mw = max(max(hi(e.wc[0]), hi(e.wc[1])), hi(e.wc[2]));
    const int mq = max(max(max(hi(e.qc[0]), hi(e.qc[1])), max(hi(e.qc[2]), hi(e.qc[3]))),
                       max(max(hi(e.qt[0]), hi(e.qt[1])), max(hi(e.qt[2]), hi(e.qt[3]))));
    if (mr < P.box_hi_r && mv < P.box_hi_v && mw < P.box_hi_w && mq < 0x3FF00000) return true;
    float ov[RDV_OBS_DIM];
    make_obs(e, obs_scale(P), ov);
    return obs_in_box(ov);
}

// What an evaluator reads after a step (monte_carlo.py:140-152): get_errors, check_collision, dist_from_koz.
struct EvalDetail { double err[4]; double koz; bool col_now, within; };

// Everything after the propagation: collision / success latch (:186-190), time and bubble (:193-198),
// observation (:205), done + end reason (:355-386), reward (:313-353).  Updates the counters.
// WANT_OBS: form the float32 observation (the policy's input, a per-step record); otherwise only its Box test.
// DETAIL: also return the evaluator quantities -- this disables the far-from-the-target shortcut below.
template <bool WANT_OBS = true, bool DETAIL = false>
RDV_DEV StepResult env_evaluate(const RdvParams &P, const EnvRegs &e, const double fuel, EnvCounters &c,
                                float (&ov)[RDV_OBS_DIM], EvalDetail *detail = nullptr)
{
    const double rc_sq = dot3(e.rc, e.rc);
    // the chaser's quaternion was normalised by env_attitude a moment ago: quat2mat's re-normalisation (a factor
    // within 1 ulp of 1) is skipped outside the evaluator's own form (measured: 9.74 -> 9.70 us per step in 20-step
    // launches, 8.90 -> 8.87 in 250-step ones)
    const Rot Rc = DETAIL ? rot_from_quat(e.qc) : rot_from_unit_quat(e.qc);
    const double att = attitude_error(P, e, Rc, rc_sq);
    // The target-relative quantities (corridor angle, position / velocity / rate errors) only matter near the
    // target: a collision needs |rc| < koz, and success (:406-422) or the reward bonus (:348-351) need a position
    // error <= max_rd_error, impossible unless | |rc| - |rd| | <= max_rd_error (|R(qt) rd| = |rd|).  Far away
    // -- every step of a random-action episode -- the target rotation matrix is never formed.
    bool col_now = false;
    ErrSq es;
    es.pos = es.vel = es.rot = 1.0e300;
    if (DETAIL || rc_sq < P.near_sq) {
        const Rot Rt = rot_from_quat(e.qt);
        if (DETAIL) {
            // the evaluator's own forms (errors_kernel): IEEE square roots, the corridor angle at any distance
            const double rc_n = sqrt(rc_sq), th = corridor_angle(P, e, Rt, rc_sq);
            col_now = rc_n < P.koz_radius && th > P.corridor_half_angle;
            es = errors_sq(P, e, Rc, Rt);
            detail->err[0] = sqrt(es.pos); detail->err[1] = sqrt(es.vel); detail->err[2] = att; detail->err[3] = sqrt(es.rot);
            detail->koz = koz_distance(P, rc_n, th);
            detail->col_now = col_now;
            detail->within = detail->err[0] <= P.max_rd_error && detail->err[1] <= P.max_vd_error &&
                             att <= P.max_qd_error && detail->err[3] <= P.max_wd_error;
        } else {
            col_now = rc_sq < P.koz_radius_sq && corridor_angle(P, e, Rt, rc_sq) > P.corridor_half_angle;
            es = errors_sq(P, e, Rc, Rt);
        }
    }
    if (!c.collided) {
        c.collided = col_now ? 1 : 0;
        if (!c.collided && es.pos <= P.max_rd_error_sq && es.vel <= P.max_vd_error_sq && att <= P.max_qd_error &&
            es.rot <= P.max_wd_error_sq)
            c.success += 1;
    }
    c.step += 1;
    const double bubble = fmax(fma(-(double)c.step, P.bubble_rate, P.bubble0), P.bubble_min);
    bool in_box;
    if (WANT_OBS) {
        make_obs(e, obs_scale(P), ov);
        in_box = obs_in_box(ov);
    } else {
        in_box = obs_in_box_state(P, e);
    }
    const bool c0 = !in_box, c1 = c.step >= P.done_steps, c2 = rc_sq > bubble * bubble,
               c3 = att > P.max_attitude_error;
    StepResult r;
    r.done = (c0 || c1 || c2 || c3) ? 1 : 0;
    r.reason = c0 ? 0 : c1 ? 1 : c2 ? 2 : c3 ? 3 : -1;
    double rew = P.att_scale * fma(-att, P.inv_max_attitude_error, 1.0);
    rew += fuel;
    if (col_now) rew -= P.collision_scale;
    if (rc_sq < P.koz_radius_sq && !c.collided && es.pos < P.max_rd_error_sq) {
        rew += P.bonus_scale * fma(-fast_sqrt(es.pos), P.inv_max_rd_error, 2.0);
        if (att < P.max_qd_error) rew += P.bonus_scale * fma(-att, P.inv_max_qd_error, 2.0);
    }
    r.rew = rew;
    c.ep_ret += rew;
    return r;
}

// Per-episode accumulators of monte_carlo.evaluate (monte_carlo.py:94-207), one sample per visited state.
// Terminal errors (:159-189): the constraint sets are nested (all four < limits  =>  pos, vel and att-or-rot  =>
// pos and vel  =>  pos), so "mean of the errors from the first index at which the most constraints are met" needs
// ONE running sum: restart it whenever a sample reaches a better level than any before, keep adding otherwise;
// with no level reached at all it holds the last sample only (index = -1).
struct McAcc {
    double sum[4], min_koz, total_reward;
    int count, level, n_col, n_suc, len;
};
RDV_DEV void mc_init(McAcc &m)
{
    m.sum[0] = m.sum[1] = m.sum[2] = m.sum[3] = 0.0;
    m.min_koz = 1.0e300; m.total_reward = 0.0;
    m.count = 0; m.level = 4; m.n_col = m.n_suc = m.len = 0;
}
RDV_DEV void mc_sample(const RdvParams &P, const EvalDetail &d, const int sticky_collided, McAcc &m)
{
    m.n_col += d.col_now ? 1 : 0;                                         // :121, :143
    if (!sticky_collided) m.n_suc += d.within ? 1 : 0;                    // :122-123, :144-145
    if (d.koz < m.min_koz) m.min_koz = d.koz;                             // :124, :146-148
    const bool pm = d.err[0] < P.max_rd_error, vm = d.err[1] < P.max_vd_error, am = d.err[2] < P.max_qd_error,
               rm = d.err[3] < P.max_wd_error;                            // strict, :166-169
    const int level = !pm ? 4 : !vm ? 3 : !(am || rm) ? 2 : !(am && rm) ? 1 : 0;
    if (level < m.level || m.level == 4) {
        m.level = level;
#pragma unroll
        for (int j = 0; j < 4; ++j) m.sum[j] = d.err[j];
        m.count = 1;
    } else {
#pragma unroll
        for (int j = 0; j < 4; ++j) m.sum[j] += d.err[j];
        m.count += 1;
    }
}
// the evaluator quantities of the CURRENT state without a step (sample 0, monte_carlo.py:117-124)
RDV_DEV void eval_detail_of_state(const RdvParams &P, const EnvRegs &e, EvalDetail &d)
{
    const Rot Rc = rot_from_quat(e.qc), Rt = rot_from_quat(e.qt);
    const double rc_sq = dot3(e.rc, e.rc), rc_n = sqrt(rc_sq);
    const double att = attitude_error(P, e, Rc, rc_sq), th = corridor_angle(P, e, Rt, rc_sq);
    const ErrSq es = errors_sq(P, e, Rc, Rt);
    d.err[0] = sqrt(es.pos); d.err[1] = sqrt(es.vel); d.err[2] = att; d.err[3] = sqrt(es.rot);
    d.koz = koz_distance(P, rc_n, th);
    d.col_now = rc_n < P.koz_radius && th > P.corridor_half_angle;
    d.within = d.err[0] <= P.max_rd_error && d.err[1] <= P.max_vd_error && att <= P.max_qd_error &&
               d.err[3] <= P.max_wd_error;
}

// one row of the trajectory record (rdv_rollout_trajectory): `row` points at column 0 of this env, columns are n apart
RDV_DEV void store_traj_row(double *row, const int64_t n, const EnvRegs &e, const EnvCounters &c, const EvalDetail &d)
{
#pragma unroll
    for (int k = 0; k < 3; ++k) { row[(RDV_RCX + k) * n] = e.rc[k]; row[(RDV_VCX + k) * n] = e.vc[k]; }
#pragma unroll
    for (int k = 0; k < 4; ++k) { row[(RDV_QCW + k) * n] = e.qc[k]; row[(RDV_QTW + k) * n] = e.qt[k]; }
#pragma unroll
    for (int k = 0; k < 3; ++k) { row[(RDV_WCX + k) * n] = e.wc[k]; row[(RDV_WTX + k) * n] = e.wt[k]; }
    row[RDV_TDV * n] = c.tdv; row[RDV_TDW * n] = c.tdw; row[RDV_EPRET * n] = c.ep_ret;
    row[RDV_TR_I_STEP * n] = (double)c.step; row[RDV_TR_I_SUCCESS * n] = (double)c.success;
    row[RDV_TR_I_COLLIDED * n] = (double)c.collided; row[RDV_TR_I_EPISODE * n] = (double)c.episode;
#pragma unroll
    for (int k = 0; k < 4; ++k) row[(RDV_TR_POS_ERR + k) * n] = d.err[k];
    row[RDV_TR_KOZ * n] = d.koz;
    row[RDV_TR_COLLISION * n] = d.col_now ? 1.0 : 0.0;
    row[RDV_TR_SUCCESS * n] = (!c.collided && d.within) ? 1.0 : 0.0;       // check_success with the sticky flag
}

RDV_DEV void load_counters(const RdvState &S, int64_t i, EnvCounters &c)
{
    const int64_t ld = S.ld;
    c.tdv = S.f64[RDV_TDV * ld + i]; c.tdw = S.f64[RDV_TDW * ld + i]; c.ep_ret = S.f64[RDV_EPRET * ld + i];
    c.step = S.i32[RDV_I_STEP * ld + i]; c.success = S.i32[RDV_I_SUCCESS * ld + i];
    c.collided = S.i32[RDV_I_COLLIDED * ld + i]; c.episode = S.i32[RDV_I_EPISODE * ld + i];
}
RDV_DEV void store_counters(const RdvState &S, int64_t i, const EnvCounters &c)
{
    const int64_t ld = S.ld;
    S.f64[RDV_TDV * ld + i] = c.tdv; S.f64[RDV_TDW * ld + i] = c.tdw; S.f64[RDV_EPRET * ld + i] = c.ep_ret;
    S.i32[RDV_I_STEP * ld + i] = c.step; S.i32[RDV_I_SUCCESS * ld + i] = c.success;
    S.i32[RDV_I_COLLIDED * ld + i] = c.collided; S.i32[RDV_I_EPISODE * ld + i] = c.episode;
}

// U(-1,1) fp64 actions from the Philox stream (action_seed; env id, step index): blocks 0x40000000 | {0,1} of the
// counter space, disjoint from the reset() draws (blocks 0..11 keyed by the episode index).  Six of the eight 32-bit
// words of the two blocks become a_j = (w_j + 0.5) 2^-31 - 1: uniform on a symmetric 2^-31 grid inside (-1, 1) --
// finer than the float32 actions gym's Box.sample() or an SB3 policy produce -- at two Philox blocks, six
// conversions and six DFMA per env-step (the 53-bit form took three blocks and 42 instructions for the conversions).
RDV_DEV void philox_actions(uint64_t action_seed, int64_t env_id, int64_t step_index, double (&a)[6])
{
    uint32_t w[8];
#pragma unroll
    for (uint32_t blk = 0; blk < 2; ++blk) {
        uint32_t c[4] = {(uint32_t)env_id, (uint32_t)((uint64_t)env_id >> 32), (uint32_t)step_index,
                         0x40000000u | blk | (((uint32_t)((uint64_t)step_index >> 32) & 0x00FFFFFFu) << 4)};
        philox4x32_10(c, (uint32_t)action_seed, (uint32_t)(action_seed >> 32));
#pragma unroll
        for (int j = 0; j < 4; ++j) w[4 * blk + j] = c[j];
    }
#pragma unroll
    for (int j = 0; j < 6; ++j) a[j] = fma((double)w[j], 4.656612873077392578125e-10, -1.0 + 2.3283064365386962890625e-10);
}

}  // namespace rdv
