// rdv_b200.cu -- kernels and C ABI of librdv_b200.so (sm_100a only).
//
// Layout in HBM: structure-of-arrays fp64 state [RDV_NF64][ld] + int32 [RDV_NI32][ld], so a warp's access to one
// row is one coalesced 256 B line.  Row-major [n][6] actions are read with 8/16-byte loads; the [n][17] float32
// observation is staged in shared memory and written out as contiguous rows.  Per-configuration constants (CW
// transition matrix, thresholds, reward coefficients, inertia) travel in the __grid_constant__ RdvParams kernel
// argument, i.e. the constant bank.
//
// Kernels (DESIGN.md section 4):
//   step_kernel     rdv_step     one launch per step, two lanes per env, team-of-8 auto-reset fused in
//   rollout_kernel  rdv_rollout  K steps per launch, state in registers, one CTA per SM, prefetched in-warp
//                                resets, actions from a tensor / Philox / the actor on the tensor cores (tcgen05);
//                                rdv_rollout_trajectory: the same launch, recording every env's fp64 state each step
//   reset_kernel, observe_kernel, errors_kernel, frame_kernel, policy_kernel, fp64_peak_kernel
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>
#include <stdlib.h>
#include <atomic>
#include <mutex>
#include <type_traits>
#include "rdv_step.cuh"
#include "rdv_policy.cuh"
#include "rdv_policy_tc.cuh"

namespace rdv {


// ---------------------------------------------------------------------------------
// warp / block reduction of the statistics vector
// ---------------------------------------------------------------------------------
RDV_DEV double warp_sum(double v)
{
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

struct StepStats {
    // per-thread contributions; integers go through REDUX (__reduce_add_sync), doubles through shuffles
    unsigned steps, episodes, succeeded, collided, end0, end1, end2, end3, rk_acc, rk_rej, fail;
    double ep_return, ep_length, delta_v, delta_w, reward;
};

template <int NWARPS>
RDV_DEV void reduce_stats(const StepStats &st, double *g_stats, double (*s_stats)[RDV_NSTATS])
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double v[RDV_NSTATS];
    v[RDV_S_STEPS] = (double)__reduce_add_sync(full, st.steps);
    v[RDV_S_EPISODES] = (double)__reduce_add_sync(full, st.episodes);
    v[RDV_S_RK_ACCEPTED] = (double)__reduce_add_sync(full, st.rk_acc);
    v[RDV_S_RK_REJECTED] = (double)__reduce_add_sync(full, st.rk_rej);
    v[RDV_S_FAILURES] = (double)__reduce_add_sync(full, st.fail);
    v[RDV_S_REWARD] = warp_sum(st.reward);
    const bool any_done = v[RDV_S_EPISODES] > 0.0;       // warp-uniform
    if (any_done) {
        v[RDV_S_SUCCEEDED] = (double)__reduce_add_sync(full, st.succeeded);
        v[RDV_S_COLLIDED] = (double)__reduce_add_sync(full, st.collided);
#pragma unroll
        for (int k = 0; k < 4; ++k) v[RDV_S_END_OBS + k] = (double)__reduce_add_sync(full, (k==0?st.end0:k==1?st.end1:k==2?st.end2:st.end3));
        v[RDV_S_RETURN] = warp_sum(st.ep_return);
        v[RDV_S_LENGTH] = warp_sum(st.ep_length);
        v[RDV_S_DELTA_V] = warp_sum(st.delta_v);
        v[RDV_S_DELTA_W] = warp_sum(st.delta_w);
    } else {
        v[RDV_S_SUCCEEDED] = v[RDV_S_COLLIDED] = v[RDV_S_RETURN] = v[RDV_S_LENGTH] = 0.0;
        v[RDV_S_DELTA_V] = v[RDV_S_DELTA_W] = 0.0;
#pragma unroll
        for (int k = 0; k < 4; ++k) v[RDV_S_END_OBS + k] = 0.0;
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < RDV_NSTATS; ++k) s_stats[warp][k] = v[k];
    }
    __syncthreads();
    if (threadIdx.x < RDV_NSTATS) {
        double acc = 0.0;
#pragma unroll
        for (int w = 0; w < NWARPS; ++w) acc += s_stats[w][threadIdx.x];
        if (acc != 0.0) atomicAdd(g_stats + threadIdx.x, acc);
    }
}

// The constants of env `env`: the call's RdvParams (constant bank), or -- per-env parameter batches -- the table entry
// of the env's block of 32.  All lanes of a warp address envs of one block, so the loads are warp-uniform.
template <bool TABLE>
RDV_DEV const RdvParams &params_of(const RdvParams &Pc, const RdvState &S, const int64_t env)
{
    if constexpr (TABLE) return S.param_table[S.param_block[env >> 5]];
    else return Pc;
}

RDV_DEV double pair_swap(double v) { return __shfl_xor_sync(0xffffffffu, v, 1); }
RDV_DEV int pair_swap(int v) { return __shfl_xor_sync(0xffffffffu, v, 1); }

// ---------------------------------------------------------------------------------
// step kernel: RendezvousEnv.step (rendezvous_env.py:160-221).
//
// TWO threads per environment, adjacent lanes of one warp:
//   lane 2e   ("chaser lane"): chaser attitude propagation, attitude error, time / bubble / done /
//                              reward assembly, counters, statistics;
//   lane 2e+1 ("target lane"): target attitude propagation, the chaser's translation (impulse + CW
//                              transition), corridor angle / collision, position / velocity / rate errors.
// The two adaptive RK45 solves -- 88 % of the reference's step time -- run concurrently, which halves the
// serial length of a thread, halves its live state (~120 registers instead of 244, so 16 warps per SM are
// resident instead of 8) and doubles the number of warps the fp64 pipe can pick from.  The lanes trade
// ~20 doubles per step through warp shuffles.  Finished envs are appended to reset_list (count in
// reset_list[0]) for the compacted reset kernel below, so the rare reset path never diverges a stepping warp.
// ---------------------------------------------------------------------------------
constexpr int STEP_MIN_CTAS = 4;    // 4 CTAs x 4 warps = 16 resident warps per SM at <= 128 registers
constexpr int EPB = 64;             // environments per CTA
constexpr int TPB = 2 * EPB;        // threads per CTA

template <bool ISO, bool ACT_F64, bool CLOSED, bool TABLE = false>
__global__ void __launch_bounds__(TPB, STEP_MIN_CTAS) step_kernel(const __grid_constant__ RdvParams Pc, const RdvState S,
                                                      const RdvStepIO io, const int64_t n, const uint64_t seed,
                                                      const int64_t env_offset)
{
    __shared__ __align__(16) float s_obs[EPB * RDV_OBS_DIM];
    __shared__ double s_stats[TPB / 32][RDV_NSTATS];
    __shared__ double s_team[TPB / RDV_TEAM][RDV_TEAM_ROW];   // scratch rows of the reset teams
    __shared__ int s_reset_idx[EPB];                          // envs of this CTA whose episode just ended
    __shared__ int s_reset_n, s_fin_base;
    __shared__ double s_fin_rec[EPB][RDV_EP_NCOL];            // episode records of the finished envs (compacted rows)
    __shared__ int s_fin_reason[EPB];
    if (threadIdx.x == 0) s_reset_n = 0;
    __syncthreads();

    const int body = threadIdx.x & 1;                         // 0: chaser lane, 1: target lane
    const int64_t base = (int64_t)blockIdx.x * EPB;
    const int64_t i_raw = base + (threadIdx.x >> 1);
    const bool active = i_raw < n;
    const int64_t i = active ? i_raw : n - 1;                 // idle pairs shadow the last env (no stores)
    const int64_t ld = S.ld;
    const double *f = S.f64 + i;
    StepStats st = {};
    const RdvParams &P = params_of<TABLE>(Pc, S, i);

    // ---- own body: attitude quaternion and body rate ----
    const int qrow = body ? RDV_QTW : RDV_QCW, wrow = body ? RDV_WTX : RDV_WCX;
    double y[7];
#pragma unroll
    for (int k = 0; k < 4; ++k) y[k] = f[(qrow + k) * ld];
#pragma unroll
    for (int k = 0; k < 3; ++k) y[4 + k] = f[(wrow + k) * ld];

    // ---- action ingest (:168-173, :201-202, :333): the target lane takes a[0:3] (delta-v), the chaser
    //      lane a[3:6] (delta-w); `total` is total_delta_v on the target lane, total_delta_w on the chaser lane
    double act[3], total = f[(body ? RDV_TDV : RDV_TDW) * ld], fuel = 0.0;
    if (ACT_F64) {
        const double *ap = static_cast<const double *>(io.actions) + 6 * i + (body ? 0 : 3);
        const double a0 = ap[0], a1 = ap[1], a2 = ap[2];
        const double scale = body ? P.max_delta_v : P.max_delta_w;
        const double sum = fabs(a0) + fabs(a1) + fabs(a2);
        act[0] = a0 * scale; act[1] = a1 * scale; act[2] = a2 * scale;
        total += sum * scale;
        fuel = P.fuel_scale * sum;
    } else {
        // float32 actions follow NumPy-2 promotion (SURVEY.md 8a row a2): delta_v, total_delta_v and the
        // fuel term are rounded in fp32; delta_w and total_delta_w are fp64.
        const float *ap = static_cast<const float *>(io.actions) + 6 * i + (body ? 0 : 3);
        const float a0 = ap[0], a1 = ap[1], a2 = ap[2];
        const float sum = __fadd_rn(__fadd_rn(fabsf(a0), fabsf(a1)), fabsf(a2));
        if (body) {
            act[0] = (double)__fmul_rn(a0, P.max_delta_v_f32);
            act[1] = (double)__fmul_rn(a1, P.max_delta_v_f32);
            act[2] = (double)__fmul_rn(a2, P.max_delta_v_f32);
            total = (double)__fadd_rn((float)total, __fmul_rn(sum, P.max_delta_v_f32));
            fuel = (double)__fdiv_rn(__fmul_rn(P.fuel_num_f32, sum), P.fuel_den_f32);
        } else {
            act[0] = (double)a0 * P.max_delta_w; act[1] = (double)a1 * P.max_delta_w;
            act[2] = (double)a2 * P.max_delta_w;
            total += (double)sum * P.max_delta_w;
        }
    }

    // ---- translation on the target lane: impulse rotated by the chaser's OLD attitude, then the CW
    //      transition (:172-177, dynamics.py:24-55).  The chaser lane applies its rate impulse (:180).
    double qo[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) qo[k] = pair_swap(y[k]);      // target lane receives qc_old
    double rc[3] = {0.0, 0.0, 0.0}, vc[3] = {0.0, 0.0, 0.0};
    if (body) {
        const Rot Rc_old = rot_from_quat(qo);
        double dv[3];
        rot_apply(Rc_old, act, dv);
        const double r0 = f[RDV_RCX * ld], r1 = f[RDV_RCY * ld], r2 = f[RDV_RCZ * ld];
        const double v0 = f[RDV_VCX * ld] + dv[0], v1 = f[RDV_VCY * ld] + dv[1], v2 = f[RDV_VCZ * ld] + dv[2];
        const double *c = P.cw;
        rc[0] = fma(c[2], v1, fma(c[1], v0, c[0] * r0));
        rc[1] = fma(c[6], v1, fma(c[5], v0, fma(c[3], r0, c[4] * r1)));
        rc[2] = fma(c[8], v2, c[7] * r2);
        vc[0] = fma(c[11], v1, fma(c[10], v0, c[9] * r0));
        vc[1] = fma(c[14], v1, fma(c[13], v0, c[12] * r0));
        vc[2] = fma(c[16], v2, c[15] * r2);
    } else {
        y[4] += act[0]; y[5] += act[1]; y[6] += act[2];
    }

    // ---- attitude: torque-free propagation of this lane's body over dt (:180-184, :552-604) ----
    int rk_acc = 0, rk_rej = 0, fail = 0;
    if (CLOSED) {
        closed_form_attitude(y, P.dt);
    } else {
        BodyConst bc;
        bc.I = body ? P.inertia_t : P.inertia_c;
        bc.Iinv = body ? P.inv_inertia_t : P.inv_inertia_c;
        bc.tau = body ? c_zero3 : P.torque_c;
        const int k = ISO ? rk45_iso_plane(y, P.dt, rk_rej) : rk45_attitude<ISO>(y, P.dt, bc, rk_rej);
        if (k < 0) fail = 1; else rk_acc = k;
    }
    {
        const double r = fast_rsqrt(dot4(y, y));               // q / |q|  (:574-575, :601-602)
#pragma unroll
        for (int k = 0; k < 4; ++k) y[k] *= r;
    }

    // ---- post-step geometry, split over the pair ----
    const Rot R = rot_from_quat(y);
    double wl[3];
    rot_apply(R, y + 4, wl);                                   // own body rate in LVLH (:451-468)
    // swap: chaser lane sends wc_L, target lane sends rc
    double got[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) got[k] = pair_swap(body ? rc[k] : wl[k]);
    double part0, part1, part2;                                // target: pos^2, vel^2, rot^2 ; chaser: att, |rc|^2, -
    int col_now = 0;
    if (body) {
        double rd_l[3], vd_l[3], ax[3], d[3];
        rot_apply(R, P.rd, rd_l);
        cross3(wl, rd_l, vd_l);
#pragma unroll
        for (int k = 0; k < 3; ++k) d[k] = rc[k] - rd_l[k];
        part0 = dot3(d, d);
#pragma unroll
        for (int k = 0; k < 3; ++k) d[k] = vc[k] - vd_l[k];
        part1 = dot3(d, d);
#pragma unroll
        for (int k = 0; k < 3; ++k) d[k] = got[k] - wl[k];     // wc_L - wt_L
        part2 = dot3(d, d);
        const double rc_sq = dot3(rc, rc);
        if (rc_sq < P.koz_radius_sq) {                         // check_collision (:388-404)
            rot_apply(R, P.corridor_axis, ax);
            const double th = rounded_angle_from(dot3(rc, ax), rc_sq, dot3(ax, ax));
            col_now = th > P.corridor_half_angle ? 1 : 0;
        }
    } else {
        double cap[3];
        rot_apply(R, P.capture_axis, cap);
        const double rc_sq = dot3(got, got);
        part0 = rounded_angle_from(-dot3(got, cap), rc_sq, dot3(cap, cap));    // attitude error (:424-434)
        part1 = rc_sq;
        part2 = 0.0;
    }
    // chaser lane collects the target lane's results
    const double pos_sq = pair_swap(part0), vel_sq = pair_swap(part1), rot_sq = pair_swap(part2);
    const double fuel_t = pair_swap(fuel), total_t = pair_swap(total);
    const int col_t = pair_swap(col_now);

    // ---- observation (:205): each lane writes the slots it owns into the shared staging row ----
    float *o = s_obs + (threadIdx.x >> 1) * RDV_OBS_DIM;
    const ObsScale sc = obs_scale(P);
    bool in_box = true;
    if (body) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float a = (float)fma(2.0 * (rc[k] + sc.hi_r), sc.inv_r, -1.0);
            const float b = (float)fma(2.0 * (vc[k] + sc.hi_v), sc.inv_v, -1.0);
            o[k] = a; o[3 + k] = b;
            in_box = in_box && a >= -1.0f && a <= 1.0f && b >= -1.0f && b <= 1.0f;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float a = (float)y[k];
            o[13 + k] = a;
            in_box = in_box && a >= -1.0f && a <= 1.0f;
        }
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float a = (float)y[k];
            o[6 + k] = a;
            in_box = in_box && a >= -1.0f && a <= 1.0f;
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float a = (float)fma(2.0 * (y[4 + k] + sc.hi_w), sc.inv_w, -1.0);
            o[10 + k] = a;
            in_box = in_box && a >= -1.0f && a <= 1.0f;
        }
    }
    const int box_t = pair_swap((int)in_box);

    // ---- state write-back: every lane stores the rows it owns ----
    double *fw = S.f64 + i;
    if (active) {
#pragma unroll
        for (int k = 0; k < 4; ++k) fw[(qrow + k) * ld] = y[k];
#pragma unroll
        for (int k = 0; k < 3; ++k) fw[(wrow + k) * ld] = y[4 + k];
        fw[(body ? RDV_TDV : RDV_TDW) * ld] = total;
        if (body) {
#pragma unroll
            for (int k = 0; k < 3; ++k) { fw[(RDV_RCX + k) * ld] = rc[k]; fw[(RDV_VCX + k) * ld] = vc[k]; }
        }
    }
    st.rk_acc = active ? rk_acc : 0; st.rk_rej = active ? rk_rej : 0; st.fail = active ? fail : 0;

    // ---- chaser lane: latch, time, bubble, done, reward, outputs ----
    int done = 0, fin_pos = 0;
    if (!body) {
        int step = S.i32[RDV_I_STEP * ld + i], success = S.i32[RDV_I_SUCCESS * ld + i];
        int collided = S.i32[RDV_I_COLLIDED * ld + i];
        double ep_ret = f[RDV_EPRET * ld];
        const double att = part0, rc_sq = part1;
        // collision / success latch (:186-190); the three vector errors are compared as squares
        if (!collided) {
            collided = col_t;
            if (!collided && pos_sq <= P.max_rd_error_sq && vel_sq <= P.max_vd_error_sq && att <= P.max_qd_error &&
                rot_sq <= P.max_wd_error_sq)
                success += 1;
        }
        // time and bubble (:193-198), derived from the step counter
        step += 1;
        const double bubble = fmax(fma(-(double)step, P.bubble_rate, P.bubble0), P.bubble_min);
        // done (:355-386): first true condition is the end reason
        const bool c0 = !(in_box && box_t), c1 = step >= P.done_steps, c2 = rc_sq > bubble * bubble,
                   c3 = att > P.max_attitude_error;
        done = (c0 || c1 || c2 || c3) ? 1 : 0;
        const int reason = c0 ? 0 : c1 ? 1 : c2 ? 2 : c3 ? 3 : -1;
        // reward (:313-353)
        double rew = P.att_scale * fma(-att, P.inv_max_attitude_error, 1.0);
        rew += fuel_t;
        if (col_t) rew -= P.collision_scale;
        if (rc_sq < P.koz_radius_sq && !collided && pos_sq < P.max_rd_error_sq) {
            rew += P.bonus_scale * fma(-fast_sqrt(pos_sq), P.inv_max_rd_error, 2.0);
            if (att < P.max_qd_error) rew += P.bonus_scale * fma(-att, P.inv_max_qd_error, 2.0);
        }
        ep_ret += rew;
        if (active) {
            io.reward[i] = rew;
            if (io.reward_f32) io.reward_f32[i] = (float)rew;
            io.done[i] = (uint8_t)done;
            if (io.end_reason) io.end_reason[i] = (int8_t)reason;
            st.steps = 1; st.reward = rew;
            fw[RDV_EPRET * ld] = ep_ret;
            S.i32[RDV_I_STEP * ld + i] = step; S.i32[RDV_I_SUCCESS * ld + i] = success;
            S.i32[RDV_I_COLLIDED * ld + i] = collided;
            if (done) {
                st.episodes = 1; st.succeeded = success > 0; st.collided = collided;
                st.end0 = reason == 0; st.end1 = reason == 1; st.end2 = reason == 2; st.end3 = reason == 3;
                st.ep_return = ep_ret; st.ep_length = (double)step; st.delta_v = total_t; st.delta_w = total;
                if (io.episode_record) {
                    double *rec = io.episode_record + RDV_EP_NCOL * i;
                    rec[RDV_EP_RETURN] = ep_ret; rec[RDV_EP_LENGTH] = (double)step;
                    rec[RDV_EP_SUCCESS] = (double)success; rec[RDV_EP_COLLIDED] = (double)collided;
                    rec[RDV_EP_DELTA_V] = total_t; rec[RDV_EP_DELTA_W] = total;
                }
                if (io.auto_reset || io.fin_rows) {
                    fin_pos = atomicAdd(&s_reset_n, 1);
                    s_reset_idx[fin_pos] = threadIdx.x >> 1;
                }
                if (io.fin_rows) {
                    double *fr = s_fin_rec[threadIdx.x >> 1];
                    fr[RDV_EP_RETURN] = ep_ret; fr[RDV_EP_LENGTH] = (double)step;
                    fr[RDV_EP_SUCCESS] = (double)success; fr[RDV_EP_COLLIDED] = (double)collided;
                    fr[RDV_EP_DELTA_V] = total_t; fr[RDV_EP_DELTA_W] = total;
                    s_fin_reason[threadIdx.x >> 1] = reason;
                }
            }
        }
    }

    // ---- terminal observation of finished episodes: the pair copies its staged row ----
    __syncwarp();
    const int done_pair = __shfl_sync(0xffffffffu, done, (threadIdx.x & 31) & ~1);
    if (io.terminal_obs) {
        if (done_pair && active) {
            float *to = io.terminal_obs + RDV_OBS_DIM * i;
            for (int k = body; k < RDV_OBS_DIM; k += 2) to[k] = o[k];
        }
    }
    // ---- compacted rows of the finished envs (what a VecEnv's infos carry), one global atomic per CTA ----
    if (io.fin_rows) {
        __syncthreads();
        if (threadIdx.x == 0) s_fin_base = s_reset_n ? atomicAdd(io.fin_count, s_reset_n) : 0;
        __syncthreads();
        const int pos_pair = __shfl_sync(0xffffffffu, fin_pos, (threadIdx.x & 31) & ~1);
        const int slot = s_fin_base + pos_pair;
        if (done_pair && active && slot < io.fin_capacity) {
            RdvFinishedRow *fr = static_cast<RdvFinishedRow *>(io.fin_rows) + slot;
            if (!body) {
                fr->env = io.fin_env_base + (int32_t)i; fr->end_reason = s_fin_reason[threadIdx.x >> 1]; fr->pad = 0.0f;
#pragma unroll
                for (int k = 0; k < RDV_EP_NCOL; ++k) fr->record[k] = s_fin_rec[threadIdx.x >> 1][k];
            }
            for (int k = body; k < RDV_OBS_DIM; k += 2) fr->terminal_obs[k] = o[k];
        }
    }

    // ---- auto-reset (what DummyVecEnv.step_wait does around step, main.py:33-34): the CTA's finished envs
    //      are reset by teams of 8 lanes, 16 envs per pass; their staged observation rows are replaced by
    //      the post-reset observation.  The stores are ordered after the step's own by the barrier.
    __syncthreads();
    if (io.auto_reset) {
        const int count = s_reset_n, team = threadIdx.x / RDV_TEAM;
        for (int b = 0; b < count; b += TPB / RDV_TEAM) {
            // the list is dense, so whole warps (4 teams each) drop out as soon as their first team is past it
            if (b + (team & ~3) >= count) break;
            const bool valid = b + team < count;
            const int local = valid ? s_reset_idx[b + team] : 0;
            const int64_t ie = base + local < n ? base + local : n - 1;
            team_reset(params_of<TABLE>(Pc, S, ie), S, seed, env_offset + ie, ie, valid, 1, nullptr, s_team[team],
                       s_obs + local * RDV_OBS_DIM);
        }
        __syncthreads();
    }

    // ---- coalesced observation write-out: the CTA's rows are contiguous in obs[n][17] ----
    {
        const int64_t rows = (n - base) < EPB ? (n - base) : EPB;
        const int total_f = (int)rows * RDV_OBS_DIM;
        float *dst = io.obs + base * RDV_OBS_DIM;              // base*17*4 B is a multiple of 16 (EPB = 64)
        const int nvec = total_f >> 2;
        const float4 *src4 = reinterpret_cast<const float4 *>(s_obs);
        float4 *dst4 = reinterpret_cast<float4 *>(dst);
        for (int k = threadIdx.x; k < nvec; k += TPB) dst4[k] = src4[k];
        for (int k = (nvec << 2) + threadIdx.x; k < total_f; k += TPB) dst[k] = s_obs[k];
    }
    if (io.stats) reduce_stats<TPB / 32>(st, io.stats, s_stats);
}

// ---------------------------------------------------------------------------------
// Fused rollout: K consecutive steps of every env in ONE launch, state resident in registers.
//
// Per step: the action comes from a caller tensor [K][n][6], from the device Philox stream (philox_actions) or
// from the actor evaluated in the launch; the env steps through the shared building blocks of rdv_step.cuh, and
// finished envs restart inside the warp: the warp's four 8-lane teams (team_reset_core) compute reset states into
// shared-memory rows -- ahead of time, one row per lane, refilled every few steps (the reset state of (env,
// episode) does not depend on the trajectory), or on demand with the fused actor.  What a per-step launch pays
// every step -- launch latency, 193 B/env of state load + store -- is paid once per K steps.  Statistics are
// accumulated in registers and reduced once.
// ---------------------------------------------------------------------------------
// Launch shape: ONE CTA per SM, every CTA owns an equal contiguous slice of the batch and walks it in
// passes of at most TPB environments, all K steps of a pass before the next pass.  The CTA's warps re-converge
// at a barrier every SYNC_PERIOD steps: the step is tens of KB of straight-line code, and warps that drift far
// apart thrash the instruction cache (measured with the first, ~60 KB step: 58 % hit rate and 3.1 of 6.2 stall
// cycles per instruction on "no instruction" with four independent 64-thread CTAs per SM; in-phase warps ran the
// same workload 1.7x faster).
// POLICY: the action of every step is the output of the SB3 MlpPolicy actor, evaluated on the tensor cores
// (tcgen05 / TMEM, rdv_policy_tc.cuh: groups of 128 threads = 128 envs = one UMMA tile) from the observation the
// previous step produced.
// PTAB (policy tables, with POLICY): every 128-env tile of the launch has its own actor, an entry of
// RdvRolloutIO.policy_table chosen by policy_tile.  Slices are cut at multiples of 128 envs and passes are 256 envs,
// so each group's tile is 128 envs starting at a multiple of 128 from env 0 of the launch; each group stages its
// entry's weights into its own weight set (TableSmem) when the entry differs from the one it holds.
constexpr int SYNC_PERIOD = 8;            // steps between the CTA barriers that keep the warps in one code region
constexpr int HELP_POST_PERIOD = 3;       // helper-warp variant: steps between the workers' request posts (1: 12 % slower, 2-4 alike)
constexpr int HELP_IDLE_NS = 500;         // helper-warp variant: sleep of an idle helper between polls
constexpr int LOCKSTEP_MAX_TPB = 256;     // CTAs up to this size interleave the two attitude solves (rk45_iso_plane_pair)
constexpr int RDV_NEXT_ROW = 22;          // doubles per prefetched reset row: state[20], collided, success
constexpr int RDV_ROW_TAG = 22;           // row of RdvRolloutIO.reset_rows holding the episode index a row belongs to

// state of `e` / counters of `c` from a reset row (stride 1 in shared memory, stride ld in the global scratch)
RDV_DEV void take_reset_row(const double *rw, const int64_t rs, EnvRegs &e, EnvCounters &c)
{
#pragma unroll
    for (int j = 0; j < 3; ++j) { e.rc[j] = rw[(RDV_RCX + j) * rs]; e.vc[j] = rw[(RDV_VCX + j) * rs]; }
#pragma unroll
    for (int j = 0; j < 4; ++j) { e.qc[j] = rw[(RDV_QCW + j) * rs]; e.qt[j] = rw[(RDV_QTW + j) * rs]; }
#pragma unroll
    for (int j = 0; j < 3; ++j) { e.wc[j] = rw[(RDV_WCX + j) * rs]; e.wt[j] = rw[(RDV_WTX + j) * rs]; }
    c.collided = (int)rw[20 * rs]; c.success = (int)rw[21 * rs];
    c.step = 0; c.episode += 1; c.tdv = c.tdw = c.ep_ret = 0.0;
}

// OBS: the float32 observation is formed every step (the actor's input, a per-step record); without it only its Box
// test is evaluated, on the raw state (obs_in_box_state), and the observation is formed once at the end of the launch.
// HELP: the CTA carries two more warps than its TPB_ / 32 worker warps.  65,536 envs are 13.84 worker warps per SM,
// which the hardware deals out 4-4-3-3 over the four schedulers: two schedulers set the pace, two idle a quarter of the
// time.  The helper warps land on those two (warp id mod 4) and take the one piece of the step that does not depend on
// the trajectory off the workers: recomputing the reset rows that were used.  Workers post (lane, episode) requests in
// shared memory and never wait -- a row that is not ready when its lane finishes is computed on the spot, as before.
// TRAJ: every step writes one row of RDV_TR_NCOL doubles per env to `traj` ([K][RDV_TR_NCOL][n], rdv_b200.h): the
// state and counters after the step's evaluation, before an auto-reset, and the evaluator quantities of that state in
// the forms of errors_kernel.  Only the TRAJ variants read `traj`.
template <bool ISO, bool CLOSED, int TPB_, bool POLICY = false, bool MC = false, bool TABLE = false, bool OBS = POLICY,
          bool HELP = false, bool PTAB = false, bool TRAJ = false>
__global__ void __launch_bounds__(TPB_ + (HELP ? 64 : 0), 1)
rollout_kernel(const __grid_constant__ RdvParams Pc, const RdvState S, const __grid_constant__ RdvRolloutIO io,
               const int64_t n, const uint64_t seed, const int64_t env_offset, double *const traj)
{
    static_assert(!HELP || (!POLICY && !MC && !TABLE && !OBS), "helper warps: plain variant only");
    static_assert(!PTAB || (POLICY && TPB_ == 256), "policy tables: the fused actor with two 128-thread groups");
    constexpr int NW = TPB_ / 32;                       // worker warps
    constexpr int NWT = NW + (HELP ? 2 : 0);            // all warps of the CTA
    extern __shared__ __align__(128) unsigned char dyn_smem[];
    typedef typename std::conditional<PTAB, tc::TableSmem, tc::TileSmem>::type TS;
    TS *ts = reinterpret_cast<TS *>(dyn_smem);
    uint32_t tmem_all = 0, mma_phase = 0;
    if constexpr (PTAB) {
        tmem_all = tc::tile_cta_setup(*ts);             // the weights are staged per group, at the start of a pass
    } else if (POLICY) {
        // the actor's weights may have been written by the previous kernel of the stream (an optimiser step), so the
        // dependency wait of a programmatic launch (below) comes before they are read
        asm volatile("griddepcontrol.wait;" ::: "memory");
        tmem_all = tc::tile_setup<TPB_>(io.policy, *ts);
    }
    // Without the actor the tensor memory (256 KB per SM) is entirely idle; the variant for the reference's bodies
    // allocates it as a parking area for cold registers (see the step phase): 128 columns for every thread.
    constexpr bool main_stash = !POLICY && !MC && ISO && !CLOSED;
    __shared__ uint32_t s_tmem_base;
    if constexpr (main_stash) {
        if (threadIdx.x < 32) {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                         :: "r"(tc::smem_u32(&s_tmem_base)), "r"(tc::TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
        tc::tc_fence_before();
        __syncthreads();
        tc::tc_fence_after();
        tmem_all = s_tmem_base;
    }
    // Staging rows of the observation write-out.  Only the variant that records an observation every step owns them;
    // the others stage the ONE observation of a launch in memory that is dead by then (below), which keeps the CTA under
    // 100 KiB of shared memory and leaves 156 KiB of L1 for the ~140 KB of register spills of 448 threads (with the
    // rows the carve-out was 132 KiB and one spill load in ten went to the L2).
    constexpr bool own_stage = !POLICY && OBS;
    __shared__ __align__(16) float s_obs[own_stage ? NW : 1][own_stage ? 32 * RDV_OBS_DIM : 4];
    __shared__ double s_stats[NWT][RDV_NSTATS];
    // scratch rows of the warps' four reset teams; with the fused actor they borrow the group's lo-activation tile
    // (behind the observation staging rows), like those dead outside the actor: the CTA then fits in 100 KiB of
    // shared memory and the L1 carve-out is 156 KiB instead of 124
    __shared__ double s_team_static[POLICY ? 1 : NWT][4][RDV_TEAM_ROW];
    // helper protocol: episode each lane's row in shared memory was computed for (-1: none), episode a row is wanted
    // for, lanes with an open request, and the end-of-launch flag
    __shared__ int s_row_ep[HELP ? NW : 1][32], s_ep_req[HELP ? NW : 1][32];
    __shared__ unsigned s_todo[HELP ? NW : 1];
    __shared__ unsigned s_cancel;                       // worker warps that are leaving the step loop
    __shared__ int s_inflight[2];                       // 1 + the worker warp each helper is serving (0: none)
    __shared__ int s_ndone;                             // worker warps that have left the step loop
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if constexpr (HELP) {
        if (threadIdx.x < NW) s_todo[threadIdx.x] = 0u;
        if (threadIdx.x == 0) { s_ndone = 0; s_cancel = 0u; s_inflight[0] = s_inflight[1] = 0; }
        __syncthreads();
    }
    const int src = io.action_source;
    const int64_t ld = S.ld;
    // Reset prefetch: the reset state of (env, episode + 1) does not depend on the trajectory, so every lane keeps its
    // NEXT reset row ready.  A finished lane just reads its row; the rows are recomputed for all lanes that used
    // theirs every `refill` steps, four per pass of the warp's 8-lane teams with every team busy, instead of one pass
    // with 1.6 of 4 teams busy on 80 % of the steps.  A lane that finishes twice between refills gets its row at once.
    // The rows live in shared memory (in the caller's global scratch when the fused actor owns the shared memory);
    // with io.reset_rows they are loaded at entry and stored at exit, so they survive from launch to launch and a
    // 16-step launch runs at the rate of a 250-step one.  Without the scratch, launches of < 2 refill periods and the
    // fused actor reset on demand.
    const bool persist = io.reset_rows != nullptr && io.auto_reset && !MC && io.reserved > 0;   // (period 0: on demand only)
    const int refill = (!MC && io.auto_reset && io.reserved > 0 && (persist || (!POLICY && io.steps >= 2 * io.reserved)))
                           ? io.reserved : 0;
    double *next_rows = reinterpret_cast<double *>(dyn_smem) + (size_t)warp * 32 * RDV_NEXT_ROW;
    // the warp's observation staging row; with the fused actor it borrows the group's activation tile, which is
    // only live between the step barrier and the end of the actor's third layer
    // (without per-step records: the warp's reset rows, 32 x 22 doubles, which have gone back to the scratch -- or are
    // simply not needed any more -- when the final observation is written)
    float *obs_stage = POLICY ? reinterpret_cast<float *>(ts->al[warp >> 2]) + (warp & 3) * (32 * RDV_OBS_DIM)
                              : own_stage ? s_obs[own_stage ? warp : 0] : reinterpret_cast<float *>(next_rows);
    double (*s_team_w)[RDV_TEAM_ROW] =
        POLICY ? reinterpret_cast<double (*)[RDV_TEAM_ROW]>(reinterpret_cast<char *>(ts->al[warp >> 2]) +
                                                             4 * 32 * RDV_OBS_DIM * sizeof(float)) + (warp & 3) * 4
               : s_team_static[POLICY ? 0 : warp];
    static_assert(4 * 32 * RDV_OBS_DIM * sizeof(float) + 4 * 4 * RDV_TEAM_ROW * sizeof(double) <= sizeof(ts->al[0]),
                  "staging rows + team rows must fit the group's activation tile");
    constexpr bool want_obs = POLICY || OBS;
    // this CTA's slice [lo, hi) and its passes; with a parameter table the slices are cut at multiples of 32 envs so
    // that a warp never straddles two parameter blocks, with a policy table at multiples of 128 so that a group's tile
    // never straddles two policy tiles (the results do not depend on the slicing)
    const int64_t units = PTAB ? (n + 127) / 128 : TABLE ? (n + 31) / 32 : n, unit = PTAB ? 128 : TABLE ? 32 : 1;
    const int64_t lo = unit * (units * (int64_t)blockIdx.x / gridDim.x);
    const int64_t hi_raw = unit * (units * ((int64_t)blockIdx.x + 1) / gridDim.x), hi = hi_raw < n ? hi_raw : n;
    const int64_t span = hi - lo;
    const int passes = (int)((span + TPB_ - 1) / TPB_);
    const int64_t chunk = (TABLE || PTAB) ? TPB_ : (passes > 0 ? (span + passes - 1) / passes : 0);
    // policy tables: the entry whose weights this thread's group holds (-1: none yet; uniform within the group), and
    // whether the group's tile of the current pass has an index outside the table
    int ptab_staged = -1;
    bool ptab_bad = false;
    StepStats st = {};
    // Programmatic dependent launch: when rdv_rollout launches with the stream-serialisation attribute, this grid may
    // become resident while the previous kernel of the stream is still draining (its CTAs finish at different times),
    // and everything above -- parameter loads, the TMEM allocation -- runs in that shadow.
    // Nothing written by an earlier kernel is read before this point; the wait returns once the previous grid has
    // completed and its writes are visible.  Dependents of THIS grid may be scheduled as soon as its CTAs start to exit.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;");

    if constexpr (HELP) {
        if (warp >= NW && passes > 0) {
            // ---- helper warp h serves worker warps h, h + 2, ... until all of them have left the step loop (the host
            //      launches this variant only when every CTA has a single pass, so env (ww, l) is
            //      env_offset + lo + 32 ww + l).  (Handing the four teams of a pass requests of different warps, so
            //      that every pass is full, measured slower: 3.9 us per pass against 2.5.)
            const RdvParams &P = Pc;
            const int h = warp - NW;
            for (;;) {
                bool worked = false;
                for (int ww = h; ww < NW; ww += 2) {
                    if (!*(volatile unsigned *)&s_todo[ww]) continue;
                    // publish the warp, then take its requests: a leaving warp either finds its requests still there
                    // (and takes them back) or sees this flag and waits for the pass in flight
                    unsigned m = 0;
                    if (lane == 0) {
                        *(volatile int *)&s_inflight[h] = ww + 1;
                        __threadfence_block();
                        m = atomicExch(&s_todo[ww], 0u);
                    }
                    m = __shfl_sync(full, m, 0);
                    worked = true;
                    double *rows = reinterpret_cast<double *>(dyn_smem) + (size_t)ww * 32 * RDV_NEXT_ROW;
                    while (m && !((*(volatile unsigned *)&s_cancel >> ww) & 1u)) {
                        const int team = lane >> 3;
                        const unsigned src_bit = __fns(m, 0, team + 1);
                        const int src_lane = src_bit < 32 ? (int)src_bit : 0;
                        const int r_episode = *(volatile int *)&s_ep_req[ww][src_lane];
                        team_reset_core(P, seed, env_offset + lo + ww * 32 + src_lane, r_episode, nullptr,
                                        src_bit < 32 ? rows + src_lane * RDV_NEXT_ROW : s_team_w[team]);
                        __threadfence_block();                           // row before tag
                        if (src_bit < 32 && (lane & 7) == 0) *(volatile int *)&s_row_ep[ww][src_lane] = r_episode;
#pragma unroll
                        for (int j = 0; j < 4; ++j) m &= m - 1;
                    }
                    __syncwarp();
                    __threadfence_block();
                    if (lane == 0) *(volatile int *)&s_inflight[h] = 0;
                }
                if (*(volatile int *)&s_ndone >= NW) break;
                if (!worked) __nanosleep(HELP_IDLE_NS);
            }
        }
    }

    for (int pass = 0; pass < ((HELP && warp >= NW) ? 0 : passes); ++pass) {
        const int64_t c_lo = lo + pass * chunk, c_hi = (c_lo + chunk < hi) ? c_lo + chunk : hi;
        const int64_t warp_base = c_lo + warp * 32;
        const int64_t i_raw = warp_base + lane;
        const bool active = i_raw < c_hi;
        const int64_t i = active ? i_raw : c_hi - 1;           // idle lanes shadow the last env (no stores)
        const int64_t env_id = env_offset + i;
        const int rows_w = (int)((c_hi - warp_base) < 32 ? ((c_hi - warp_base) > 0 ? (c_hi - warp_base) : 0) : 32);
        const RdvParams &P = params_of<TABLE>(Pc, S, i);
        if constexpr (PTAB) {
            // The group's tile: idle lanes shadow the slice's last env, which lies in the tile of the group's active
            // envs (or, for a group with none, is the same env for all 128 threads), so `want` is group-uniform.
            const int g = threadIdx.x >> 7;
            const int32_t want = io.policy_tile[i >> 7];
            ptab_bad = want < 0 || want >= io.policy_count;         // never read outside the table: zero actions
            if (!ptab_bad) {
                // an entry the actor cannot run is treated the same way: another width (the staging reads 64-wide
                // matrices), a missing weight, or no Gaussian head when sampling
                const RdvPolicy &pe = io.policy_table[want];
                ptab_bad = pe.hidden != tc::H || !pe.w0 || !pe.b0 || !pe.w1 || !pe.b1 || !pe.w2 || !pe.b2 ||
                           (src == RDV_ACTIONS_POLICY_SAMPLE && !pe.log_std);
            }
            if (!ptab_bad && want != ptab_staged) {
                // the group's MMAs of its previous tile have completed (every thread waited for them), but a thread may
                // still read the previous biases / std: wait for the group, restage, publish to the async proxy
                tc::group_sync(g, tc::TM);
                tc::stage_weights<tc::TM>(io.policy_table[want], ts->w[g], threadIdx.x & (tc::TM - 1));
                tc::fence_async_smem();
                tc::group_sync(g, tc::TM);
                ptab_staged = want;
            }
        }

        EnvRegs e;
        EnvCounters c;
        load_env(S, i, e);
        load_counters(S, i, c);
        float ov[RDV_OBS_DIM];
        if (want_obs) make_obs(e, obs_scale(P), ov);
        unsigned fresh = 0;                                    // lanes whose next reset row is ready
        int countdown = HELP ? HELP_POST_PERIOD : refill;      // steps until the next refill of the rows (HELP: next post)
        // where this lane's row lives
        double *my_row = POLICY ? io.reset_rows + i : next_rows + lane * RDV_NEXT_ROW;
        const int64_t row_stride = POLICY ? ld : 1;
        if (persist) {
            const bool ok = active && io.reset_rows[RDV_ROW_TAG * ld + i] == (double)(c.episode + 1);
            fresh = __ballot_sync(full, ok);
            if (!POLICY && ok) {
#pragma unroll
                for (int j = 0; j < RDV_NEXT_ROW; ++j) my_row[j] = io.reset_rows[j * ld + i];
            }
            __syncwarp();
        }
        // posts a request for every active lane whose row is not the one its NEXT reset needs
        auto post_requests = [&]() {
            if constexpr (HELP) {
                const bool want = active && *(volatile int *)&s_row_ep[warp][lane] != c.episode + 1;
                if (want) s_ep_req[warp][lane] = c.episode + 1;
                const unsigned wm = __ballot_sync(full, want);
                __threadfence_block();
                if (lane == 0 && wm) atomicOr(&s_todo[warp], wm);
            }
        };
        if constexpr (HELP) {
            s_row_ep[warp][lane] = ((fresh >> lane) & 1u) ? c.episode + 1 : -1;
            __syncwarp();
            post_requests();
        }
        // rows for the lanes of `todo`, four per pass of the warp's teams
        auto fill_rows = [&](unsigned todo) {
            while (todo) {
                const int team = lane >> 3;
                const unsigned src_bit = __fns(todo, 0, team + 1);            // team-th lane of the set, or ~0u
                const int src_lane = src_bit < 32 ? (int)src_bit : lane;
                const int64_t r_env = __shfl_sync(full, env_id, src_lane);
                const int r_episode = __shfl_sync(full, c.episode, src_lane) + 1;
                if (POLICY) {
                    // computed in the team's scratch row, then copied to the env's column of the global scratch
                    double *tr = s_team_w[team];
                    team_reset_core(P, seed, r_env, r_episode, nullptr, tr);
                    if (src_bit < 32) {
                        double *dst = io.reset_rows + (r_env - env_offset);
                        for (int j = lane & 7; j < RDV_NEXT_ROW; j += 8) dst[j * ld] = tr[j];
                        if ((lane & 7) == 0) dst[RDV_ROW_TAG * ld] = (double)r_episode;
                    }
                    __syncwarp();
                } else {
                    team_reset_core(P, seed, r_env, r_episode, nullptr,
                                    src_bit < 32 ? next_rows + src_lane * RDV_NEXT_ROW : s_team_w[team]);
                }
#pragma unroll
                for (int j = 0; j < 4; ++j) todo &= todo - 1;                  // drop the four handled lanes
            }
        };

        // Monte-Carlo evaluator mode: sample 0 is the state at launch (monte_carlo.py:117-124)
        McAcc mc;
        bool alive = true;
        int mc_reason = -1;
        EvalDetail d_last;                                     // TRAJ + MC: the detail of the env's last state
        if constexpr (MC) {
            mc_init(mc);
            EvalDetail d;
            eval_detail_of_state(P, e, d);
            mc_sample(P, d, c.collided, mc);
            if constexpr (TRAJ) d_last = d;
        }

        // One env step = an action phase (actor on the tensor cores, or a tensor / Philox action) and a step phase
        // (propagation, evaluation, in-warp reset, records), written as lambdas over the pass's registers.
        ActionTerms t;
        auto policy_action = [&](const int k) {
            const int64_t row = (int64_t)k * n + i;
            // the CTA's threads form groups of 128 (the last one may be smaller); a group runs its tile of envs
            // through the actor on the tensor cores: thread = row = TMEM lane
            float a[RDV_ACT_DIM];
            const int g = threadIdx.x >> 7;
            if (PTAB && ptab_bad) {
                // tile index outside the policy table, or an entry the actor cannot run: zero actions, one failure
                // per env-step
#pragma unroll
                for (int j = 0; j < RDV_ACT_DIM; ++j) a[j] = 0.0f;
                if (active && (!MC || alive)) st.fail += 1;
            } else {
                tc::tile_forward(ts->al[g], &ts->mma_bar[g], ts->w[PTAB ? g : 0], g, threadIdx.x & 127,
                                 TPB_ - 128 * g < 128 ? TPB_ - 128 * g : 128, ov, tmem_all + (uint32_t)g * tc::GROUP_COLS,
                                 mma_phase, a, [] {});
            }
            const bool sample = src == RDV_ACTIONS_POLICY_SAMPLE;
            if (sample && !(PTAB && ptab_bad)) {              // a ~ N(mean, exp(log_std)^2)
                float z[RDV_ACT_DIM];
                philox_normals(io.action_seed, env_id, io.step_base + k, z);
#pragma unroll
                for (int j = 0; j < RDV_ACT_DIM; ++j) a[j] = fmaf(ts->w[PTAB ? g : 0].std[j], z[j], a[j]);
            }
            float ac[RDV_ACT_DIM];
#pragma unroll
            for (int j = 0; j < RDV_ACT_DIM; ++j) ac[j] = fminf(1.0f, fmaxf(-1.0f, a[j]));   // np.clip to the Box
            if (io.actions_out && active) {
                // sampling: the unclipped draw (what SB3's rollout buffer stores); deterministic: the clipped
                // action model.predict returns
                const float *rec = sample ? a : ac;
                float2 *op = reinterpret_cast<float2 *>(reinterpret_cast<float *>(io.actions_out) + 6 * row);
                op[0] = make_float2(rec[0], rec[1]); op[1] = make_float2(rec[2], rec[3]);
                op[2] = make_float2(rec[4], rec[5]);
            }
#pragma unroll
            for (int j = 0; j < RDV_ACT_DIM; ++j) a[j] = ac[j];
            if (!MC || alive) ingest_action_f32(P, a, c, t);
        };
        auto step_phase = [&](const int k) {
            const int64_t row = (int64_t)k * n + i;
            // ---- step ----
            int rk_acc = 0, rk_rej = 0, fail = 0;
            StepResult r;
            if constexpr (MC) {
                // evaluator mode: an env stops at its first done (its lanes idle from then on)
                r.rew = 0.0; r.done = 0; r.reason = -1;
                if (alive) {
                    env_advance<ISO, CLOSED, (TPB_ <= LOCKSTEP_MAX_TPB)>(P, e, t, rk_acc, rk_rej, fail);
                    EvalDetail d;
                    r = env_evaluate<true, true>(P, e, t.fuel, c, ov, &d);
                    mc_sample(P, d, c.collided, mc);                          // monte_carlo.py:140-149
                    if constexpr (TRAJ) d_last = d;
                    mc.total_reward += r.rew;
                    mc.len += 1;
                    if (r.done) { alive = false; mc_reason = r.reason; }
                }
            } else if constexpr (POLICY || main_stash) {
                // The fused actor owns 196 KiB of shared memory, which leaves 60 KiB of L1 for 136 KB of register
                // spills (local loads hit 58 %, and the misses cost an L2 round trip: 22 % of this variant's issue
                // latency were long-scoreboard stalls).  During the env step the group's tensor memory is idle -- D and
                // the A operand are only live inside the actor -- so everything the two attitude solves do not touch
                // (position, velocity, totals, counters, the statistics accumulators: 45 words per env) is parked in
                // the thread's own TMEM lane across them instead of being spilled: three tcgen05.st / three
                // tcgen05.ld per step instead of ~50 local stores and loads.
                env_translate(P, e, t);
                // a warp reaches the 32 lanes of its quadrant (warp id mod 4); warps of one quadrant take different
                // column blocks.  With the actor: the group's own 128 columns (thread = TMEM lane there anyway).
                const uint32_t lane_addr = tmem_all + (uint32_t)(threadIdx.x >> 7) * tc::GROUP_COLS +
                                           ((uint32_t)(threadIdx.x & 96) << 16);
                {
                    uint32_t w[48];
                    int q = 0;
                    auto put = [&](double v) { w[q++] = (uint32_t)__double2loint(v); w[q++] = (uint32_t)__double2hiint(v); };
#pragma unroll
                    for (int j = 0; j < 3; ++j) { put(e.rc[j]); put(e.vc[j]); }
                    put(c.tdv); put(c.tdw); put(c.ep_ret); put(t.fuel);
                    put(st.ep_return); put(st.ep_length); put(st.delta_v); put(st.delta_w); put(st.reward);
                    w[q++] = (uint32_t)c.step; w[q++] = (uint32_t)c.success; w[q++] = (uint32_t)c.collided;
                    w[q++] = (uint32_t)c.episode;
                    w[q++] = st.steps; w[q++] = st.episodes; w[q++] = st.succeeded; w[q++] = st.collided;
                    w[q++] = st.end0; w[q++] = st.end1; w[q++] = st.end2; w[q++] = st.end3;
                    w[q++] = st.rk_acc; w[q++] = st.rk_rej; w[q++] = st.fail;
                    while (q < 48) w[q++] = 0u;
                    tc::tmem_st16(lane_addr, reinterpret_cast<const uint32_t (&)[16]>(w[0]));
                    tc::tmem_st16(lane_addr + 16, reinterpret_cast<const uint32_t (&)[16]>(w[16]));
                    tc::tmem_st16(lane_addr + 32, reinterpret_cast<const uint32_t (&)[16]>(w[32]));
                    tc::tmem_st_wait();
                }
                // (parking, in addition, the body that is not being propagated around each solve measured no faster)
                env_attitude<ISO, CLOSED, (TPB_ <= LOCKSTEP_MAX_TPB)>(P, e, t, rk_acc, rk_rej, fail);
                {
                    uint32_t w[48];
                    tc::tmem_ld16_issue(lane_addr, reinterpret_cast<uint32_t (&)[16]>(w[0]));
                    tc::tmem_ld16_issue(lane_addr + 16, reinterpret_cast<uint32_t (&)[16]>(w[16]));
                    tc::tmem_ld16_issue(lane_addr + 32, reinterpret_cast<uint32_t (&)[16]>(w[32]));
                    tc::tmem_ld_wait(reinterpret_cast<uint32_t (&)[16]>(w[0]));
                    tc::tmem_ld_wait(reinterpret_cast<uint32_t (&)[16]>(w[16]));
                    tc::tmem_ld_wait(reinterpret_cast<uint32_t (&)[16]>(w[32]));
                    int q = 0;
                    auto get = [&]() { const double v = __hiloint2double((int)w[q + 1], (int)w[q]); q += 2; return v; };
#pragma unroll
                    for (int j = 0; j < 3; ++j) { e.rc[j] = get(); e.vc[j] = get(); }
                    c.tdv = get(); c.tdw = get(); c.ep_ret = get(); t.fuel = get();
                    st.ep_return = get(); st.ep_length = get(); st.delta_v = get(); st.delta_w = get(); st.reward = get();
                    c.step = (int)w[q++]; c.success = (int)w[q++]; c.collided = (int)w[q++]; c.episode = (int)w[q++];
                    st.steps = w[q++]; st.episodes = w[q++]; st.succeeded = w[q++]; st.collided = w[q++];
                    st.end0 = w[q++]; st.end1 = w[q++]; st.end2 = w[q++]; st.end3 = w[q++];
                    st.rk_acc = w[q++]; st.rk_rej = w[q++]; st.fail = w[q++];
                }
                r = env_evaluate<want_obs>(P, e, t.fuel, c, ov);
            } else {
                env_advance<ISO, CLOSED, (TPB_ <= LOCKSTEP_MAX_TPB)>(P, e, t, rk_acc, rk_rej, fail);
                r = env_evaluate<want_obs>(P, e, t.fuel, c, ov);
            }
            const bool done = r.done && active;
            if (active) {
                if (io.rewards) io.rewards[row] = r.rew;
                if (io.dones) io.dones[row] = (uint8_t)r.done;
                if (!MC || r.reason != -1 || alive) {
                    st.steps += 1; st.reward += r.rew; st.rk_acc += rk_acc; st.rk_rej += rk_rej; st.fail += fail;
                }
                if (r.done) {
                    st.episodes += 1; st.succeeded += c.success > 0; st.collided += c.collided;
                    st.end0 += r.reason == 0; st.end1 += r.reason == 1; st.end2 += r.reason == 2;
                    st.end3 += r.reason == 3;
                    st.ep_return += c.ep_ret; st.ep_length += (double)c.step; st.delta_v += c.tdv; st.delta_w += c.tdw;
                }
            }
            // ---- trajectory record: the state this step left, before an auto-reset replaces it ----
            if constexpr (TRAJ) {
                if (active) {
                    // The step's own evaluation skips quat2mat's re-normalisation and, far from the target, the
                    // errors, so the record's quantities are formed here as errors_kernel forms them; the evaluator
                    // mode has them already (a finished env repeats its last row).
                    EvalDetail d;
                    if constexpr (MC) d = d_last;
                    else eval_detail_of_state(P, e, d);
                    store_traj_row(traj + (int64_t)k * RDV_TR_NCOL * n + i, n, e, c, d);
                }
            }
            // ---- auto-reset inside the warp ----
            if constexpr (HELP) {
                // rows come from the helper warps; what is not ready is computed here, four lanes per pass
                const unsigned m = __ballot_sync(full, done);
                if (m) {
                    const bool have = done && *(volatile int *)&s_row_ep[warp][lane] == c.episode + 1;
                    unsigned need = m & ~__ballot_sync(full, have);
                    if (have) {
                        __threadfence_block();                                   // tag before row
                        take_reset_row(my_row, 1, e, c);
                    }
                    while (need) {
                        const int team = lane >> 3;
                        const unsigned src_bit = __fns(need, 0, team + 1);
                        const int src_lane = src_bit < 32 ? (int)src_bit : lane;
                        const int64_t r_env = __shfl_sync(full, env_id, src_lane);
                        const int r_episode = __shfl_sync(full, c.episode, src_lane) + 1;
                        team_reset_core(P, seed, r_env, r_episode, nullptr, s_team_w[team]);
                        const int rank = __popc(need & ((1u << lane) - 1));
                        if (((need >> lane) & 1u) && rank < 4) take_reset_row(s_team_w[rank], 1, e, c);
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 4; ++j) need &= need - 1;
                    }
                }
                if (--countdown <= 0) {
                    countdown = HELP_POST_PERIOD;
                    post_requests();
                }
            } else if (!MC && io.auto_reset && refill) {
                // prefetched rows: compute what is missing right now (rare), consume, refill periodically
                const unsigned m = __ballot_sync(full, done);
                const unsigned need = m & ~fresh;
                if (need) fill_rows(need);
                if (done) {
                    take_reset_row(my_row, row_stride, e, c);
                    if (want_obs) make_obs(e, obs_scale(P), ov);               // post-reset observation
                }
                fresh = (fresh | need) & ~m;
                __syncwarp();
                if (--countdown == 0 && k + 1 < io.steps) {
                    countdown = refill;
                    const unsigned todo = __ballot_sync(full, active) & ~fresh;
                    fill_rows(todo);                  // (serving only full passes of four measured no faster)
                    fresh |= todo;
                }
            } else if (!MC && io.auto_reset) {
                // four finished lanes per pass, one 8-lane team each
                unsigned m = __ballot_sync(full, done);
                while (m) {
                    const int team = lane >> 3;
                    const unsigned src_bit = __fns(m, 0, team + 1);           // team-th finished lane, or ~0u
                    const int src_lane = src_bit < 32 ? (int)src_bit : lane;
                    const int64_t r_env = __shfl_sync(full, env_id, src_lane);
                    const int r_episode = __shfl_sync(full, c.episode, src_lane) + 1;
                    team_reset_core(P, seed, r_env, r_episode, nullptr, s_team_w[team]);
                    const int rank = __popc(m & ((1u << lane) - 1));
                    if (((m >> lane) & 1u) && rank < 4) {
                        take_reset_row(s_team_w[rank], 1, e, c);
                        if (want_obs) make_obs(e, obs_scale(P), ov);           // post-reset observation
                    }
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 4; ++j) m &= m - 1;                    // drop the four handled lanes
                }
            }
            // ---- per-step observation record (post-reset for finished envs), coalesced via the warp's row ----
            if (want_obs && io.obs_steps) {
                float *o = obs_stage + lane * RDV_OBS_DIM;
#pragma unroll
                for (int j = 0; j < RDV_OBS_DIM; ++j) o[j] = ov[j];
                __syncwarp();
                float *dst = io.obs_steps + ((int64_t)k * n + warp_base) * RDV_OBS_DIM;
                for (int j = lane; j < rows_w * RDV_OBS_DIM; j += 32) dst[j] = obs_stage[j];
                __syncwarp();
            }
        };

        if constexpr (POLICY) {
            // The fused actor keeps the CTA barrier of every step: its staging rows alias the activation tiles of the
            // next step's actor, and the groups run best in phase.  Measured alternatives at 65,536 envs: no barrier
            // (groups drift) 24.0 us per step against 22.7; odd groups shifted by half a step behind a barrier per
            // half-phase (half of the warps in the actor, half in the solver at any time, so that the tiles' MMAs do
            // not queue on the one tensor pipe) 29.2 against 22.9 -- with only half of the SM's warps in the solver
            // the fp64 latency is no longer hidden, which costs more than the MMA queueing it removes; a named barrier
            // per 128-thread group instead of the CTA barrier (the staging rows only alias the group's own tile)
            // 21.5 against 21.1; a second CTA barrier between the actor and the env step 21.6 against 21.1.
            for (int k = 0; k < io.steps; ++k) {
                __syncthreads();
                policy_action(k);
                step_phase(k);
            }
        } else {
            for (int k = 0; k < io.steps; ++k) {
                // Keep the CTA's warps in the same code region (instruction-cache locality).  With the first, ~60 KB
                // step a barrier every step was best (every 2 / 4 steps: 1 % / 8 % slower); the plane solver's step is
                // smaller and tolerates drift: every step 12.06, every 4-8 steps 11.66, every 32 steps 11.77, never
                // 12.1-12.2 us per step.
                if ((k % SYNC_PERIOD) == 0) {
                    if constexpr (HELP) asm volatile("bar.sync 2, %0;" :: "n"(TPB_) : "memory");   // the workers only
                    else __syncthreads();
                }
                // ---- action ----
                const int64_t row = (int64_t)k * n + i;
                if (src == RDV_ACTIONS_F32) {
                    const float2 *ap = reinterpret_cast<const float2 *>(static_cast<const float *>(io.actions) + 6 * row);
                    const float2 a01 = ap[0], a23 = ap[1], a45 = ap[2];
                    const float a[6] = {a01.x, a01.y, a23.x, a23.y, a45.x, a45.y};
                    if (!MC || alive) ingest_action_f32(P, a, c, t);
                } else {
                    double a[6];
                    if (src == RDV_ACTIONS_F64) {
                        const double2 *ap = reinterpret_cast<const double2 *>(static_cast<const double *>(io.actions) + 6 * row);
                        const double2 a01 = ap[0], a23 = ap[1], a45 = ap[2];
                        a[0] = a01.x; a[1] = a01.y; a[2] = a23.x; a[3] = a23.y; a[4] = a45.x; a[5] = a45.y;
                    } else {
                        philox_actions(io.action_seed, env_id, io.step_base + k, a);
                        if (io.actions_out && active) {
                            double2 *op = reinterpret_cast<double2 *>(io.actions_out + 6 * row);
                            op[0] = make_double2(a[0], a[1]); op[1] = make_double2(a[2], a[3]);
                            op[2] = make_double2(a[4], a[5]);
                        }
                    }
                    if (!MC || alive) ingest_action_f64(P, a, c, t);
                }
                step_phase(k);
            }
        }

        // ---- the rows that were used since the last refill are recomputed before they go back to the scratch,
        //      so the next launch starts with every row ready ----
        if constexpr (HELP) {
            // leave: no more requests of this warp are picked up, a pass that is working on one of its rows is waited
            // for (under 3 us, one time in ten), and what is not ready is computed below.  No CTA barrier: the warps
            // leave at their own pace, as in the plain variant.
            if (lane == 0) {
                atomicOr(&s_cancel, 1u << warp);
                atomicExch(&s_todo[warp], 0u);
                __threadfence_block();
                while (*(volatile int *)&s_inflight[warp & 1] == warp + 1) { }
                atomicAdd(&s_ndone, 1);
            }
            __syncwarp();
            __threadfence_block();
            fresh = __ballot_sync(full, active && *(volatile int *)&s_row_ep[warp][lane] == c.episode + 1);
        }
        if (persist) {
            // (helper variant: what is not ready stays not ready -- the tag says so -- and is the helpers' first work
            //  of the next launch, when they would otherwise idle)
            const unsigned todo = HELP ? 0u : __ballot_sync(full, active) & ~fresh;
            fill_rows(todo);
            if (!POLICY && active) {
                const bool ready = !HELP || ((fresh >> lane) & 1u);
                if (ready) {
#pragma unroll
                    for (int j = 0; j < RDV_NEXT_ROW; ++j) io.reset_rows[j * ld + i] = my_row[j];
                }
                io.reset_rows[RDV_ROW_TAG * ld + i] = ready ? (double)(c.episode + 1) : -1.0;
            }
            __syncwarp();
        }
        // ---- write the state back once per pass, and the final observation ----
        if (active) {
            store_env(S, i, e);
            store_counters(S, i, c);
            if constexpr (MC) {
                double *mo = io.mc_out + (size_t)RDV_MC_NCOL * i;
                const double inv = 1.0 / (double)(mc.count > 0 ? mc.count : 1);
                mo[RDV_MC_EP_LEN] = (double)mc.len; mo[RDV_MC_NUM_COLLISIONS] = (double)mc.n_col;
                mo[RDV_MC_COLLIDED] = mc.n_col > 0 ? 1.0 : 0.0; mo[RDV_MC_TOTAL_REWARD] = mc.total_reward;
                mo[RDV_MC_TOTAL_DELTA_V] = c.tdv; mo[RDV_MC_NUM_SUCCESSES] = (double)mc.n_suc;
                mo[RDV_MC_SUCCEEDED] = mc.n_suc > 0 ? 1.0 : 0.0; mo[RDV_MC_MIN_KOZ] = mc.min_koz;
                mo[RDV_MC_POS_ERR] = mc.sum[0] * inv; mo[RDV_MC_VEL_ERR] = mc.sum[1] * inv;
                mo[RDV_MC_ATT_ERR] = mc.sum[2] * inv; mo[RDV_MC_ROT_ERR] = mc.sum[3] * inv;
                mo[RDV_MC_LEVEL] = (double)mc.level; mo[RDV_MC_TAIL_COUNT] = (double)mc.count;
                mo[RDV_MC_END_REASON] = (double)mc_reason; mo[RDV_MC_TOTAL_DELTA_W] = c.tdw;
            }
        }
        if (!want_obs || MC) make_obs(e, obs_scale(P), ov);
        float *o = obs_stage + lane * RDV_OBS_DIM;
#pragma unroll
        for (int j = 0; j < RDV_OBS_DIM; ++j) o[j] = ov[j];
        __syncwarp();
        float *dst = io.obs + warp_base * RDV_OBS_DIM;
        for (int j = lane; j < rows_w * RDV_OBS_DIM; j += 32) dst[j] = obs_stage[j];
        __syncwarp();
    }
    if (io.stats) reduce_stats<NWT>(st, io.stats, s_stats);
    if (POLICY || main_stash) tc::tile_teardown(tmem_all);
}

// ---------------------------------------------------------------------------------
// reset() for masked envs (rendezvous_env.py:223-270): 8 lanes per env (team_reset), 16 envs per CTA.
// Draws come from Philox or from the caller's uniforms (test hook).
// ---------------------------------------------------------------------------------
template <bool TABLE>
__global__ void __launch_bounds__(128) reset_kernel(const __grid_constant__ RdvParams Pc, const RdvState S,
                                                    const uint8_t *mask, const double *uniforms, float *obs,
                                                    int64_t n, uint64_t seed, int64_t env_offset, int bump)
{
    __shared__ double s_team[128 / RDV_TEAM][RDV_TEAM_ROW];
    const int team = threadIdx.x / RDV_TEAM;
    const int64_t i_raw = (int64_t)blockIdx.x * (128 / RDV_TEAM) + team;
    const int64_t i = i_raw < n ? i_raw : n - 1;
    const bool valid = i_raw < n && (!mask || mask[i]);
    team_reset(params_of<TABLE>(Pc, S, i), S, seed, env_offset + i, i, valid, bump, uniforms ? uniforms + RDV_N_UNIFORMS * i : nullptr,
               s_team[team], obs ? obs + RDV_OBS_DIM * i : nullptr);
}

template <bool TABLE>
__global__ void __launch_bounds__(128) observe_kernel(const __grid_constant__ RdvParams Pc, const RdvState S,
                                                      float *obs, int64_t n)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const RdvParams &P = params_of<TABLE>(Pc, S, i);
    EnvRegs e;
    load_env(S, i, e);
    float ov[RDV_OBS_DIM];
    make_obs(e, obs_scale(P), ov);
#pragma unroll
    for (int k = 0; k < RDV_OBS_DIM; ++k) obs[RDV_OBS_DIM * i + k] = ov[k];
}

// get_errors / check_collision / check_success / dist_from_koz for evaluators
template <bool TABLE>
__global__ void __launch_bounds__(128) errors_kernel(const __grid_constant__ RdvParams Pc, const RdvState S,
                                                     double *errors, uint8_t *collision, uint8_t *success,
                                                     double *koz, int64_t n, int refresh_flags)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const RdvParams &P = params_of<TABLE>(Pc, S, i);
    EnvRegs e;
    load_env(S, i, e);
    const Rot Rc = rot_from_quat(e.qc), Rt = rot_from_quat(e.qt);
    const double rc_sq = dot3(e.rc, e.rc), rc_n = sqrt(rc_sq);      // evaluator path: IEEE sqrt, values are returned
    const double att = attitude_error(P, e, Rc, rc_sq);
    const double th = corridor_angle(P, e, Rt, rc_sq);
    const bool col = rc_n < P.koz_radius && th > P.corridor_half_angle;
    ErrSq es = errors_sq(P, e, Rc, Rt);
    const double pe = sqrt(es.pos), ve = sqrt(es.vel), re = sqrt(es.rot);
    const bool within = pe <= P.max_rd_error && ve <= P.max_vd_error && att <= P.max_qd_error && re <= P.max_wd_error;
    if (refresh_flags) {
        S.i32[RDV_I_COLLIDED * S.ld + i] = col ? 1 : 0;
        S.i32[RDV_I_SUCCESS * S.ld + i] = (!col && within) ? 1 : 0;
        return;
    }
    const int sticky = S.i32[RDV_I_COLLIDED * S.ld + i];
    if (errors) { errors[4 * i] = pe; errors[4 * i + 1] = ve; errors[4 * i + 2] = att; errors[4 * i + 3] = re; }
    if (collision) collision[i] = col ? 1 : 0;
    if (success) success[i] = (!sticky && within) ? 1 : 0;
    if (koz) koz[i] = koz_distance(P, rc_n, th);
}

// chaser2lvlh / target2lvlh / lvlh2chaser / lvlh2target for evaluators (rendezvous_env.py:470-508)
__global__ void __launch_bounds__(128) frame_kernel(const double *q, const double *v, double *out, int64_t n,
                                                    int transpose)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double qq[4] = {q[4 * i], q[4 * i + 1], q[4 * i + 2], q[4 * i + 3]};
    const double vv[3] = {v[3 * i], v[3 * i + 1], v[3 * i + 2]};
    double o[3];
    const Rot R = rot_from_quat(qq);
    if (transpose) rot_apply_T(R, vv, o); else rot_apply(R, vv, o);
    out[3 * i] = o[0]; out[3 * i + 1] = o[1]; out[3 * i + 2] = o[2];
}

// ---------------------------------------------------------------------------------
// fp32 MLP policy forward, 17 -> 64 -> 64 -> 6 with tanh (SB3 MlpPolicy, main.py:39-48);
// deterministic action = clip(mean, -1, 1) (monte_carlo.py:128-133).  One thread per env, fp32
// FFMA with sequential accumulation over the input index (the order torch's CPU kernel is
// compared against to ~1e-6); weights are staged in shared memory once per CTA.
// ---------------------------------------------------------------------------------
constexpr int PH = 64;
constexpr int PTPB = 128;
__global__ void __launch_bounds__(PTPB) policy_kernel(const RdvPolicy pi, const float *obs, float *actions, int64_t n)
{
    extern __shared__ __align__(16) float sm[];
    float *w0 = sm, *w1 = w0 + PH * 17, *w2 = w1 + PH * PH, *b0 = w2 + 6 * PH, *b1 = b0 + PH, *b2 = b1 + PH;
    float *hid = b2 + 8;                               // [PH][PTPB] hidden activations, column per thread
    for (int k = threadIdx.x; k < PH * 17; k += PTPB) w0[k] = pi.w0[k];
    for (int k = threadIdx.x; k < PH * PH; k += PTPB) w1[k] = pi.w1[k];
    for (int k = threadIdx.x; k < 6 * PH; k += PTPB) w2[k] = pi.w2[k];
    for (int k = threadIdx.x; k < PH; k += PTPB) { b0[k] = pi.b0[k]; b1[k] = pi.b1[k]; }
    if (threadIdx.x < 6) b2[threadIdx.x] = pi.b2[threadIdx.x];
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * PTPB + threadIdx.x;
    if (i >= n) return;
    float x[17];
#pragma unroll
    for (int k = 0; k < 17; ++k) x[k] = obs[17 * i + k];
    float h[PH];
#pragma unroll
    for (int j = 0; j < PH; ++j) {
        float acc = b0[j];
#pragma unroll
        for (int k = 0; k < 17; ++k) acc = fmaf(w0[j * 17 + k], x[k], acc);
        h[j] = tanhf(acc);
    }
#pragma unroll 1
    for (int j = 0; j < PH; ++j) {
        float acc = b1[j];
        const float4 *wr = reinterpret_cast<const float4 *>(w1 + j * PH);
#pragma unroll
        for (int k4 = 0; k4 < PH / 4; ++k4) {
            float4 w = wr[k4];
            acc = fmaf(w.x, h[4 * k4], acc); acc = fmaf(w.y, h[4 * k4 + 1], acc);
            acc = fmaf(w.z, h[4 * k4 + 2], acc); acc = fmaf(w.w, h[4 * k4 + 3], acc);
        }
        hid[j * PTPB + threadIdx.x] = tanhf(acc);
    }
#pragma unroll
    for (int k = 0; k < PH; ++k) h[k] = hid[k * PTPB + threadIdx.x];
#pragma unroll
    for (int j = 0; j < 6; ++j) {
        float acc = b2[j];
#pragma unroll
        for (int k = 0; k < PH; ++k) acc = fmaf(w2[j * PH + k], h[k], acc);
        actions[6 * i + j] = fminf(1.0f, fmaxf(-1.0f, acc));
    }
}

// element-wise evaluation of the device math helpers, for tests/test_gpu_math.py
__global__ void math_probe_kernel(const double *x, double *y, int64_t n, int op)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double v = x[i];
    double r;
    switch (op) {
        case 0: r = fast_rsqrt(v); break;
        case 1: r = fast_rcp(v); break;
        case 2: r = fast_sqrt(v); break;
        case 3: r = pow_neg_tenth(v); break;
        case 4: r = (double)pow_neg_tenth_f32((float)v); break;
        case 5: r = rounded_angle_from(v, 1.0, 1.0); break;       // acos(round(v, 5))
        default: {
            // the attempted plane step at x = v = s^2 > 0: P, Q, R, I of rdv_plane_poly.h (ops 6-9), and the same
            // four quantities from the stagewise attempt at (a, b, g, om2, h) = (1, 0, 1, 1, sqrt(x)) (ops 10-13)
            double P, Q, R, I;
            if (op < 10) {
                plane_poly(v, P, Q, R, I);
            } else {
                const double h = sqrt(v);
                plane_attempt<false>(1.0, 0.0, 1.0, 1.0, h, P, Q, R, I);
                Q /= h; R /= v * v * v; I /= h * v * v;
            }
            const int k = (op - 6) & 3;
            r = k == 0 ? P : k == 1 ? Q : k == 2 ? R : I;
            break;
        }
    }
    y[i] = r;
}

// DFMA-saturating probe for the measured fp64 peak (16 independent accumulators per thread)
__global__ void fp64_peak_kernel(double *sink, int iters)
{
    double a[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = 1.0 + 1e-9 * (threadIdx.x + k);
    const double m = 1.0 + 1e-12 * threadIdx.x, c = 1e-15;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < 16; ++k) a[k] = fma(a[k], m, c);
    }
    double s = 0.0;
#pragma unroll
    for (int k = 0; k < 16; ++k) s += a[k];
    sink[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = s;
}

}  // namespace rdv

// =====================================================================================
// C ABI
// =====================================================================================
using namespace rdv;

static int check_state(const RdvState *s, int64_t n)
{
    if (!s || !s->f64 || !s->i32) return RDV_ERR_NULL;
    if (n < 0 || s->ld < n) return RDV_ERR_SIZE;
    if (((uintptr_t)s->f64 & 7) || ((uintptr_t)s->i32 & 3)) return RDV_ERR_ALIGN;
    if (s->param_table && !s->param_block) return RDV_ERR_NULL;
    if (((uintptr_t)s->param_table & 7) || ((uintptr_t)s->param_block & 3)) return RDV_ERR_ALIGN;
    return RDV_OK;
}
static int launch_status()
{
    cudaError_t e = cudaGetLastError();
    return e == cudaSuccess ? RDV_OK : RDV_ERR_CUDA;
}

// Per-device facts, keyed by the CUDA device ordinal: one process may drive several GPUs, and both the SM count
// and cudaFuncSetAttribute(MaxDynamicSharedMemorySize) are per device.
constexpr int RDV_MAX_DEVICES = 64;
static std::atomic<int> g_sm_count[RDV_MAX_DEVICES];
static int current_device(int *sm_count)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= RDV_MAX_DEVICES) return -1;
    int sms = g_sm_count[dev].load(std::memory_order_relaxed);
    if (sms == 0) {
        if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0) return -1;
        g_sm_count[dev].store(sms, std::memory_order_relaxed);
    }
    *sm_count = sms;
    return dev;
}
// opt a kernel into `bytes` of dynamic shared memory once per device (mask: one bit per device, per kernel)
template <class K>
static bool ensure_smem(K kernel, std::atomic<uint64_t> &mask, int dev, size_t bytes)
{
    const uint64_t bit = 1ull << dev;
    if (mask.load(std::memory_order_acquire) & bit) return true;
    if (cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes) != cudaSuccess) return false;
    mask.fetch_or(bit, std::memory_order_release);
    return true;
}

// The angle table of rounded_angle_from (rdv_math.cuh), filled once per device before the first kernel that reads it.
// The fill runs on the caller's stream and is waited for (once per device and process), so that launches on other
// streams find it complete; a stream that is being captured into a graph cannot be waited for -- the first call on a
// device has to come from outside a capture (any reset / step / rollout does).
__global__ void acos_table_kernel()
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= 2 * ACOS_TABLE_HALF) g_acos_table[i] = acos_of_rounded((double)(i - ACOS_TABLE_HALF));
}
static bool ensure_tables(cudaStream_t st)
{
    static std::atomic<uint64_t> mask{0};
    static std::mutex mtx;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= RDV_MAX_DEVICES) return false;
    const uint64_t bit = 1ull << dev;
    if (mask.load(std::memory_order_acquire) & bit) return true;
    std::lock_guard<std::mutex> lock(mtx);
    if (mask.load(std::memory_order_acquire) & bit) return true;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) != cudaSuccess || cap != cudaStreamCaptureStatusNone) return false;
    acos_table_kernel<<<(2 * ACOS_TABLE_HALF + 256) / 256, 256, 0, st>>>();
    if (cudaGetLastError() != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess) return false;
    mask.fetch_or(bit, std::memory_order_release);
    return true;
}

// development / test knobs: the environment variables are read once, rdv_tune changes them at run time
static int env_int(const char *name, int fallback)
{
    const char *v = getenv(name);
    return v ? atoi(v) : fallback;
}
static std::atomic<int> g_tune_tpb{env_int("RDV_ROLLOUT_TPB", 0)};
static std::atomic<int> g_tune_refill{env_int("RDV_RESET_REFILL", 12)};
static std::atomic<int> g_tune_pdl{env_int("RDV_ROLLOUT_PDL", 1)};
static std::atomic<int> g_tune_helpers{env_int("RDV_ROLLOUT_HELPERS", 1)};

extern "C" {

int rdv_abi_version(void) { return RDV_ABI_VERSION; }

int rdv_tune(int key, int value)
{
    if (key == RDV_TUNE_ROLLOUT_TPB) return g_tune_tpb.exchange(value);
    if (key == RDV_TUNE_RESET_REFILL) return g_tune_refill.exchange(value);
    if (key == RDV_TUNE_ROLLOUT_PDL) return g_tune_pdl.exchange(value);
    if (key == RDV_TUNE_ROLLOUT_HELPERS) return g_tune_helpers.exchange(value);
    return RDV_ERR_SIZE;
}
int rdv_sizeof_params(void) { return (int)sizeof(RdvParams); }
int rdv_sizeof(int which)
{
    switch (which) {
        case 0: return (int)sizeof(RdvParams);
        case 1: return (int)sizeof(RdvState);
        case 2: return (int)sizeof(RdvStepIO);
        case 3: return (int)sizeof(RdvRolloutIO);
        case 4: return (int)sizeof(RdvPolicy);
        case 5: return (int)sizeof(RdvFinishedRow);
        default: return -1;
    }
}

const char *rdv_strerror(int status)
{
    switch (status) {
        case RDV_OK: return "ok";
        case RDV_ERR_NULL: return "required pointer is NULL";
        case RDV_ERR_SIZE: return "bad size, leading dimension or enum value";
        case RDV_ERR_ALIGN: return "pointer not aligned for vector access";
        case RDV_ERR_PARAMS: return "invalid environment parameters";
        case RDV_ERR_CUDA: return "CUDA launch/runtime failure (is a B200 visible?)";
        case RDV_ERR_UNSUPPORTED: return "unsupported configuration";
        default: return "unknown status";
    }
}

void rdv_params_default(RdvParams *p)
{
    memset(p, 0, sizeof(*p));
    const double rad = M_PI / 180.0;
    p->rc0[1] = -10.0; p->qc0[0] = 1.0; p->qt0[0] = 1.0;
    p->rc0_range = 1; p->vc0_range = 0.1; p->qc0_range = 1 * rad; p->wc0_range = 0.1 * rad;
    p->qt0_range = 45 * rad; p->wt0_range = 3 * rad;
    p->koz_radius = 5; p->corridor_half_angle = 30 * rad; p->h = 800e3; p->dt = 1; p->t_max = 120;
    p->collision_coef = 0.5; p->bonus_coef = 8; p->fuel_coef = 0.2; p->att_coef = 1;
    const double diag = 1.0 * 1 / 12 * 100 * 2;        // eye * 1/12 * m * (2*1**2), left to right
    for (int i = 0; i < 3; ++i) { p->inertia_c[4 * i] = diag; p->inertia_t[4 * i] = diag; }
    p->integrator = RDV_INTEGRATOR_RK45;
}

static int invert3(const double *m, double *o)
{
    double c00 = m[4] * m[8] - m[5] * m[7], c01 = m[5] * m[6] - m[3] * m[8], c02 = m[3] * m[7] - m[4] * m[6];
    double det = m[0] * c00 + m[1] * c01 + m[2] * c02;
    if (!(fabs(det) > 0.0)) return -1;
    bool diag = m[1] == 0 && m[2] == 0 && m[3] == 0 && m[5] == 0 && m[6] == 0 && m[7] == 0;
    if (diag) {
        for (int i = 0; i < 9; ++i) o[i] = 0.0;
        o[0] = 1.0 / m[0]; o[4] = 1.0 / m[4]; o[8] = 1.0 / m[8];
        return 0;
    }
    o[0] = c00 / det; o[1] = (m[2] * m[7] - m[1] * m[8]) / det; o[2] = (m[1] * m[5] - m[2] * m[4]) / det;
    o[3] = c01 / det; o[4] = (m[0] * m[8] - m[2] * m[6]) / det; o[5] = (m[2] * m[3] - m[0] * m[5]) / det;
    o[6] = c02 / det; o[7] = (m[1] * m[6] - m[0] * m[7]) / det; o[8] = (m[0] * m[4] - m[1] * m[3]) / det;
    return 0;
}
static int is_isotropic(const double *m, const double *tau)
{
    bool off = m[1] == 0 && m[2] == 0 && m[3] == 0 && m[5] == 0 && m[6] == 0 && m[7] == 0;
    bool eq = m[0] == m[4] && m[4] == m[8];
    bool t0 = !tau || (tau[0] == 0 && tau[1] == 0 && tau[2] == 0);
    return off && eq && t0;
}

int rdv_params_derive(RdvParams *p)
{
    if (!p) return RDV_ERR_NULL;
    const double rad = M_PI / 180.0;
    const double nominal_diag = 1.0 * 1 / 12 * 100 * 2;
    if (invert3(p->inertia_c, p->inv_inertia_c) || invert3(p->inertia_t, p->inv_inertia_t)) return RDV_ERR_PARAMS;
    p->max_delta_v = 10.0 / 100 * 0.5;                                   // rendezvous_env.py:81
    p->max_delta_w = 0.2 / nominal_diag * 0.5;                           // :82
    p->max_axial_distance = sqrt(p->rc0[0] * p->rc0[0] + p->rc0[1] * p->rc0[1] + p->rc0[2] * p->rc0[2]) + 10;  // :85
    p->max_axial_speed = 5; p->max_wc = 10 * rad; p->max_attitude_error = 30 * rad;   // :86-89
    p->max_rd_error = 0.5; p->max_vd_error = 0.1; p->max_qd_error = 5 * rad; p->max_wd_error = 1 * rad;  // :105-108
    p->rd[0] = 0; p->rd[1] = -2; p->rd[2] = 0;                           // :104
    p->capture_axis[0] = 0; p->capture_axis[1] = 1; p->capture_axis[2] = 0;        // :73
    p->corridor_axis[0] = 0; p->corridor_axis[1] = -1; p->corridor_axis[2] = 0;    // :95
    p->bubble0 = p->max_axial_distance;                                  // :113
    p->bubble_rate = 0.5 * p->dt;                                        // :114
    const double rd_n = 2.0;
    p->bubble_min = rd_n + 2 * p->max_rd_error;                          // :115
    const double ro = 6371e3 + p->h;
    p->n = sqrt(3.986004418e14 / (ro * ro * ro));                        // :122-126
    if (!(rd_n < p->koz_radius) || !(rd_n - p->max_rd_error > 0)) return RDV_ERR_PARAMS;   // :155-156
    if (!(p->dt > 0) || !(p->t_max > 0)) return RDV_ERR_PARAMS;
    // t = round(t + dt, 3) each step (:193) is reproduced as round(step * dt, 3), which is the same number only
    // when dt lies on the 1 ms grid the reference rounds to
    if (fabs(p->dt * 1000.0 - rint(p->dt * 1000.0)) > 1e-9 * p->dt * 1000.0) return RDV_ERR_UNSUPPORTED;
    // CW transition matrix, non-zero entries row by row (utils/dynamics.py:40-47)
    const double n = p->n, nt = n * p->dt, s = sin(nt), c = cos(nt);
    double *w = p->cw;
    w[0] = 4 - 3 * c;          w[1] = 1 / n * s;            w[2] = 2 / n * (1 - c);
    w[3] = 6 * (s - nt);       w[4] = 1;                    w[5] = -2 / n * (1 - c);  w[6] = 1 / n * (4 * s - 3 * nt);
    w[7] = c;                  w[8] = 1 / n * s;
    w[9] = 3 * n * s;          w[10] = c;                   w[11] = 2 * s;
    w[12] = -6 * n * (1 - c);  w[13] = -2 * s;              w[14] = 4 * c - 3;
    w[15] = -n * s;            w[16] = c;
    p->max_delta_v_f32 = (float)p->max_delta_v;
    p->fuel_num_f32 = (float)(p->dt * p->fuel_coef);
    p->fuel_den_f32 = (float)(3 * p->max_delta_v);
    p->inv_max_attitude_error = 1.0 / p->max_attitude_error;
    p->inv_max_rd_error = 1.0 / p->max_rd_error;
    p->inv_max_qd_error = 1.0 / p->max_qd_error;
    p->koz_radius_sq = p->koz_radius * p->koz_radius;
    p->max_rd_error_sq = p->max_rd_error * p->max_rd_error;
    p->max_vd_error_sq = p->max_vd_error * p->max_vd_error;
    p->max_wd_error_sq = p->max_wd_error * p->max_wd_error;
    p->fuel_scale = p->dt * p->fuel_coef / (3 * p->max_delta_v);
    p->att_scale = p->dt * p->att_coef;
    p->bonus_scale = p->dt * p->bonus_coef;
    p->collision_scale = p->dt * p->collision_coef;
    p->obs_inv_r = 1.0 / (2.0 * p->max_axial_distance);
    p->obs_inv_v = 1.0 / (2.0 * p->max_axial_speed);
    p->obs_inv_w = 1.0 / (2.0 * p->max_wc);
    {   // high words of hi * (1 - 1e-6): a state entry whose |x| has a smaller high word maps into the Box for sure
        auto hiword = [](double x) { uint64_t b; memcpy(&b, &x, 8); return (int32_t)((b >> 32) & 0x7fffffffu); };
        p->box_hi_r = hiword(p->max_axial_distance * (1.0 - 1e-6));
        p->box_hi_v = hiword(p->max_axial_speed * (1.0 - 1e-6));
        p->box_hi_w = hiword(p->max_wc * (1.0 - 1e-6));
        p->reserved1 = 0;
    }
    {
        const double reach = rd_n + p->max_rd_error, lim = reach > p->koz_radius ? reach : p->koz_radius;
        p->near_sq = lim * lim * (1.0 + 1e-9);
    }
    {   // first step count whose time stamp t = round(k*dt, 3) reaches t_max (:193, :369)
        double k = ceil(p->t_max / p->dt) - 2.0;
        if (k < 1.0) k = 1.0;
        while (rint(k * p->dt * 1000.0) / 1000.0 < p->t_max) k += 1.0;
        if (k > 2147483647.0) return RDV_ERR_PARAMS;
        p->done_steps = (int32_t)k;
    }
    p->iso_c = is_isotropic(p->inertia_c, p->torque_c);
    p->iso_t = is_isotropic(p->inertia_t, nullptr);
    if (p->integrator != RDV_INTEGRATOR_RK45 && p->integrator != RDV_INTEGRATOR_CLOSED_FORM) return RDV_ERR_SIZE;
    if (p->integrator == RDV_INTEGRATOR_CLOSED_FORM && !(p->iso_c && p->iso_t)) return RDV_ERR_UNSUPPORTED;
    return RDV_OK;
}

int rdv_step(const RdvParams *p, const RdvState *s, const RdvStepIO *io, int64_t n, uint64_t seed,
             int64_t env_offset, void *cuda_stream)
{
    if (!p || !io || !io->actions || !io->obs || !io->reward || !io->done) return RDV_ERR_NULL;
    int rc = check_state(s, n);
    if (rc) return rc;
    if (n == 0) return RDV_OK;
    if (((uintptr_t)io->actions & (io->act_f64 ? 15 : 7)) || ((uintptr_t)io->obs & 15) || ((uintptr_t)io->reward & 7))
        return RDV_ERR_ALIGN;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const unsigned grid = (unsigned)((n + EPB - 1) / EPB);
    const bool iso = p->iso_c && p->iso_t;
    const bool closed = p->integrator == RDV_INTEGRATOR_CLOSED_FORM;
    if (io->auto_reset != 0 && io->auto_reset != 1) return RDV_ERR_SIZE;
    if (io->fin_rows) {
        if (!io->fin_count) return RDV_ERR_NULL;
        if (io->fin_capacity < 0) return RDV_ERR_SIZE;
        if (((uintptr_t)io->fin_rows & 15) || ((uintptr_t)io->fin_count & 3)) return RDV_ERR_ALIGN;
        if (!io->fin_append && cudaMemsetAsync(io->fin_count, 0, sizeof(int32_t), st) != cudaSuccess) return RDV_ERR_CUDA;
    }
    if ((uintptr_t)io->reward_f32 & 3) return RDV_ERR_ALIGN;
    if (!ensure_tables(st)) return RDV_ERR_CUDA;
#define RDV_LAUNCH(ISO_, F64_, CL_) \
    step_kernel<ISO_, F64_, CL_><<<grid, TPB, 0, st>>>(*p, *s, *io, n, seed, env_offset)
    if (s->param_table) {
        if (!iso || closed) return RDV_ERR_UNSUPPORTED;      // parameter tables: the reference's bodies, RK45
        if (io->act_f64) step_kernel<true, true, false, true><<<grid, TPB, 0, st>>>(*p, *s, *io, n, seed, env_offset);
        else step_kernel<true, false, false, true><<<grid, TPB, 0, st>>>(*p, *s, *io, n, seed, env_offset);
    }
    else if (closed) { if (io->act_f64) RDV_LAUNCH(true, true, true); else RDV_LAUNCH(true, false, true); }
    else if (iso) { if (io->act_f64) RDV_LAUNCH(true, true, false); else RDV_LAUNCH(true, false, false); }
    else { if (io->act_f64) RDV_LAUNCH(false, true, false); else RDV_LAUNCH(false, false, false); }
#undef RDV_LAUNCH
    return launch_status();
}

// rdv_rollout (traj NULL) and rdv_rollout_trajectory (traj checked by the caller)
static int rollout_launch(const RdvParams *p, const RdvState *s, const RdvRolloutIO *io, double *traj, int64_t n,
                          uint64_t seed, int64_t env_offset, void *cuda_stream)
{
    if (!p || !io || !io->obs) return RDV_ERR_NULL;
    int rc = check_state(s, n);
    if (rc) return rc;
    if (io->steps < 0 || io->action_source < 0 || io->action_source > RDV_ACTIONS_POLICY_SAMPLE) return RDV_ERR_SIZE;
    if (io->auto_reset != 0 && io->auto_reset != 1) return RDV_ERR_SIZE;
    const bool policy = io->action_source == RDV_ACTIONS_POLICY || io->action_source == RDV_ACTIONS_POLICY_SAMPLE;
    const bool ptab = io->policy_table != nullptr;
    if (ptab) {
        // policy tables: the fused actor only; entries are checked by the caller (hidden = 64, log_std for sampling)
        if (!policy) return RDV_ERR_SIZE;
        if (!io->policy_tile) return RDV_ERR_NULL;
        if (io->policy_count < 1) return RDV_ERR_SIZE;
        if (((uintptr_t)io->policy_table & 7) || ((uintptr_t)io->policy_tile & 3)) return RDV_ERR_ALIGN;
        if (!(p->iso_c && p->iso_t) || p->integrator == RDV_INTEGRATOR_CLOSED_FORM) return RDV_ERR_UNSUPPORTED;
    } else if (policy) {
        const RdvPolicy *pi = &io->policy;
        if (io->action_source == RDV_ACTIONS_POLICY_SAMPLE && !pi->log_std) return RDV_ERR_NULL;
        if (!pi->w0 || !pi->b0 || !pi->w1 || !pi->b1 || !pi->w2 || !pi->b2) return RDV_ERR_NULL;
        if (pi->hidden != PI_H) return RDV_ERR_UNSUPPORTED;
    } else if (io->action_source != RDV_ACTIONS_PHILOX && !io->actions) return RDV_ERR_NULL;
    if (((uintptr_t)io->actions & (io->action_source == RDV_ACTIONS_F64 ? 15 : 7)) || ((uintptr_t)io->actions_out & 15) ||
        ((uintptr_t)io->obs & 3) || ((uintptr_t)io->rewards & 7))
        return RDV_ERR_ALIGN;
    if (n == 0 || io->steps == 0) return RDV_OK;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const bool iso = p->iso_c && p->iso_t;
    const bool closed = p->integrator == RDV_INTEGRATOR_CLOSED_FORM;
    // one CTA per SM; the CTA size is the smallest instantiated one that covers a slice in the fewest passes
    int sm_count = 0;
    const int dev = current_device(&sm_count);
    if (dev < 0 || !ensure_tables(st)) return RDV_ERR_CUDA;
    if (io->sm_reserve < 0 || io->sm_reserve >= sm_count) return RDV_ERR_SIZE;
    const int64_t sms = sm_count - io->sm_reserve;
    const int64_t grid = n < sms ? n : sms;
    const int64_t per_cta = (n + grid - 1) / grid;
    const bool mc = io->mc_out != nullptr;
    if (mc && (io->auto_reset || ((uintptr_t)io->mc_out & 7))) return io->auto_reset ? RDV_ERR_UNSUPPORTED : RDV_ERR_ALIGN;
    if ((uintptr_t)io->reset_rows & 7) return RDV_ERR_ALIGN;
    // development / test override of the CTA size (rdv_tune): 256 | 384 | 448 | 512; the evaluator mode has one size
    const bool table = s->param_table != nullptr;
    const int force_tpb = (mc || table || ptab) ? 256 : g_tune_tpb.load(std::memory_order_relaxed);
    const int64_t max_tpb = force_tpb > 0 ? force_tpb : 512;
    const int64_t passes = (per_cta + max_tpb - 1) / max_tpb;
    const int64_t chunk = force_tpb > 0 ? force_tpb : (per_cta + passes - 1) / passes;
    // reset prefetch period (steps between refills of the per-lane reset rows; 0 = reset on demand only)
    RdvRolloutIO io_k = *io;
    io_k.reserved = g_tune_refill.load(std::memory_order_relaxed);
    if (io_k.reserved < 0 || io_k.reserved > 64) io_k.reserved = 0;
#define RDV_LAUNCH_K(KERNEL, T_, SMEM)                                                                            \
    {                                                                                                             \
        static std::atomic<uint64_t> attr_mask{0};                                                                \
        if (!ensure_smem(KERNEL, attr_mask, dev, SMEM)) return RDV_ERR_CUDA;                                      \
        if (g_tune_pdl.load(std::memory_order_relaxed)) {                                                         \
            cudaLaunchConfig_t cfg = {};                                                                          \
            cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(T_); cfg.dynamicSmemBytes = SMEM; cfg.stream = st; \
            cudaLaunchAttribute at[1];                                                                            \
            at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                                        \
            at[0].val.programmaticStreamSerializationAllowed = 1;                                                 \
            cfg.attrs = at; cfg.numAttrs = 1;                                                                     \
            if (cudaLaunchKernelEx(&cfg, KERNEL, *p, *s, io_k, n, seed, env_offset, traj) != cudaSuccess) {       \
                cudaGetLastError();                                                                               \
                return RDV_ERR_CUDA;                                                                              \
            }                                                                                                     \
        } else {                                                                                                  \
            KERNEL<<<(unsigned)grid, T_, SMEM, st>>>(*p, *s, io_k, n, seed, env_offset, traj);                    \
        }                                                                                                         \
    }
#define RDV_ROWS_SMEM(T_) ((size_t)(T_ / 32) * 32 * RDV_NEXT_ROW * sizeof(double))
#define RDV_LAUNCH_R(ISO_, CL_, T_) RDV_LAUNCH_K((rollout_kernel<ISO_, CL_, T_, false, false>), T_, RDV_ROWS_SMEM(T_))
    // per-step observation records: one CTA shape with the observation formed every step (every shape gives the same bits)
#define RDV_LAUNCH_OBS(ISO_, CL_) \
    RDV_LAUNCH_K((rollout_kernel<ISO_, CL_, 256, false, false, false, true>), 256, RDV_ROWS_SMEM(256))
    // 14 worker warps + 2 helper warps (see rollout_kernel): single-pass launches of the 448-env shape with auto-reset
    const bool helpers = g_tune_helpers.load(std::memory_order_relaxed) && io->auto_reset && io_k.reserved > 0 &&
                         (io_k.reset_rows != nullptr || io->steps >= 2 * io_k.reserved) &&
                         passes == 1 && chunk > 384 && chunk <= 448;
#define RDV_LAUNCH_H(ISO_, CL_) \
    RDV_LAUNCH_K((rollout_kernel<ISO_, CL_, 448, false, false, false, false, true>), 512, RDV_ROWS_SMEM(448))
#define RDV_PICK_R(ISO_, CL_)                                 \
    if (io->obs_steps) RDV_LAUNCH_OBS(ISO_, CL_)              \
    else if (chunk <= 256) RDV_LAUNCH_R(ISO_, CL_, 256)       \
    else if (chunk <= 384) RDV_LAUNCH_R(ISO_, CL_, 384)       \
    else if (chunk <= 448) { if (helpers && ISO_ && !CL_) RDV_LAUNCH_H(true, false) else RDV_LAUNCH_R(ISO_, CL_, 448) } \
    else RDV_LAUNCH_R(ISO_, CL_, 512)
#define RDV_LAUNCH_P(T_) RDV_LAUNCH_K((rollout_kernel<true, false, T_, true, false>), T_, sizeof(tc::TileSmem))
#define RDV_LAUNCH_PT(MC_, TABLE_) \
    RDV_LAUNCH_K((rollout_kernel<true, false, 256, true, MC_, TABLE_, true, false, true>), 256, sizeof(tc::TableSmem))
    // trajectory records: one CTA shape per configuration, with the observation formed every step (as for obs_steps)
#define RDV_LAUNCH_T(ISO_, CL_, POLICY_, MC_, TABLE_, PTAB_)                                                       \
    RDV_LAUNCH_K((rollout_kernel<ISO_, CL_, 256, POLICY_, MC_, TABLE_, true, false, PTAB_, true>), 256,            \
                 PTAB_ ? sizeof(tc::TableSmem) : POLICY_ ? sizeof(tc::TileSmem) : RDV_ROWS_SMEM(256))
    // the policy-table variants are instantiated after all others, and the trajectory variants after those: ptxas
    // handles a module's kernels in that order, and with them first the register allocation of an existing variant
    // (POLICY + TABLE) came out differently
    if (!ptab && !traj) {
        if (table) {
            if (!iso || closed) return RDV_ERR_UNSUPPORTED;      // parameter tables: the reference's bodies, RK45
            if (mc && policy) RDV_LAUNCH_K((rollout_kernel<true, false, 256, true, true, true>), 256, sizeof(tc::TileSmem))
            else if (mc) RDV_LAUNCH_K((rollout_kernel<true, false, 256, false, true, true, true>), 256, RDV_ROWS_SMEM(256))
            else if (policy) RDV_LAUNCH_K((rollout_kernel<true, false, 256, true, false, true>), 256, sizeof(tc::TileSmem))
            else RDV_LAUNCH_K((rollout_kernel<true, false, 256, false, false, true, true>), 256, RDV_ROWS_SMEM(256))
        }
        else if (mc) {
            if (!iso || closed) return RDV_ERR_UNSUPPORTED;      // the evaluator mode is built for the reference's env
            if (policy) RDV_LAUNCH_K((rollout_kernel<true, false, 256, true, true>), 256, sizeof(tc::TileSmem))
            else RDV_LAUNCH_K((rollout_kernel<true, false, 256, false, true, false, true>), 256, RDV_ROWS_SMEM(256))
        }
        else if (policy) {
            if (!iso || closed) return RDV_ERR_UNSUPPORTED;      // the fused policy is built for the reference's env
            if (chunk <= 256) RDV_LAUNCH_P(256)
            else if (chunk <= 384) RDV_LAUNCH_P(384)
            else if (chunk <= 448) RDV_LAUNCH_P(448)
            else RDV_LAUNCH_P(512)
        }
        else if (closed) { RDV_PICK_R(true, true) }
        else if (iso) { RDV_PICK_R(true, false) }
        else RDV_LAUNCH_OBS(false, false)                          // general inertia / held torque: one shape
    } else if (!traj) {                                         // (bodies and integrator checked above)
        if (mc && table) RDV_LAUNCH_PT(true, true)
        else if (mc) RDV_LAUNCH_PT(true, false)
        else if (table) RDV_LAUNCH_PT(false, true)
        else RDV_LAUNCH_PT(false, false)
    } else {
        // the configurations rdv_rollout accepts, each in its one trajectory variant
        if ((table || mc || policy) && (!iso || closed)) return RDV_ERR_UNSUPPORTED;
        if (ptab) {
            if (mc && table) RDV_LAUNCH_T(true, false, true, true, true, true)
            else if (mc) RDV_LAUNCH_T(true, false, true, true, false, true)
            else if (table) RDV_LAUNCH_T(true, false, true, false, true, true)
            else RDV_LAUNCH_T(true, false, true, false, false, true)
        } else if (table) {
            if (mc && policy) RDV_LAUNCH_T(true, false, true, true, true, false)
            else if (mc) RDV_LAUNCH_T(true, false, false, true, true, false)
            else if (policy) RDV_LAUNCH_T(true, false, true, false, true, false)
            else RDV_LAUNCH_T(true, false, false, false, true, false)
        } else if (mc) {
            if (policy) RDV_LAUNCH_T(true, false, true, true, false, false)
            else RDV_LAUNCH_T(true, false, false, true, false, false)
        }
        else if (policy) RDV_LAUNCH_T(true, false, true, false, false, false)
        else if (closed) RDV_LAUNCH_T(true, true, false, false, false, false)
        else if (iso) RDV_LAUNCH_T(true, false, false, false, false, false)
        else RDV_LAUNCH_T(false, false, false, false, false, false)
    }
#undef RDV_LAUNCH_T
#undef RDV_LAUNCH_OBS
#undef RDV_LAUNCH_P
#undef RDV_LAUNCH_PT
#undef RDV_PICK_R
#undef RDV_LAUNCH_H
#undef RDV_LAUNCH_R
#undef RDV_ROWS_SMEM
#undef RDV_LAUNCH_K
    return launch_status();
}

int rdv_rollout(const RdvParams *p, const RdvState *s, const RdvRolloutIO *io, int64_t n, uint64_t seed,
                int64_t env_offset, void *cuda_stream)
{
    return rollout_launch(p, s, io, nullptr, n, seed, env_offset, cuda_stream);
}

int rdv_rollout_trajectory(const RdvParams *p, const RdvState *s, const RdvRolloutIO *io, double *traj, int64_t n,
                           uint64_t seed, int64_t env_offset, void *cuda_stream)
{
    if (!traj) return RDV_ERR_NULL;
    if ((uintptr_t)traj & 7) return RDV_ERR_ALIGN;
    return rollout_launch(p, s, io, traj, n, seed, env_offset, cuda_stream);
}

int rdv_reset(const RdvParams *p, const RdvState *s, const uint8_t *mask, const double *uniforms, float *obs,
              int64_t n, uint64_t seed, int64_t env_offset, int bump_episode, void *cuda_stream)
{
    if (!p) return RDV_ERR_NULL;
    int rc = check_state(s, n);
    if (rc) return rc;
    if (n == 0) return RDV_OK;
    const int64_t per_cta = 128 / RDV_TEAM;
    const unsigned grid = (unsigned)((n + per_cta - 1) / per_cta);
    if (s->param_table)
        reset_kernel<true><<<grid, 128, 0, (cudaStream_t)cuda_stream>>>(*p, *s, mask, uniforms, obs, n, seed, env_offset,
                                                                        bump_episode ? 1 : 0);
    else
        reset_kernel<false><<<grid, 128, 0, (cudaStream_t)cuda_stream>>>(*p, *s, mask, uniforms, obs, n, seed, env_offset,
                                                                         bump_episode ? 1 : 0);
    return launch_status();
}

int rdv_observe(const RdvParams *p, const RdvState *s, float *obs, int64_t n, void *cuda_stream)
{
    if (!p || !obs) return RDV_ERR_NULL;
    int rc = check_state(s, n);
    if (rc) return rc;
    if (n == 0) return RDV_OK;
    if (s->param_table) observe_kernel<true><<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)cuda_stream>>>(*p, *s, obs, n);
    else observe_kernel<false><<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)cuda_stream>>>(*p, *s, obs, n);
    return launch_status();
}

int rdv_errors(const RdvParams *p, const RdvState *s, double *errors, uint8_t *collision, uint8_t *success,
               double *koz, int64_t n, void *cuda_stream)
{
    if (!p) return RDV_ERR_NULL;
    int rc = check_state(s, n);
    if (rc) return rc;
    if (n == 0) return RDV_OK;
    if (!ensure_tables((cudaStream_t)cuda_stream)) return RDV_ERR_CUDA;
    if (s->param_table)
        errors_kernel<true><<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)cuda_stream>>>(*p, *s, errors, collision,
                                                                                                 success, koz, n, 0);
    else
        errors_kernel<false><<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)cuda_stream>>>(*p, *s, errors, collision,
                                                                                                  success, koz, n, 0);
    return launch_status();
}

int rdv_refresh_flags(const RdvParams *p, const RdvState *s, int64_t n, void *cuda_stream)
{
    if (!p) return RDV_ERR_NULL;
    int rc = check_state(s, n);
    if (rc) return rc;
    if (n == 0) return RDV_OK;
    if (!ensure_tables((cudaStream_t)cuda_stream)) return RDV_ERR_CUDA;
    if (s->param_table)
        errors_kernel<true><<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)cuda_stream>>>(*p, *s, nullptr, nullptr,
                                                                                                 nullptr, nullptr, n, 1);
    else
        errors_kernel<false><<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)cuda_stream>>>(*p, *s, nullptr, nullptr,
                                                                                                  nullptr, nullptr, n, 1);
    return launch_status();
}

int rdv_frame_transform(const double *q, const double *v, double *out, int64_t n, int transpose, void *cuda_stream)
{
    if (!q || !v || !out) return RDV_ERR_NULL;
    if (n < 0) return RDV_ERR_SIZE;
    if (n == 0) return RDV_OK;
    frame_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)cuda_stream>>>(q, v, out, n, transpose);
    return launch_status();
}

int rdv_policy_forward(const RdvPolicy *pi, const float *obs, float *actions, int64_t n, void *cuda_stream)
{
    if (!pi || !obs || !actions || !pi->w0 || !pi->b0 || !pi->w1 || !pi->b1 || !pi->w2 || !pi->b2) return RDV_ERR_NULL;
    if (pi->hidden != tc::H) return RDV_ERR_UNSUPPORTED;
    if (n < 0) return RDV_ERR_SIZE;
    if (n == 0) return RDV_OK;
    int sm_count = 0;
    const int dev = current_device(&sm_count);
    if (dev < 0) return RDV_ERR_CUDA;
    static std::atomic<uint64_t> attr_mask{0};
    if (!ensure_smem(tc::policy_tc_kernel, attr_mask, dev, sizeof(tc::Smem))) return RDV_ERR_CUDA;
    const int64_t tiles = (n + tc::TM - 1) / tc::TM;              // tile t -> CTA t % grid, group (t / grid) % GROUPS
    const unsigned grid = (unsigned)(tiles < sm_count ? tiles : sm_count);
    tc::policy_tc_kernel<<<grid, tc::GROUPS * tc::TM, sizeof(tc::Smem), (cudaStream_t)cuda_stream>>>(*pi, obs, actions, n);
    return launch_status();
}

int rdv_policy_forward_ffma(const RdvPolicy *pi, const float *obs, float *actions, int64_t n, void *cuda_stream)
{
    if (!pi || !obs || !actions || !pi->w0 || !pi->b0 || !pi->w1 || !pi->b1 || !pi->w2 || !pi->b2) return RDV_ERR_NULL;
    if (pi->hidden != PH) return RDV_ERR_UNSUPPORTED;
    if (n < 0) return RDV_ERR_SIZE;
    if (n == 0) return RDV_OK;
    const size_t smem = sizeof(float) * (PH * 17 + PH * PH + 6 * PH + PH + PH + 8 + PH * PTPB);
    int sm_count = 0;
    const int dev = current_device(&sm_count);
    if (dev < 0) return RDV_ERR_CUDA;
    static std::atomic<uint64_t> attr_mask{0};
    if (!ensure_smem(policy_kernel, attr_mask, dev, smem)) return RDV_ERR_CUDA;
    policy_kernel<<<(unsigned)((n + PTPB - 1) / PTPB), PTPB, smem, (cudaStream_t)cuda_stream>>>(*pi, obs, actions, n);
    return launch_status();
}

int rdv_math_probe(const double *x, double *y, int64_t n, int op, void *cuda_stream)
{
    if (!x || !y) return RDV_ERR_NULL;
    if (n < 0 || op < 0 || op > 13) return RDV_ERR_SIZE;
    if (n == 0) return RDV_OK;
    if (!ensure_tables((cudaStream_t)cuda_stream)) return RDV_ERR_CUDA;
    math_probe_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)cuda_stream>>>(x, y, n, op);
    return launch_status();
}

int rdv_fp64_peak_probe(double *sink, int blocks, int threads, int iters, void *cuda_stream)
{
    if (!sink) return RDV_ERR_NULL;
    if (blocks <= 0 || threads <= 0 || threads > 1024 || iters <= 0) return RDV_ERR_SIZE;
    fp64_peak_kernel<<<blocks, threads, 0, (cudaStream_t)cuda_stream>>>(sink, iters);
    return launch_status();
}

}  // extern "C"
