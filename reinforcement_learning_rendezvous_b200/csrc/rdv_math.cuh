// rdv_math.cuh -- device-side fp64 math of the RendezvousEnv hot path for sm_100a.
//
// One thread owns one environment; everything here works on registers.  The
// functions restate reference behaviour (file:line under /root/reference) but are
// written for the B200 fp64 pipe: divisions by run-time values use MUFU seeds +
// FMA refinement (<= 1 ulp), divisions by constants use host-precomputed
// reciprocals, the quaternion normalisation inside the ODE right-hand side is done
// once with an rsqrt, and err**-0.2 of the step-size controller is a MUFU seed +
// two Newton steps instead of a generic pow().  The deviations from the reference's
// operation order are at the 1e-16 level; the parity bar is 1e-9 (BASELINE.json).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "rdv_b200.h"
#include "rdv_plane_poly.h"

#define RDV_DEV __device__ __forceinline__

namespace rdv {

// ---------------------------------------------------------------------------------
// scalar helpers
// ---------------------------------------------------------------------------------
// 1/x for normal positive/negative x: MUFU.RCP64H seed (>= 20 good bits) + 2 Newton steps.
RDV_DEV double fast_rcp(double x)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    double e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    e = fma(-x, r, 1.0);
    r = fma(r, e, r);
    return r;
}

// 1/sqrt(x) for normal positive x: MUFU.RSQ64H seed (>= 20 good bits) + one cubic (Halley-type) step:
// r (1 + e/2 + 3 e^2/8) with e = 1 - x r^2 leaves (5/16) e^3 < 2^-61, i.e. the result is good to the rounding of
// the five operations (<= 2 ulp, checked by tests/test_gpu_math.py).  This sits inside the ODE right-hand side,
// ~45 times per env step.
RDV_DEV double fast_rsqrt(double x)
{
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
    const double m = x * r;
    const double e = fma(-m, r, 1.0);                 // 1 - x r^2
    const double p = fma(0.375, e, 0.5);
    return fma(r * e, p, r);                          // r (1 + e/2 + 3e^2/8)
}

// x**(-0.1) for x in [1e-30, 1e30]: fp32 MUFU.LG2/EX2 seed (rel. err ~1e-6) and two Newton
// steps on y -> y (1 + (1 - x y^10)/10), which converge quadratically (11/2 e^2).
// Used for err_norm**-0.2 with x = err_norm^2 (scipy rk.py:160,170) and for
// (0.01/max(d1,d2))**0.2 (scipy common.py:131) with x = max(d1,d2)^2 / 1e-4.
RDV_DEV double pow_neg_tenth(double x)
{
    if (!(x >= 1e-30 && x <= 1e30)) return pow(x, -0.1);     // cold path, keeps exact semantics
    float lf = __log2f((float)x);
    double y = (double)exp2f(-0.1f * lf);
#pragma unroll
    for (int it = 0; it < 2; ++it) {
        double y2 = y * y, y4 = y2 * y2, y8 = y4 * y4, y10 = y8 * y2;
        double res = fma(-x, y10, 1.0);
        y = fma(y * 0.1, res, y);
    }
    return y;
}

RDV_DEV double dot3(const double a[3], const double b[3]) { return fma(a[2], b[2], fma(a[1], b[1], a[0] * b[0])); }
RDV_DEV double dot4(const double a[4], const double b[4])
{
    return fma(a[3], b[3], fma(a[2], b[2], fma(a[1], b[1], a[0] * b[0])));
}
RDV_DEV void cross3(const double a[3], const double b[3], double o[3])
{
    o[0] = fma(a[1], b[2], -(a[2] * b[1]));
    o[1] = fma(a[2], b[0], -(a[0] * b[2]));
    o[2] = fma(a[0], b[1], -(a[1] * b[0]));
}

// Rotation matrix of quat2mat (utils/quaternions.py:48-68), including its re-normalisation.
struct Rot { double m[9]; };
RDV_DEV Rot rot_from_quat(const double q_in[4])
{
    double r = fast_rsqrt(dot4(q_in, q_in));
    double w = q_in[0] * r, x = q_in[1] * r, y = q_in[2] * r, z = q_in[3] * r;
    double ww = w * w;
    Rot R;
    R.m[0] = fma(2.0, fma(x, x, ww), -1.0); R.m[1] = 2.0 * fma(x, y, -(w * z)); R.m[2] = 2.0 * fma(x, z, w * y);
    R.m[3] = 2.0 * fma(x, y, w * z); R.m[4] = fma(2.0, fma(y, y, ww), -1.0); R.m[5] = 2.0 * fma(y, z, -(w * x));
    R.m[6] = 2.0 * fma(x, z, -(w * y)); R.m[7] = 2.0 * fma(y, z, w * x); R.m[8] = fma(2.0, fma(z, z, ww), -1.0);
    return R;
}
// the same matrix for a quaternion that is already a unit vector (no re-normalisation)
RDV_DEV Rot rot_from_unit_quat(const double q[4])
{
    const double w = q[0], x = q[1], y = q[2], z = q[3];
    const double ww = w * w;
    Rot R;
    R.m[0] = fma(2.0, fma(x, x, ww), -1.0); R.m[1] = 2.0 * fma(x, y, -(w * z)); R.m[2] = 2.0 * fma(x, z, w * y);
    R.m[3] = 2.0 * fma(x, y, w * z); R.m[4] = fma(2.0, fma(y, y, ww), -1.0); R.m[5] = 2.0 * fma(y, z, -(w * x));
    R.m[6] = 2.0 * fma(x, z, -(w * y)); R.m[7] = 2.0 * fma(y, z, w * x); R.m[8] = fma(2.0, fma(z, z, ww), -1.0);
    return R;
}
RDV_DEV void rot_apply(const Rot &R, const double v[3], double o[3])            // body -> LVLH (:490-508)
{
#pragma unroll
    for (int i = 0; i < 3; ++i) o[i] = fma(R.m[3 * i + 2], v[2], fma(R.m[3 * i + 1], v[1], R.m[3 * i] * v[0]));
}
RDV_DEV void rot_apply_T(const Rot &R, const double v[3], double o[3])          // LVLH -> body (:470-488)
{
#pragma unroll
    for (int i = 0; i < 3; ++i) o[i] = fma(R.m[6 + i], v[2], fma(R.m[3 + i], v[1], R.m[i] * v[0]));
}

// sqrt(x) for x >= 0 (<= 1 ulp): x * rsqrt(x)
RDV_DEV double fast_sqrt(double x) { return x > 0.0 ? x * fast_rsqrt(x) : 0.0; }

// angle_between_vectors (utils/general.py:163-181): acos(round(cos, 5)), with numpy's
// round == rint(x*1e5)/1e5.  k/1e5 is formed as k*1e-5 plus one Markstein correction step, which equals the
// IEEE quotient for every integer |k| <= 1e5 (checked exhaustively) -- in particular +-1 stay exactly +-1.
RDV_DEV double acos_of_rounded(double k)
{
    const double x0 = k * 1e-5;
    return acos(fma(fma(-x0, 1e5, k), 1e-5, x0));
}
// The rounded cosine takes only 200,001 values, so the angle is a table look-up (1.6 MB, resident in the L2): one
// load instead of the ~85 instructions of acos().  The table is filled by acos_table_kernel with acos_of_rounded
// itself, once per device, before the first kernel that reads it (ensure_tables in rdv_b200.cu).
constexpr int ACOS_TABLE_HALF = 100000;
__device__ double g_acos_table[2 * ACOS_TABLE_HALF + 1];
RDV_DEV double rounded_angle_from(double dot, double n1sq, double n2sq)
{
    const double c = dot * fast_rsqrt(n1sq * n2sq);
    const double k = rint(c * 1e5);
    if (fabs(k) <= (double)ACOS_TABLE_HALF) return g_acos_table[(int)k + ACOS_TABLE_HALF];
    return acos_of_rounded(k);                       // NaN (a zero vector) or out of range: the library's answer
}

// ---------------------------------------------------------------------------------
// Attitude ODE right-hand side (utils/dynamics.py:93-175).
//   ISO = true : inertia is c*Identity and the torque is zero, so w_dot == 0 exactly and
//                only the four quaternion derivatives are live (hw = 0.5*w is constant).
//   ISO = false: full 3x3 inertia, held torque.
// ---------------------------------------------------------------------------------
struct BodyConst { const double *I, *Iinv, *tau; };

template <bool ISO>
RDV_DEV void attitude_rhs(const double *y, const double *hw_iso, const BodyConst &b, double *f)
{
    double r = fast_rsqrt(dot4(y, y));             // q/|q| (dynamics.py:108, :134 -- applied once)
    double h1, h2, h3;
    if (ISO) { h1 = hw_iso[0]; h2 = hw_iso[1]; h3 = hw_iso[2]; }
    else     { h1 = 0.5 * y[4]; h2 = 0.5 * y[5]; h3 = 0.5 * y[6]; }
    // 0.5 * Omega(w) q  (dynamics.py:137-150), scaled by 1/|q| afterwards
    double g0 = -fma(h3, y[3], fma(h2, y[2], h1 * y[1]));
    double g1 = fma(-h2, y[3], fma(h3, y[2], h1 * y[0]));
    double g2 = fma(h1, y[3], fma(-h3, y[1], h2 * y[0]));
    double g3 = fma(-h1, y[2], fma(h2, y[1], h3 * y[0]));
    f[0] = g0 * r; f[1] = g1 * r; f[2] = g2 * r; f[3] = g3 * r;
    if (!ISO) {
        const double *w = y + 4;
        double L[3], c[3], t[3];
#pragma unroll
        for (int i = 0; i < 3; ++i) L[i] = fma(b.I[3 * i + 2], w[2], fma(b.I[3 * i + 1], w[1], b.I[3 * i] * w[0]));
        cross3(w, L, c);
#pragma unroll
        for (int i = 0; i < 3; ++i) t[i] = b.tau[i] - c[i];
#pragma unroll
        for (int i = 0; i < 3; ++i)
            f[4 + i] = fma(b.Iinv[3 * i + 2], t[2], fma(b.Iinv[3 * i + 1], t[1], b.Iinv[3 * i] * t[0]));
    }
}

// Dormand-Prince tableau (scipy rk.py, class RK45).  Kept in the constant bank so that DFMA reads each
// coefficient as a c[][] operand instead of materialising a 64-bit immediate with two moves per use.
__constant__ double c_rk[26] = {
    1.0 / 5,
    3.0 / 40,
    9.0 / 40,
    44.0 / 45,
    -56.0 / 15,
    32.0 / 9,
    19372.0 / 6561,
    -25360.0 / 2187,
    64448.0 / 6561,
    -212.0 / 729,
    9017.0 / 3168,
    -355.0 / 33,
    46732.0 / 5247,
    49.0 / 176,
    -5103.0 / 18656,
    35.0 / 384,
    500.0 / 1113,
    125.0 / 192,
    -2187.0 / 6784,
    11.0 / 84,
    -71.0 / 57600,
    71.0 / 16695,
    -71.0 / 1920,
    17253.0 / 339200,
    -22.0 / 525,
    1.0 / 40,
};
#define RK_A21 c_rk[0]
#define RK_A31 c_rk[1]
#define RK_A32 c_rk[2]
#define RK_A41 c_rk[3]
#define RK_A42 c_rk[4]
#define RK_A43 c_rk[5]
#define RK_A51 c_rk[6]
#define RK_A52 c_rk[7]
#define RK_A53 c_rk[8]
#define RK_A54 c_rk[9]
#define RK_A61 c_rk[10]
#define RK_A62 c_rk[11]
#define RK_A63 c_rk[12]
#define RK_A64 c_rk[13]
#define RK_A65 c_rk[14]
#define RK_B1 c_rk[15]
#define RK_B3 c_rk[16]
#define RK_B4 c_rk[17]
#define RK_B5 c_rk[18]
#define RK_B6 c_rk[19]
#define RK_E1 c_rk[20]
#define RK_E3 c_rk[21]
#define RK_E4 c_rk[22]
#define RK_E5 c_rk[23]
#define RK_E6 c_rk[24]
#define RK_E7 c_rk[25]
#define RK_RTOL 1e-7     /* rendezvous_env.py:567, :594 */
#define RK_ATOL 1e-6     /* rendezvous_env.py:568, :595 */

// solve_ivp(fun, (0, dt), y, method='RK45', t_eval=[dt], rtol=1e-7, atol=1e-6) -- the adaptive
// controller of scipy (RungeKutta.__init__ rk.py:85-103, select_initial_step common.py:68-134,
// _step_impl rk.py:111-179, rk_step rk.py:14-69).  On the step that reaches dt the t_eval
// branch (ivp.py:710-728) evaluates the dense-output polynomial at x == 1, which equals y_new
// up to ~1 ulp; y_new is used.  Returns accepted steps, or -1 on TOO_SMALL_STEP / non-finite
// error norm (the reference raises there); y is left at the last accepted state.
// ---------------------------------------------------------------------------------
// Step-size controller arithmetic in float32.
//
// The error norm, the scale vector, the step factor 0.9 err^-0.2 and select_initial_step only steer the
// step size; the propagated state never sees them except through h.  One accepted step changes by
// d(y_new)/dh * dh ~ 5 err/h * dh, i.e. a 1e-6 relative error in h (what float32 + fast log2/exp2 give) moves
// the state by ~1e-14 -- five orders below the 1e-9 parity bar -- while the fp64 pipe, the bottleneck, is
// relieved of ~18 % of its instructions (4 reciprocals, the norm and a pow per attempt; 7 reciprocals,
// three norms and a pow per solve).  The error ESTIMATE itself (the E-weighted sum of the stages, a
// cancellation) stays fp64.  The accept test err < 1 is re-evaluated in full fp64 whenever the float32
// value lies within 1e-3 of the threshold, so accept / reject decisions are those of the fp64 controller.
// ---------------------------------------------------------------------------------
// float32 helpers of the controller: single MUFU instructions without the denormal-range fix-ups of
// __fdividef / __log2f / exp2f (every argument here is a normal number: scales >= atol = 1e-6, clamped norms)
RDV_DEV float rcp_f32(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
RDV_DEV float lg2_f32(float x) { float r; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
RDV_DEV float ex2_f32(float x) { float r; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
RDV_DEV float pow_neg_tenth_f32(float x) { return ex2_f32(-0.1f * lg2_f32(x)); }

template <bool ISO>
RDV_DEV int rk45_attitude(double (&y)[7], const double dt, const BodyConst &b, int &n_rejected)
{
    constexpr int NA = ISO ? 4 : 7;         // components with a non-zero derivative
    double hw[3] = {0.5 * y[4], 0.5 * y[5], 0.5 * y[6]};
    double K[7][NA];
    attitude_rhs<ISO>(y, hw, b, K[0]);

    // ---- select_initial_step (order 4) ----
    double h_abs;
    {
        float inv_sc[7], d0s = 0.0f, d1s = 0.0f;
#pragma unroll
        for (int i = 0; i < 7; ++i) {
            const float yi = (float)y[i];
            inv_sc[i] = rcp_f32(fmaf(fabsf(yi), (float)RK_RTOL, (float)RK_ATOL));
            const float a = yi * inv_sc[i];
            d0s = fmaf(a, a, d0s);
        }
#pragma unroll
        for (int i = 0; i < NA; ++i) {
            const float a = (float)K[0][i] * inv_sc[i];
            d1s = fmaf(a, a, d1s);
        }
        d0s *= (1.0f / 7.0f);
        d1s *= (1.0f / 7.0f);                                // squares of the rms norms d0, d1
        float h0f;
        if (d0s < 1e-10f || d1s < 1e-10f) h0f = 1e-6f;
        else h0f = 0.01f * sqrtf(d0s * rcp_f32(d1s));
        const double h0 = fmin((double)h0f, dt);
        double y1[7], f1[NA];
#pragma unroll
        for (int i = 0; i < NA; ++i) y1[i] = fma(h0, K[0][i], y[i]);
#pragma unroll
        for (int i = NA; i < 7; ++i) y1[i] = y[i];
        attitude_rhs<ISO>(y1, hw, b, f1);
        float d2s = 0.0f;
#pragma unroll
        for (int i = 0; i < NA; ++i) {
            const float a = (float)(f1[i] - K[0][i]) * inv_sc[i];
            d2s = fmaf(a, a, d2s);
        }
        const float inv_h0 = rcp_f32((float)h0);
        d2s = d2s * (1.0f / 7.0f) * inv_h0 * inv_h0;
        float h1;
        if (d1s <= 1e-30f && d2s <= 1e-30f) h1 = fmaxf(1e-6f, (float)h0 * 1e-3f);
        else h1 = pow_neg_tenth_f32(fminf(fmaxf(d1s, d2s), 1e30f) * 1e4f);   // (0.01/max(d1,d2))**(1/5)
        h_abs = fmin(fmin(100.0 * h0, (double)h1), dt);
    }

    double t = 0.0;
    int accepted = 0;
    for (;;) {
        // ---- one solver.step(): _step_impl ----
        const double min_step = 10.0 * (__longlong_as_double(__double_as_longlong(t) + 1) - t);
        if (h_abs < min_step) h_abs = min_step;
        bool rejected = false;
        double t_new, h;
        double y_new[NA];
        for (;;) {
            if (h_abs < min_step) return -1;
            t_new = t + h_abs;
            if (t_new - dt > 0.0) t_new = dt;
            h = t_new - t;
            h_abs = fabs(h);
            // ---- rk_step: six stages, FSAL row K[6] ----
            double ys[7];
            if (ISO) { ys[4] = y[4]; ys[5] = y[5]; ys[6] = y[6]; }
#pragma unroll
            for (int i = 0; i < NA; ++i) ys[i] = fma(K[0][i] * RK_A21, h, y[i]);
            attitude_rhs<ISO>(ys, hw, b, K[1]);
#pragma unroll
            for (int i = 0; i < NA; ++i) ys[i] = fma(fma(K[1][i], RK_A32, K[0][i] * RK_A31), h, y[i]);
            attitude_rhs<ISO>(ys, hw, b, K[2]);
#pragma unroll
            for (int i = 0; i < NA; ++i)
                ys[i] = fma(fma(K[2][i], RK_A43, fma(K[1][i], RK_A42, K[0][i] * RK_A41)), h, y[i]);
            attitude_rhs<ISO>(ys, hw, b, K[3]);
#pragma unroll
            for (int i = 0; i < NA; ++i)
                ys[i] = fma(fma(K[3][i], RK_A54, fma(K[2][i], RK_A53, fma(K[1][i], RK_A52, K[0][i] * RK_A51))), h,
                            y[i]);
            attitude_rhs<ISO>(ys, hw, b, K[4]);
#pragma unroll
            for (int i = 0; i < NA; ++i)
                ys[i] = fma(fma(K[4][i], RK_A65,
                                fma(K[3][i], RK_A64, fma(K[2][i], RK_A63, fma(K[1][i], RK_A62, K[0][i] * RK_A61)))),
                            h, y[i]);
            attitude_rhs<ISO>(ys, hw, b, K[5]);
#pragma unroll
            for (int i = 0; i < NA; ++i)
                ys[i] = fma(h,
                            fma(K[5][i], RK_B6,
                                fma(K[4][i], RK_B5, fma(K[3][i], RK_B4, fma(K[2][i], RK_B3, K[0][i] * RK_B1)))),
                            y[i]);
            attitude_rhs<ISO>(ys, hw, b, K[6]);
#pragma unroll
            for (int i = 0; i < NA; ++i) y_new[i] = ys[i];
            // ---- error norm: rms((K^T E) h / scale), scale = atol + max(|y|,|y_new|) rtol ----
            double eh[NA];
#pragma unroll
            for (int i = 0; i < NA; ++i)
                eh[i] = h * fma(K[6][i], RK_E7,
                                fma(K[5][i], RK_E6,
                                    fma(K[4][i], RK_E5, fma(K[3][i], RK_E4, fma(K[2][i], RK_E3, K[0][i] * RK_E1)))));
            float esf = 0.0f;
#pragma unroll
            for (int i = 0; i < NA; ++i) {
                const float m = (float)fmax(fabs(y[i]), fabs(y_new[i]));
                const float q = (float)eh[i] * rcp_f32(fmaf(m, (float)RK_RTOL, (float)RK_ATOL));
                esf = fmaf(q, q, esf);
            }
            esf *= (1.0f / 7.0f);                      // err_norm^2
            if (!(esf < 1.0e30f)) return -1;           // NaN / inf: the reference shrinks h to failure
            bool accept = esf < 1.0f;
            if (fabsf(esf - 1.0f) < 1.0e-3f) {         // threshold region: decide with the fp64 norm
                double es = 0.0;
#pragma unroll
                for (int i = 0; i < NA; ++i) {
                    const double e = eh[i] * fast_rcp(fma(fmax(fabs(y[i]), fabs(y_new[i])), RK_RTOL, RK_ATOL));
                    es = fma(e, e, es);
                }
                accept = es * (1.0 / 7.0) < 1.0;
            }
            // 0.9 err^-0.2, clamped where the controller's min / max saturate anyway
            const float p = 0.9f * pow_neg_tenth_f32(fminf(fmaxf(esf, 1e-12f), 1e8f));
            if (accept) {
                float factor = fminf(10.0f, p);
                if (rejected) factor = fminf(1.0f, factor);
                h_abs *= (double)factor;
                break;
            }
            h_abs *= (double)fmaxf(0.2f, p);
            rejected = true;
            ++n_rejected;
        }
        ++accepted;
        t = t_new;
#pragma unroll
        for (int i = 0; i < NA; ++i) { y[i] = y_new[i]; K[0][i] = K[6][i]; }
        if (t - dt >= 0.0) return accepted;
    }
}

// ---------------------------------------------------------------------------------
// The same solver for the reference's bodies (isotropic inertia, no torque: w is constant over the solve), in the
// invariant plane of the motion.
//
// With M = 0.5 Omega(w) the equation is q' = M q / |q|, and M is skew with M^2 = -omega^2 I (omega = |w| / 2).
// Every vector the Runge-Kutta scheme ever forms -- stage vectors, slopes, y_new, the error estimate -- is a
// linear combination of q0 (the state at the start of the solve) and p = M q0:  for y = a q0 + b p,
//
//     M y = a p - b omega^2 q0,     |y|^2 = |q0|^2 (a^2 + omega^2 b^2)      (p is orthogonal to q0, |p| = omega |q0|),
//
// so the scheme is advanced on the coordinates (a, b): a slope costs 11 fp64 operations instead of 25 and the
// stage sums, the 5th-order solution and the embedded error run on 2 components instead of 4.  What the
// controller looks at is NOT basis independent (scale_i = atol + rtol max(|y_i|, |y_new,i|) per component of the
// reference's state vector), so y_new and the error estimate are mapped back to the four quaternion components
// (2 operations per component) before the norm: accept / reject decisions and step sizes are those of the
// 4-component solver, and the propagated state agrees with it to rounding (~1e-15, the plane is invariant in
// exact arithmetic) at 159 instead of 307 fp64 operations per attempted step.  No division by omega occurs:
// w = 0 gives p = 0 and a constant quaternion.
// ---------------------------------------------------------------------------------
// Slope of y = a q0 + b p in plane coordinates.  The basis is scaled so that |q0| drops out: p = (M / |q0|) q0 and
// om2 = omega^2 / |q0|^2, hence y' = M y / |y| = (M / |q0|) y / sqrt(a^2 + om2 b^2).
RDV_DEV void rhs_plane(const double a, const double b, const double om2, double &ka, double &kb)
{
    const double t = om2 * b;
    const double g = fast_rsqrt(fma(t, b, a * a));                // |q0| / |y|
    ka = -(t * g);
    kb = a * g;
}
// g = |q0| / |y| at y = a q0 + b p, formed exactly as inside rhs_plane: a point carries g instead of its slope, which is
// (-(om2 b) g, a g) bit for bit.
RDV_DEV double plane_g(const double a, const double b, const double om2) { return fast_rsqrt(fma(om2 * b, b, a * a)); }

// ---------------------------------------------------------------------------------
// One attempted step in closed form.
//
// With z = a + i w b, w^2 = om2, the plane equation is z' = i w z / |z|: rotation-equivariant and homogeneous of
// degree 0.  Every stage of one Dormand-Prince attempt from z with step h is therefore z times a function of
// s = h w / |z| alone, and so are the 5th-order point and the error estimate:  z_new = z S(s), (K^T E) h = z E(s).
// S and E satisfy f(-s) = conj f(s); with x = s^2 = h^2 om2 g^2 (g = 1 / |z|)
//
//     Re S = 1 + x P1(x),   Im S = s (1 + x Q1(x)),   Re E = x^3 R(x),   Im E = s x^2 I(x),
//
// polynomials fitted at 50 digits by tools/gen_plane_poly.py (rdv_plane_poly.h; 6-7 coefficients each on
// x <= X_MAX = 1/32, P and Q to < 0.01 ulp, R and I to < 1e-14).  Back in plane coordinates, with u = h g a and
// v = h g om2 b (no division by w; w = 0 gives x = 0, P = 1 and a_new = a exactly):
//
//     a_new = a P - v Q,   b_new = b P + u Q,   ea = a x^3 R - v x^2 I,   eb = b x^3 R + u x^2 I.
//
// That is ~40 fp64 operations and no MUFU per attempt against ~130 operations and 7 RSQ for the six slopes of the
// stagewise form, and the critical path is one Horner chain instead of six dependent slope chains.  The results
// agree with the stagewise attempt to its rounding (~1e-16 on the state; the stagewise error estimate carries
// ~1e-16 h of cancellation noise that the polynomial does not).
//
// Where it applies: h <= dt and g = 1 at the start of a solve, and |z| moves by at most DRIFT_PER_S s per accepted
// step (4e-10 s), i.e. by < 1e-10 over a whole solve (sum of s <= sqrt(om2) dt).  So om2 dt^2 (1 + 2^-20) <= X_MAX
// keeps every attempt of the solve inside the fitted range; the 2^-20 also covers the rounding of om2 and x.  Faster
// spins (om2 dt^2 > X_MAX ~ |w| dt > 0.35 rad) take the stagewise attempt for the whole solve, out of line.
// Measured (B200): 9.72 -> 9.30 us per step (20-step launches), 8.86 -> 8.65 (250-step).
// ---------------------------------------------------------------------------------
constexpr int PP_P1 = 0, PP_Q1 = PP_P1 + RDV_PP_N_P1, PP_R = PP_Q1 + RDV_PP_N_Q1, PP_I = PP_R + RDV_PP_N_R;
__constant__ double c_pp[PP_I + RDV_PP_N_I] = {RDV_PP_P1, RDV_PP_Q1, RDV_PP_R, RDV_PP_I};

template <int OFF, int N>
RDV_DEV double pp_horner(const double x)
{
    double r = c_pp[OFF + N - 1];
#pragma unroll
    for (int k = N - 2; k >= 0; --k) r = fma(r, x, c_pp[OFF + k]);
    return r;
}
// Re S, Im S / s, Re E / x^3, Im E / (s x^2) at x = s^2
RDV_DEV void plane_poly(const double x, double &P, double &Q, double &R, double &I)
{
    P = fma(x, pp_horner<PP_P1, RDV_PP_N_P1>(x), 1.0);
    Q = fma(x, pp_horner<PP_Q1, RDV_PP_N_Q1>(x), 1.0);
    R = pp_horner<PP_R, RDV_PP_N_R>(x);
    I = pp_horner<PP_I, RDV_PP_N_I>(x);
}
// whether every attempt of the solve from y over dt stays inside the polynomials' range (see above); false for a
// non-finite rate.  0.25 |w|^2 / |q0|^2 is om2 of plane_basis to a few ulp.
RDV_DEV bool plane_poly_covers(const double (&y)[7], const double dt)
{
    const double w2 = fma(y[6], y[6], fma(y[5], y[5], y[4] * y[4]));
    const double q2 = fma(y[3], y[3], fma(y[2], y[2], fma(y[1], y[1], y[0] * y[0])));
    return 0.25 * w2 * (dt * dt) <= (RDV_PP_X_MAX * (1.0 - 0x1p-20)) * q2;
}

// One attempted step of rk_step (scipy rk.py:14-69) in plane coordinates from y = a q0 + b p (g = |q0| / |y|) with
// step h: the candidate (a_new, b_new) and the error estimate (K^T E) h = ea q0 + eb p.  POLY: the closed form above;
// otherwise the six stages and the slope at the new point, the first slope (FSAL) rebuilt from g bit for bit.  Both
// solvers and every launch shape call this one function, so they give identical bits.
template <bool POLY>
RDV_DEV void plane_attempt(const double a, const double b, const double g, const double om2, const double h,
                           double &a_new, double &b_new, double &ea, double &eb)
{
    if (POLY) {
        const double hg = h * g, t = hg * om2;
        const double u = hg * a, v = t * b, x = t * hg;
        double P, Q, R, I;
        plane_poly(x, P, Q, R, I);
        a_new = fma(a, P, -(v * Q));
        b_new = fma(b, P, u * Q);
        const double x2 = x * x, xr = x * R;
        ea = x2 * fma(a, xr, -(v * I));
        eb = x2 * fma(b, xr, u * I);
    } else {
        double ka[7], kb[7], as, bs;
        ka[0] = -((om2 * b) * g); kb[0] = a * g;
        as = fma(ka[0] * RK_A21, h, a);
        bs = fma(kb[0] * RK_A21, h, b);
        rhs_plane(as, bs, om2, ka[1], kb[1]);
        as = fma(fma(ka[1], RK_A32, ka[0] * RK_A31), h, a);
        bs = fma(fma(kb[1], RK_A32, kb[0] * RK_A31), h, b);
        rhs_plane(as, bs, om2, ka[2], kb[2]);
        as = fma(fma(ka[2], RK_A43, fma(ka[1], RK_A42, ka[0] * RK_A41)), h, a);
        bs = fma(fma(kb[2], RK_A43, fma(kb[1], RK_A42, kb[0] * RK_A41)), h, b);
        rhs_plane(as, bs, om2, ka[3], kb[3]);
        as = fma(fma(ka[3], RK_A54, fma(ka[2], RK_A53, fma(ka[1], RK_A52, ka[0] * RK_A51))), h, a);
        bs = fma(fma(kb[3], RK_A54, fma(kb[2], RK_A53, fma(kb[1], RK_A52, kb[0] * RK_A51))), h, b);
        rhs_plane(as, bs, om2, ka[4], kb[4]);
        as = fma(fma(ka[4], RK_A65, fma(ka[3], RK_A64, fma(ka[2], RK_A63, fma(ka[1], RK_A62, ka[0] * RK_A61)))), h, a);
        bs = fma(fma(kb[4], RK_A65, fma(kb[3], RK_A64, fma(kb[2], RK_A63, fma(kb[1], RK_A62, kb[0] * RK_A61)))), h, b);
        rhs_plane(as, bs, om2, ka[5], kb[5]);
        a_new = fma(h, fma(ka[5], RK_B6, fma(ka[4], RK_B5, fma(ka[3], RK_B4, fma(ka[2], RK_B3, ka[0] * RK_B1)))), a);
        b_new = fma(h, fma(kb[5], RK_B6, fma(kb[4], RK_B5, fma(kb[3], RK_B4, fma(kb[2], RK_B3, kb[0] * RK_B1)))), b);
        rhs_plane(a_new, b_new, om2, ka[6], kb[6]);
        ea = h * fma(ka[6], RK_E7, fma(ka[5], RK_E6, fma(ka[4], RK_E5, fma(ka[3], RK_E4, fma(ka[2], RK_E3, ka[0] * RK_E1)))));
        eb = h * fma(kb[6], RK_E7, fma(kb[5], RK_E6, fma(kb[4], RK_E5, fma(kb[3], RK_E4, fma(kb[2], RK_E3, kb[0] * RK_E1)))));
    }
}

// What the controller sees of one attempted step, in float32 (rationale at rk45_attitude): the candidate state
// y_new = a_new q0 + b_new p and the error estimate e = ea q0 + eb p in quaternion components, and
// err^2 = mean((e_i / (atol + rtol max(|y_i|, |y_new,i|)))^2) over the reference's seven components (the three
// rate components contribute 0).  q0 is orthogonal to p, so sum e_i^2 = ea^2 |q0|^2 + eb^2 |p|^2 and cancellation
// inside single components cannot amplify the float32 rounding of the norm beyond ~2e-7 relative.
RDV_DEV float plane_err2_f32(const double ea, const double eb, const double a_new, const double b_new,
                             const float (&q0f)[4], const float (&pf)[4], const float (&ycf)[4], float (&ynf)[4])
{
    const float eaf = (float)ea, ebf = (float)eb, anf = (float)a_new, bnf = (float)b_new;
    float esf = 0.0f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        ynf[i] = fmaf(bnf, pf[i], anf * q0f[i]);
        const float e = fmaf(ebf, pf[i], eaf * q0f[i]);
        const float m = fmaxf(fabsf(ycf[i]), fabsf(ynf[i]));
        const float q = e * rcp_f32(fmaf(m, (float)RK_RTOL, (float)RK_ATOL));
        esf = fmaf(q, q, esf);
    }
    return esf * (1.0f / 7.0f);
}
// the same quantity in fp64, for the accept decision when the float32 value lies within 1e-3 of the threshold
RDV_DEV double plane_err2_f64(const double ea, const double eb, const double a, const double b, const double a_new,
                              const double b_new, const double (&q0)[4], const double (&p)[4])
{
    double es = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const double yc = fma(b, p[i], a * q0[i]), yn = fma(b_new, p[i], a_new * q0[i]);
        const double e = fma(eb, p[i], ea * q0[i]) * fast_rcp(fma(fmax(fabs(yc), fabs(yn)), RK_RTOL, RK_ATOL));
        es = fma(e, e, es);
    }
    return es * (1.0 / 7.0);
}
// select_initial_step (scipy common.py:68-134, order 4).  The first slope at (a, b) = (1, 0) is (0, 1) exactly:
// f0 = M q0 / |q0| = p.
// d2 = rms((f(y0 + h0 f0) - f0) / scale) / h0 only enters through max(d1, d2).  In plane coordinates
// f1 - f0 = da q0 + db p with |da| <= om2 h0 and |db| <= om2 h0^2 / 2, hence d2 <= om2 (rms(q0 / scale) + h0 d1 / 2):
// of the order omega d1, i.e. below d1 unless the body spins at ~1 rad/s.  When this bound (with 5 % slack for the
// float32 arithmetic) is below d1 the second slope is not evaluated at all; otherwise d2 is formed exactly as scipy does.
// The returned value is min(100 h0, h1, dt) with 100 h0 = d0 / d1, and d0 only grows when the three rate components
// join its norm: whenever the quaternion part alone already puts 100 h0 above min(h1, dt) -- always, unless a body
// spins at several rad/s -- the rate part of d0 is never formed.  The bound that lets the second slope go is then
// taken with h0 <= dt instead of h0 itself, which needs d0 too (measured against forming d0 first: 10.12 -> 9.93 us
// per step in 20-step launches, 9.33 -> 9.12 in 250-step ones).
RDV_DEV double plane_initial_step(const double (&y)[7], const float (&q0f)[4], const float (&pf)[4], const double om2,
                                  const double dt)
{
    float inv_sc[4], d0r = 0.0f, d1s = 0.0f;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        inv_sc[i] = rcp_f32(fmaf(fabsf(q0f[i]), (float)RK_RTOL, (float)RK_ATOL));
        const float v = q0f[i] * inv_sc[i], f = pf[i] * inv_sc[i];               // y0 / scale, f0 / scale
        d0r = fmaf(v, v, d0r);
        d1s = fmaf(f, f, d1s);
    }
    const float d0q = d0r * (1.0f / 7.0f);                                       // the quaternion part of d0^2
    d1s *= (1.0f / 7.0f);
    const float dtf = (float)dt;
    // d2 <= om2 (sqrt(d0q) + dt sqrt(d1s) / 2) with h0 <= dt; "bound^2 * 1.05 <= d1s" without a square root:
    // om2 sqrt(d0q) <= sqrt(d1s) (0.975 - om2 dt / 2), both sides non-negative, squared
    // (measured against the two square roots: 9.94 -> 9.76 us per step in 20-step launches, 9.13 -> 8.94 in 250-step)
    const float om2f = (float)om2, room = fmaf(-0.5f * dtf, om2f, 0.975f);
    const bool d2_small = room > 0.0f && om2f * om2f * d0q <= d1s * room * room;
    if (d0q >= 1e-10f && d1s >= 1e-10f && d2_small) {
        // common case: d2 <= d1, so h1 = (0.01 / d1)^(1/5); and 100 h0 >= sqrt(d0q / d1s) (or 100 dt)
        const float h1 = pow_neg_tenth_f32(fminf(d1s, 1e30f) * 1e4f);
        const float lim = fminf(h1, dtf);
        if (d0q >= lim * lim * d1s * 1.0001f) return fmin((double)h1, dt);       // 100 h0 cannot be the minimum
    }
    // general path: scipy's select_initial_step term by term
    float d0s = d0r;
#pragma unroll
    for (int i = 4; i < 7; ++i) {                                                // the rate components: f0 = 0
        const float yi = (float)y[i];
        const float v = yi * rcp_f32(fmaf(fabsf(yi), (float)RK_RTOL, (float)RK_ATOL));
        d0s = fmaf(v, v, d0s);
    }
    d0s *= (1.0f / 7.0f);
    float h0f;
    if (d0s < 1e-10f || d1s < 1e-10f) h0f = 1e-6f;
    else h0f = 0.01f * sqrtf(d0s * rcp_f32(d1s));
    const double h0 = fmin((double)h0f, dt);
    const float h0c = (float)h0;
    const float ub2 = (float)om2 * fmaf(0.5f * h0c, sqrtf(d1s), sqrtf(d0q));
    float dmax = d1s;
    if (!(ub2 * ub2 * 1.05f <= d1s)) {
        double ka1, kb1;
        rhs_plane(1.0, h0, om2, ka1, kb1);                       // y1 = y0 + h0 f0
        const float daf = (float)ka1, dbf = (float)(kb1 - 1.0);  // f1 - f0 in plane coordinates
        float d2s = 0.0f;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float v = fmaf(dbf, pf[i], daf * q0f[i]) * inv_sc[i];
            d2s = fmaf(v, v, d2s);
        }
        const float inv_h0 = rcp_f32(h0c);
        d2s = d2s * (1.0f / 7.0f) * inv_h0 * inv_h0;
        dmax = fmaxf(d1s, d2s);
    }
    float h1;
    if (dmax <= 1e-30f) h1 = fmaxf(1e-6f, h0c * 1e-3f);     // d1 <= 1e-15 and d2 <= 1e-15
    else h1 = pow_neg_tenth_f32(fminf(dmax, 1e30f) * 1e4f);  // (0.01/max(d1,d2))**(1/5)
    return fmin(fmin(100.0 * h0, (double)h1), dt);
}

// basis of the invariant plane of one body: q0, p = (0.5 Omega(w) / |q0|) q0 (dynamics.py:137-150), om2 = |0.5 w|^2 / |q0|^2
RDV_DEV void plane_basis(const double (&y)[7], double (&q0)[4], double (&p)[4], double &om2)
{
#pragma unroll
    for (int i = 0; i < 4; ++i) q0[i] = y[i];
    const double hs = 0.5 * fast_rsqrt(dot4(q0, q0));
    const double hw[3] = {hs * y[4], hs * y[5], hs * y[6]};
    p[0] = -fma(hw[2], q0[3], fma(hw[1], q0[2], hw[0] * q0[1]));
    p[1] = fma(-hw[1], q0[3], fma(hw[2], q0[2], hw[0] * q0[0]));
    p[2] = fma(hw[0], q0[3], fma(-hw[2], q0[1], hw[1] * q0[0]));
    p[3] = fma(-hw[0], q0[2], fma(hw[1], q0[1], hw[2] * q0[0]));
    om2 = fma(hw[2], hw[2], fma(hw[1], hw[1], hw[0] * hw[0]));
}

// One point of the solution in plane coordinates, with what the next step needs from it: g = |q0| / |y| (which also
// gives the FSAL slope of the stagewise attempt) and the float32 quaternion components the controller's scale vector
// uses.
struct PlanePoint { double a, b, g, t; float yf[4]; };

// One solver.step() of scipy's RungeKutta._step_impl (rk.py:111-179): attempts from `s` until one is accepted; the
// accepted point goes to `n` (`s` is left untouched).  Returns 0 on TOO_SMALL_STEP / a non-finite error norm, 2 when
// the accepted step reaches t = dt (known when t_new is clipped, so the caller need not re-derive it from t), else 1.
// The attempt that is clipped to t = dt ends the solve when it is accepted -- the step factor and the float32 copy of
// the new point are never used again -- so all it needs from the controller is the accept decision.  With
// scale_i >= atol,  err^2 <= sum e_i^2 / (7 atol^2) <= 2 (ea^2 |q0|^2 + eb^2 |p|^2) / (7 atol^2) (q0 is orthogonal to
// p; the factor 2 covers the rounding of that): below 0.99 the attempt is accepted without forming the per-component
// norm, anything else takes the full path (measured: 9.76 -> 9.74 us per step in 20-step launches, 8.94 -> 8.91 in
// 250-step ones).
template <bool POLY>
RDV_DEV int plane_step(const PlanePoint &s, PlanePoint &n, double &h_abs, int &n_rejected, const double om2, const double dt,
                        const double (&q0)[4], const double (&p)[4], const float (&q0f)[4], const float (&pf)[4])
{
    const double a = s.a, b = s.b, t = s.t;
    const double min_step = 10.0 * (__longlong_as_double(__double_as_longlong(t) + 1) - t);
    if (h_abs < min_step) h_abs = min_step;
    bool rejected = false;
    for (;;) {
        if (h_abs < min_step) return 0;
        double t_new = t + h_abs;
        const double over = t_new - dt;
        if (over > 0.0) t_new = dt;
        const bool last = over >= 0.0;
        const double h = t_new - t;
        h_abs = fabs(h);
        // ---- rk_step and the error estimate (K^T E) h in the plane; the controller's norm in quaternion components ----
        double a_new, b_new, ea, eb;
        plane_attempt<POLY>(a, b, s.g, om2, h, a_new, b_new, ea, eb);
        if (last) {
            const float eaf = (float)ea, ebf = (float)eb;
            float nq = 0.0f, np = 0.0f;
#pragma unroll
            for (int i = 0; i < 4; ++i) { nq = fmaf(q0f[i], q0f[i], nq); np = fmaf(pf[i], pf[i], np); }
            const float ub = fmaf(eaf * eaf, nq, ebf * ebf * np) * (2.0f / 7.0f * 1.0e12f);   // atol^-2 = 1e12
            if (ub < 0.99f) {
                n.a = a_new; n.b = b_new; n.t = t_new;          // the solve ends here: g is not needed
                return 2;
            }
        }
        const float esf = plane_err2_f32(ea, eb, a_new, b_new, q0f, pf, s.yf, n.yf);
        // one branch for both rare cases: a non-finite norm (the reference shrinks h to failure) and the threshold
        // region, where the accept decision is taken with the fp64 norm (measured against two branches: 10.20 -> 10.13
        // us per step in 20-step launches, 9.415 -> 9.37 in 250-step ones)
        bool accept = esf < 1.0f;
        if (!(fabsf(esf - 1.0f) >= 1.0e-3f && esf < 1.0e30f)) {
            if (!(esf < 1.0e30f)) return 0;
            accept = plane_err2_f64(ea, eb, a, b, a_new, b_new, q0, p) < 1.0;
        }
        // 0.9 err^-0.2, clamped where the controller's min / max saturate anyway
        const float pw = 0.9f * pow_neg_tenth_f32(fminf(fmaxf(esf, 1e-12f), 1e8f));
        if (accept) {
            float factor = fminf(10.0f, pw);
            if (rejected) factor = fminf(1.0f, factor);
            h_abs *= (double)factor;
            n.a = a_new; n.b = b_new; n.g = plane_g(a_new, b_new, om2); n.t = t_new;
            return last ? 2 : 1;
        }
        h_abs *= (double)fmaxf(0.2f, pw);
        rejected = true;
        ++n_rejected;
    }
}

// The float32 copies of the basis are used by every attempted step.  Left alone, the compiler re-converts them from
// the fp64 values inside the loop (8 F2F per attempt on the 16-lane XU pipe) rather than keep eight more registers;
// the empty asm makes the converted value opaque, so it is kept (or spilled as 4 bytes) instead (measured: 11.29 ->
// 10.93 us per step at 65,536 envs).
template <bool POLY>
RDV_DEV int rk45_iso_plane_solve(double (&y)[7], const double dt, int &n_rejected)
{
    double q0[4], p[4], om2;
    plane_basis(y, q0, p, om2);
    float q0f[4], pf[4];
    PlanePoint X, Y;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        q0f[i] = (float)q0[i]; pf[i] = (float)p[i];
        asm volatile("" : "+f"(q0f[i])); asm volatile("" : "+f"(pf[i]));
        X.yf[i] = q0f[i];
    }
    X.a = 1.0; X.b = 0.0; X.g = 1.0; X.t = 0.0;                 // y = a q0 + b p; slope there = p
    double h_abs = plane_initial_step(y, q0f, pf, om2, dt);
    int accepted = 0;
    // One copy of the step, and the accepted point is copied back.  Two copies that alternate between X and Y, so that
    // nothing is copied, measured slower on B200 (12.1 vs 11.3 us per step at 65,536 envs: the second copy costs more
    // spills than the ~30 moves per accepted step it saves).
    for (;;) {
        const int r = plane_step<POLY>(X, Y, h_abs, n_rejected, om2, dt, q0, p, q0f, pf);
        if (!r) return -1;
        ++accepted;
        X = Y;
        if (r == 2) break;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) y[i] = fma(X.b, p[i], X.a * q0[i]);
    return accepted;
}
// the stagewise solve for rates outside the polynomials' range, out of line: the hot loop holds one form only
__device__ __noinline__ int rk45_iso_plane_stagewise(double (&y)[7], const double dt, int &n_rejected)
{
    return rk45_iso_plane_solve<false>(y, dt, n_rejected);
}
RDV_DEV int rk45_iso_plane(double (&y)[7], const double dt, int &n_rejected)
{
    if (!plane_poly_covers(y, dt)) return rk45_iso_plane_stagewise(y, dt, n_rejected);
    return rk45_iso_plane_solve<true>(y, dt, n_rejected);
}

// Lock-step form of rk45_iso_plane for TWO bodies in one thread (chaser and target of one env): the control flow of
// scipy's _step_impl (accept / reject, the factor clamps, the rejected-step rule, TOO_SMALL_STEP) is written as
// predicated updates, a body that has reached t = dt keeps stepping in the shadow without committing anything, and
// the two bodies are interleaved stage by stage in the source, so that two independent slope chains (norm ->
// rsqrt -> scale) sit next to each other in every basic block.  Arithmetic per body is that of rk45_iso_plane,
// operation for operation (tests/test_gpu_rollout.py compares the bits).
RDV_DEV int rk45_iso_plane_pair_solve(double (&ya)[7], double (&yb)[7], const double dt, int &n_rejected)
{
    double q0[2][4], p[2][4], om2[2], a[2], b[2], g[2], h_abs[2], t[2];
    float q0f[2][4], pf[2][4], ycf[2][4];
    int accepted[2] = {0, 0};
    bool done[2] = {false, false}, rejected[2] = {false, false}, failed[2] = {false, false};
    plane_basis(ya, q0[0], p[0], om2[0]);
    plane_basis(yb, q0[1], p[1], om2[1]);
#pragma unroll
    for (int c = 0; c < 2; ++c) {
        a[c] = 1.0; b[c] = 0.0; g[c] = 1.0;
#pragma unroll
        for (int i = 0; i < 4; ++i) { q0f[c][i] = (float)q0[c][i]; pf[c][i] = (float)p[c][i]; ycf[c][i] = q0f[c][i]; }
    }
    h_abs[0] = plane_initial_step(ya, q0f[0], pf[0], om2[0], dt);
    h_abs[1] = plane_initial_step(yb, q0f[1], pf[1], om2[1], dt);
    t[0] = t[1] = 0.0;
    // ---- attempted steps, both bodies per pass, predicated commit ----
    while (!((done[0] || failed[0]) && (done[1] || failed[1]))) {
        double h[2], t_new[2], ha[2], as[2], bs[2], ea[2], eb[2];
        bool fail_now[2];
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            const double min_step = 10.0 * (__longlong_as_double(__double_as_longlong(t[c]) + 1) - t[c]);
            fail_now[c] = rejected[c] && h_abs[c] < min_step;
            ha[c] = rejected[c] ? h_abs[c] : fmax(h_abs[c], min_step);
            t_new[c] = t[c] + ha[c];
            if (t_new[c] - dt > 0.0) t_new[c] = dt;
            h[c] = t_new[c] - t[c];
            ha[c] = fabs(h[c]);
        }
#pragma unroll
        for (int c = 0; c < 2; ++c) plane_attempt<true>(a[c], b[c], g[c], om2[c], h[c], as[c], bs[c], ea[c], eb[c]);
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            // as / bs hold (a_new, b_new) of the attempted step
            float ynf[4];
            const float esf = plane_err2_f32(ea[c], eb[c], as[c], bs[c], q0f[c], pf[c], ycf[c], ynf);
            const bool live = !done[c] && !failed[c];
            const bool bad = fail_now[c] || !(esf < 1.0e30f);
            bool accept = esf < 1.0f;
            if (fabsf(esf - 1.0f) < 1.0e-3f)           // threshold region: decide with the fp64 norm
                accept = plane_err2_f64(ea[c], eb[c], a[c], b[c], as[c], bs[c], q0[c], p[c]) < 1.0;
            const float pw = 0.9f * pow_neg_tenth_f32(fminf(fmaxf(esf, 1e-12f), 1e8f));
            float factor = accept ? fminf(10.0f, pw) : fmaxf(0.2f, pw);
            if (accept && rejected[c]) factor = fminf(1.0f, factor);
            const bool commit = live && !bad && accept;
            if (live) {
                failed[c] = bad;
                h_abs[c] = bad ? h_abs[c] : ha[c] * (double)factor;
                rejected[c] = !accept;
                n_rejected += (!bad && !accept) ? 1 : 0;
            }
            if (commit) {
                a[c] = as[c]; b[c] = bs[c]; g[c] = plane_g(as[c], bs[c], om2[c]);
#pragma unroll
                for (int i = 0; i < 4; ++i) ycf[c][i] = ynf[i];
                t[c] = t_new[c];
                accepted[c] += 1;
                done[c] = t_new[c] - dt >= 0.0;
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        ya[i] = fma(b[0], p[0][i], a[0] * q0[0][i]);
        yb[i] = fma(b[1], p[1][i], a[1] * q0[1][i]);
    }
    return (failed[0] || failed[1]) ? -1 : accepted[0] + accepted[1];
}
// a pair with a body outside the polynomials' range: the two solves one after the other, each in its own form (the
// same bits as in the lock-step form), out of line
__device__ __noinline__ int rk45_iso_plane_pair_mixed(double (&ya)[7], double (&yb)[7], const double dt, int &n_rejected)
{
    const int ka = rk45_iso_plane(ya, dt, n_rejected);
    const int kb = rk45_iso_plane(yb, dt, n_rejected);
    return (ka < 0 || kb < 0) ? -1 : ka + kb;
}
RDV_DEV int rk45_iso_plane_pair(double (&ya)[7], double (&yb)[7], const double dt, int &n_rejected)
{
    if (!(plane_poly_covers(ya, dt) && plane_poly_covers(yb, dt))) return rk45_iso_plane_pair_mixed(ya, yb, dt, n_rejected);
    return rk45_iso_plane_pair_solve(ya, yb, dt, n_rejected);
}

// Closed-form alternative (opt-in, RDV_INTEGRATOR_CLOSED_FORM; only valid for ISO bodies):
// with w constant, q' = 0.5 Omega(w) q/|q| has the exact solution
// q(dt) = q cos(a) + (Omega(w) q) sin(a)/|w|, a = |w| dt / (2|q|).  The RK45 replica itself
// is only accurate to ~1e-10..1e-8 per step, so this differs from the reference by the
// reference's own truncation error (SURVEY.md section 7 hard part 7); callers gate it.
RDV_DEV void closed_form_attitude(double (&y)[7], const double dt)
{
    double wsq = fma(y[6], y[6], fma(y[5], y[5], y[4] * y[4]));
    if (wsq == 0.0) return;
    double rq = fast_rsqrt(dot4(y, y));
    double wn = sqrt(wsq);
    double s, c;
    sincos(0.5 * wn * dt * rq, &s, &c);
    double k = s / wn;
    double g0 = -fma(y[6], y[3], fma(y[5], y[2], y[4] * y[1]));
    double g1 = fma(-y[5], y[3], fma(y[6], y[2], y[4] * y[0]));
    double g2 = fma(y[4], y[3], fma(-y[6], y[1], y[5] * y[0]));
    double g3 = fma(-y[4], y[2], fma(y[5], y[1], y[6] * y[0]));
    y[0] = fma(g0, k, y[0] * c); y[1] = fma(g1, k, y[1] * c);
    y[2] = fma(g2, k, y[2] * c); y[3] = fma(g3, k, y[3] * c);
}

// ---------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11) -- counter-based generator for reset().
// counter = (env_id lo, env_id hi, episode index, block), key = seed.
// ---------------------------------------------------------------------------------
RDV_DEV void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1)
{
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t hi0 = __umulhi(0xD2511F53u, c[0]), lo0 = 0xD2511F53u * c[0];
        uint32_t hi1 = __umulhi(0xCD9E8D57u, c[2]), lo1 = 0xCD9E8D57u * c[2];
        uint32_t n0 = hi1 ^ c[1] ^ k0, n2 = hi0 ^ c[3] ^ k1;
        c[0] = n0; c[1] = lo1; c[2] = n2; c[3] = lo0;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
}
// uniforms 2*blk, 2*blk+1 in [0,1) with 53 random bits each (numpy's random_sample recipe)
RDV_DEV void philox_uniform_pair(uint64_t seed, int64_t env_id, int32_t episode, uint32_t blk, double &u0,
                                 double &u1)
{
    uint32_t c[4] = {(uint32_t)env_id, (uint32_t)((uint64_t)env_id >> 32), (uint32_t)episode, blk};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    u0 = ((double)(c[0] >> 5) * 67108864.0 + (double)(c[1] >> 6)) * (1.0 / 9007199254740992.0);
    u1 = ((double)(c[2] >> 5) * 67108864.0 + (double)(c[3] >> 6)) * (1.0 / 9007199254740992.0);
}

}  // namespace rdv
