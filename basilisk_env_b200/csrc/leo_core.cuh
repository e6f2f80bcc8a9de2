// leo_core.cuh -- per-environment body of the fused LEO power/attitude decision step.
//
// One call of leo_step_env() replaces one `LEOPowerAttitudeSimulator.run_sim(action)`
// (/root/reference/basilisk_env/simulators/leoPowerAttitudeSimulator.py:535-644, cited SIM:line) PLUS
// the bookkeeping of `leoPowerAttEnv.step` (/root/reference/basilisk_env/envs/
// leoPowerAttitudeEnvironment.py:65-145, cited ENV:line) for ONE spacecraft: the Basilisk scheduler,
// message bus and 19 modules are flattened into a fixed schedule held in registers
// (DESIGN.md "Fused schedule").  One CUDA thread owns one spacecraft.
//
// Everything here is __host__ __device__ so that tests/hostcore can compile the same source with
// g++ and compare it with the independent oracle on a CPU-only box; the PRODUCT only ever runs it
// on the GPU (leo_kernels.cu) -- there is no CPU fallback in the library.
#pragma once
#include <math.h>
#include <stdint.h>
#include "leo_params.h"

#if defined(__CUDACC__)
#define LEO_HD __host__ __device__ __forceinline__
#define LEO_HD_NOINLINE static __host__ __device__ __noinline__
#else
#define LEO_HD inline
#define LEO_HD_NOINLINE static inline
#endif

#ifndef LEO_UNROLL_STAGES
#define LEO_UNROLL_STAGES 0
#endif

namespace leo {

// Where the functions below read the per-spacecraft parameters (bskenv_set_param_pool): a policy template parameter.
// ParBatch, the default of every batch-global kernel, returns the field of the parameter block (a constant-bank operand);
// ParEnv reads the env's own derived values.  PAt locates them.  Both are defined with the message bus (MBus) below.
struct ParBatch;
struct ParEnv;
struct PAt;

// ------------------------------------------------------------------------------------------------
// small vector algebra
// ------------------------------------------------------------------------------------------------
struct V3 { double x, y, z; };
struct M3 { V3 a, b, c; };   // rows
LEO_HD V3 mk(double x, double y, double z) { V3 v; v.x = x; v.y = y; v.z = z; return v; }
LEO_HD V3 operator+(V3 p, V3 q) { return mk(p.x + q.x, p.y + q.y, p.z + q.z); }
LEO_HD V3 operator-(V3 p, V3 q) { return mk(p.x - q.x, p.y - q.y, p.z - q.z); }
LEO_HD V3 operator-(V3 p) { return mk(-p.x, -p.y, -p.z); }
LEO_HD V3 operator*(V3 p, double s) { return mk(p.x * s, p.y * s, p.z * s); }
LEO_HD V3 operator*(double s, V3 p) { return mk(p.x * s, p.y * s, p.z * s); }
LEO_HD double dot(V3 p, V3 q) { return p.x * q.x + p.y * q.y + p.z * q.z; }
LEO_HD V3 cross(V3 p, V3 q) { return mk(p.y * q.z - p.z * q.y, p.z * q.x - p.x * q.z, p.x * q.y - p.y * q.x); }
LEO_HD double norm(V3 p) { return sqrt(dot(p, p)); }
LEO_HD V3 mv(const M3 &m, V3 v) { return mk(dot(m.a, v), dot(m.b, v), dot(m.c, v)); }
LEO_HD V3 mtv(const M3 &m, V3 v) { return m.a * v.x + m.b * v.y + m.c * v.z; }
LEO_HD V3 mv9(const double *m, V3 v)
{
    return mk(m[0] * v.x + m[1] * v.y + m[2] * v.z, m[3] * v.x + m[4] * v.y + m[5] * v.z, m[6] * v.x + m[7] * v.y + m[8] * v.z);
}
LEO_HD V3 arr(const double *p) { return mk(p[0], p[1], p[2]); }
LEO_HD V3 unit_or_zero(V3 v)
{ // Basilisk v3Normalize: scale by 1/|v|, zero vector below 1e-30
    double n = norm(v);
    return n > 1e-30 ? v * (1. / n) : mk(0., 0., 0.);
}
// Reciprocal square root / reciprocal of a finite, normal, positive operand: the MUFU seed (about 20 bits)
// followed by one third-order correction (relative error ~2^-60 before the final rounding).  Unlike
// rsqrt() / 1.0/x there is no special-operand test, hence no branch and no slow-path call in the hot loop.
LEO_HD double rsq(double x)
{
#ifdef __CUDA_ARCH__
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double t = y * y;
    double e = fma(-x, t, 1.0);
    double p = fma(e, 0.375, 0.5);
    double q = y * e;
    return fma(p, q, y);
#else
    return 1.0 / sqrt(x);
#endif
}
LEO_HD double frcp(double x)
{
#ifdef __CUDA_ARCH__
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-x, y, 1.0);
    e = fma(e, e, e);
    return fma(y, e, y);
#else
    return 1.0 / x;
#endif
}
// Fused multiply-add: a true FMA on the device; plain arithmetic on the host (tests/hostcore is built with
// -ffp-contract=off and must not depend on a libm fma()).
LEO_HD double fmad(double p, double q, double r)
{
#ifdef __CUDA_ARCH__
    return fma(p, q, r);
#else
    return p * q + r;
#endif
}
LEO_HD double clamp_asin(double x) { return x > 1. ? asin(1.) : (x < -1. ? asin(-1.) : asin(x)); }
LEO_HD double clamp_acos(double x) { return x > 1. ? acos(1.) : (x < -1. ? acos(-1.) : acos(x)); }

// Time arithmetic that feeds discrete decisions must round exactly like the scalar reference code:
// keep the compiler from contracting it into FMAs.
LEO_HD double t_mul(double p, double q)
{
#ifdef __CUDA_ARCH__
    return __dmul_rn(p, q);
#else
    return p * q;
#endif
}
LEO_HD double t_add(double p, double q)
{
#ifdef __CUDA_ARCH__
    return __dadd_rn(p, q);
#else
    return p + q;
#endif
}
LEO_HD double t_sub(double p, double q)
{
#ifdef __CUDA_ARCH__
    return __dsub_rn(p, q);
#else
    return p - q;
#endif
}
LEO_HD double t_div(double p, double q)
{
#ifdef __CUDA_ARCH__
    return __ddiv_rn(p, q);
#else
    return p / q;
#endif
}
LEO_HD double ns2sec(int64_t ns) { return t_mul((double)ns, 1e-9); }   // CurrentSimNanos*NANO2SEC

// ------------------------------------------------------------------------------------------------
// attitude kinematics (Schaub & Junkins; same conventions as Basilisk RigidBodyKinematics)
// ------------------------------------------------------------------------------------------------
LEO_HD M3 mrp_to_BN(V3 q)
{
    double d1 = dot(q, q), S = 1. - d1, inv = 1. / ((1. + d1) * (1. + d1));
    M3 C;
    C.a = mk(4. * (2. * q.x * q.x - d1) + S * S, 8. * q.x * q.y + 4. * q.z * S, 8. * q.x * q.z - 4. * q.y * S) * inv;
    C.b = mk(8. * q.y * q.x - 4. * q.z * S, 4. * (2. * q.y * q.y - d1) + S * S, 8. * q.y * q.z + 4. * q.x * S) * inv;
    C.c = mk(8. * q.z * q.x + 4. * q.y * S, 8. * q.z * q.y - 4. * q.x * S, 4. * (2. * q.z * q.z - d1) + S * S) * inv;
    return C;
}
LEO_HD V3 dcm_to_mrp(const M3 &C)
{ // C2MRP via Sheppard's method (C2EP) with the non-negative scalar part.  The largest of the four squared
  // Euler parameters is >= 1/4, so its reciprocal square root needs no guard.
    double tr = C.a.x + C.b.y + C.c.z;
    double b2_0 = (1. + tr) * 0.25, b2_1 = (1. + 2. * C.a.x - tr) * 0.25, b2_2 = (1. + 2. * C.b.y - tr) * 0.25, b2_3 = (1. + 2. * C.c.z - tr) * 0.25;
    int i = 0;
    double mx = b2_0;
    if (b2_1 > mx) { i = 1; mx = b2_1; }
    if (b2_2 > mx) { i = 2; mx = b2_2; }
    if (b2_3 > mx) { i = 3; mx = b2_3; }
    const double irt = rsq(mx), rt = mx * irt, q = 0.25 * irt;     // sqrt(mx), 1 / (4 sqrt(mx))
    double b0, b1, b2, b3;
    if (i == 0) {
        b0 = rt;
        b1 = (C.b.z - C.c.y) * q; b2 = (C.c.x - C.a.z) * q; b3 = (C.a.y - C.b.x) * q;
    } else if (i == 1) {
        b1 = rt; b0 = (C.b.z - C.c.y) * q; b2 = (C.a.y + C.b.x) * q; b3 = (C.c.x + C.a.z) * q;
    } else if (i == 2) {
        b2 = rt; b0 = (C.c.x - C.a.z) * q; b1 = (C.a.y + C.b.x) * q; b3 = (C.b.z + C.c.y) * q;
    } else {
        b3 = rt; b0 = (C.a.y - C.b.x) * q; b1 = (C.c.x + C.a.z) * q; b2 = (C.b.z + C.c.y) * q;
    }
    // a negative scalar part flips the pivot before the other two components are divided by it (C2EP):
    // the whole Euler-parameter set changes sign
    if (i != 0 && b0 < 0.) { b0 = -b0; b1 = -b1; b2 = -b2; b3 = -b3; }
    const double inv = frcp(1. + b0);
    return mk(b1 * inv, b2 * inv, b3 * inv);
}
LEO_HD V3 mrp_inner(V3 q)
{
    double m = dot(q, q);
    double f = -frcp(m);                    // discarded (possibly non-finite) when m <= 1
    return m > 1.0 ? q * f : q;
}
LEO_HD V3 mrp_sub(V3 q1, V3 q2)
{ // sigma(q1 relative to q2) with the shadow-set guard near the singular denominator, mapped to |s|<=1
    V3 s1 = q1;
    double det = 1. + dot(s1, s1) * dot(q2, q2) + 2. * dot(s1, q2);
    if (fabs(det) < 0.1) {
        s1 = s1 * (-1.0 / dot(s1, s1));
        det = 1. + dot(s1, s1) * dot(q2, q2) + 2. * dot(s1, q2);
    }
    V3 v1 = cross(s1, q2) * 2.;
    V3 res = s1 * (1. - dot(q2, q2)) - q2 * (1. - dot(s1, s1)) + v1;
    return mrp_inner(res * frcp(det));
}

// ------------------------------------------------------------------------------------------------
// Sun ephemeris latch (SpiceTask, period = step_duration, SIM:102,357) with the eclipse constants that
// only depend on the latched Sun position.  Analytic substitute for SPICE de430 (DESIGN.md).
// ------------------------------------------------------------------------------------------------
struct SunLatch {
    V3 r, v;            // Sun relative to Earth, inertial, at the message time
    double hp2;         // |s_HP|^2
    double inv_hp;      // 1/|s_HP|
    double c1off, c2off, tan1, tan2;   // R_p/sin f_1, R_p/sin f_2, tan f_1, tan f_2
};
// Chebyshev table look-up (SURVEY 8(f)-4; layout of SPK type 2 / binary PCK type 2 records): value by Clenshaw's
// recurrence on the T_k series, rate as the derivative of the same polynomial (Clenshaw on sum (k+1) a_{k+1} U_k).
// Times outside the table use its first / last segment (bskenv_set_ephemeris checks that an episode is covered).
// Branch hints for the tick loop: the rare blocks are laid out away from the straight-line path, which then touches fewer
// instruction-cache lines per tick (the L0 instruction cache holds ~6 KB; twelve warps per SM share a 32 KB L1.5)
#if defined(__GNUC__) || defined(__CUDACC__)
#define LEO_RARE(c) __builtin_expect(!!(c), 0)
#else
#define LEO_RARE(c) (c)
#endif
LEO_HD_NOINLINE void cheb_eval(const LeoEph &E, double t, V3 &val, V3 &rate)
{
    int i = (int)floor((t - E.t0) / E.seg_len);
    i = i < 0 ? 0 : (i >= E.nseg ? E.nseg - 1 : i);
    const double half = 0.5 * E.seg_len, sc = (t - (E.t0 + (i + 0.5) * E.seg_len)) / half, s2 = 2. * sc;
    double v[3], d[3];
    for (int c = 0; c < 3; c++) {
        const double *a = E.coef + ((int64_t)i * 3 + c) * E.ncoef;
        double b1 = 0., b2 = 0., d1 = 0., d2 = 0.;
        for (int k = E.ncoef - 1; k >= 1; k--) {
            const double ak = a[k];
            const double b0 = ak + s2 * b1 - b2, d0 = (double)k * ak + s2 * d1 - d2;
            b2 = b1; b1 = b0; d2 = d1; d1 = d0;
        }
        v[c] = a[0] + sc * b1 - b2;
        d[c] = d1 / half;
    }
    val = mk(v[0], v[1], v[2]); rate = mk(d[0], d[1], d[2]);
}

LEO_HD_NOINLINE SunLatch sun_latch(const LeoParams &P, int64_t msg_ns)
{
    const double D2R = 3.14159265358979323846 / 180.0;
    const double AUm = 149597870.693 * 1000.0;
    double t = ns2sec(msg_ns);
    double n = P.epoch_days + t / 86400.0;
    double nd = 1.0 / 86400.0;
    double L = (280.460 + 0.9856474 * n) * D2R, Ld = 0.9856474 * D2R * nd;
    double g = (357.528 + 0.9856003 * n) * D2R, gd = 0.9856003 * D2R * nd;
    double sg = sin(g), cg = cos(g), s2g = sin(2. * g), c2g = cos(2. * g);
    double lam = L + (1.915 * sg + 0.020 * s2g) * D2R;
    double lamd = Ld + (1.915 * cg + 0.040 * c2g) * D2R * gd;
    double eps = (23.439 - 4e-7 * n) * D2R, epsd = -4e-7 * D2R * nd;
    double R = (1.00014 - 0.01671 * cg - 0.00014 * c2g) * AUm;
    double Rd = (0.01671 * sg + 0.00028 * s2g) * gd * AUm;
    double sl = sin(lam), cl = cos(lam), se = sin(eps), ce = cos(eps);
    V3 u = mk(cl, ce * sl, se * sl);
    V3 ud = mk(-sl * lamd, ce * cl * lamd - se * sl * epsd, se * cl * lamd + ce * sl * epsd);
    SunLatch s;
    s.r = u * R;
    s.v = u * Rd + ud * R;
    if (P.eph_sun.nseg > 0) cheb_eval(P.eph_sun, t, s.r, s.v);      // ephemeris table instead of the analytic Sun
    s.hp2 = dot(s.r, s.r);
    double hp = sqrt(s.hp2);
    s.inv_hp = 1. / hp;
    double f1 = asin((P.R_sun + P.R_planet) / hp), f2 = asin((P.R_sun - P.R_planet) / hp);
    s.c1off = P.R_planet / sin(f1);
    s.c2off = P.R_planet / sin(f2);
    s.tan1 = tan(f1);
    s.tan2 = tan(f2);
    return s;
}

// ------------------------------------------------------------------------------------------------
// integrated state and equations of motion
// ------------------------------------------------------------------------------------------------
// Integrated hub state.  The wheel speeds are NOT integrated: with balanced wheels the wheel equation
// Omega_i' = u_i/Js_i - g_i.omega' is linear, so  Omega_i + g_i.omega = C_i + (u_i/Js_i) (t - t0)  holds exactly for the
// continuous solution AND for every Runge-Kutta stage and step value (linear invariants are preserved by RK
// methods).  The wheel momentum seen by the hub at stage time t0 + ct is then
//   sum_i g_i Js_i Omega_i = HB + ct tau_u - (sum_i Js_i g_i g_i^T) omega,   HB = sum_i g_i Js_i C_i, tau_u = sum_i g_i u_i,
// i.e. h = I omega + (wheel momentum) = D omega + HB + ct tau_u with the back-substitution matrix D.
struct Dyn { V3 r, v, s, w; };

// Thruster force/torque at one RK stage (thrusterDynamicEffector::computeForceTorque without ramps).
// Rare path (only while a desat pulse may still burn): state stays in global memory.
struct ThrOut { V3 F, L; int factor, active; };
// The thruster command in force (start time + on-times): constant over a dynamics tick, so the four stages of a step read
// it from registers -- one global-memory round trip per step instead of four (the path is latency-bound: DESIGN.md 6)
struct ThrCmd { double start, on[LEO_NTHR]; };
LEO_HD ThrCmd thr_cmd_load(const double *S, int64_t stride, int64_t e)
{
    ThrCmd c;
    c.start = S[(int64_t)F_THRSTART * stride + e];
#pragma unroll
    for (int k = 0; k < LEO_NTHR; k++) c.on[k] = S[(int64_t)(F_THRON + k) * stride + e];
    return c;
}
LEO_HD_NOINLINE ThrOut thr_stage(const LeoParams &P, const ThrCmd &c, double tau, double dtFire, int factor)
{
    double start = c.start;
    double tol = t_mul(-dtFire, 10E-10);
    ThrOut o;
    o.F = mk(0., 0., 0.); o.L = mk(0., 0., 0.);
    int any = 0;
#pragma unroll
    for (int k = 0; k < LEO_NTHR; k++) {
        double on = c.on[k];
        bool fire = (t_sub(t_add(on, start), tau) >= tol) && (on > 0.0);
        if (fire) {
            factor |= (1 << k);
            V3 f = arr(P.thr_dir[k]) * (P.thr_Fmax * 1.0);
            o.F = f + o.F;
            o.L = cross(arr(P.thr_loc[k]), f) + o.L;
            any = 1;
        } else {
            factor &= ~(1 << k);
        }
    }
    o.factor = factor;
    o.active = any;   // expiry is monotone in time: once nothing fires, nothing fires until the next command
    return o;
}

// MRP rotation without forming the DCM:  [BN] = I + (8 [s~]^2 - 4 (1 - s^2) [s~]) / (1 + s^2)^2
struct MrpRot { double a8, b4, oms2; };       // 8/(1+s^2)^2, 4(1-s^2)/(1+s^2)^2 and 1 - s^2
LEO_HD MrpRot mrp_rot(V3 s)
{
    double s2 = dot(s, s), den = 1. + s2, inv = frcp(den * den);
    MrpRot m; m.oms2 = 1. - s2; m.a8 = 8. * inv; m.b4 = 4. * m.oms2 * inv;
    return m;
}
LEO_HD V3 rot_BN(const MrpRot &m, V3 s, V3 x)   // [BN] x   (inertial -> body)
{
    V3 t = cross(s, x), uu = cross(s, t);
    return x + uu * m.a8 - t * m.b4;
}
LEO_HD V3 rot_NB(const MrpRot &m, V3 s, V3 x)   // [BN]^T x (body -> inertial)
{
    V3 t = cross(s, x), uu = cross(s, t);
    return x + uu * m.a8 + t * m.b4;
}

// Sun "indirect" third-body term  -mu_sun * rs / |rs|^3  at Sun position rs (depends on time only)
LEO_HD V3 sun_indirect(const LeoParams &P, V3 rs)
{
    double is = rsq(dot(rs, rs));
    return rs * (-P.mu_sun * (is * is * is));
}

// ------------------------------------------------------------------------------------------------
// flight software, one pass per fswRate
// ------------------------------------------------------------------------------------------------
struct AttRef { V3 sigma_RN, omega_RN_N, domega_RN_N; };
struct AttGuid { V3 sigma_BR, omega_BR_B, omega_RN_B, domega_RN_B; };

LEO_HD AttRef hill_point(V3 r, V3 v, V3 cel_r, V3 cel_v)
{ // hillPoint.computeHillPointingReference (v3Normalize: zero vector below a norm of 1e-30)
    V3 rel_r = r - cel_r, rel_v = v - cel_v;
    const double r2 = dot(rel_r, rel_r);
    double ir = rsq(r2);
    ir = r2 > 1e-60 ? ir : 0.0;
    V3 h = cross(rel_r, rel_v);
    const double h2 = dot(h, h);
    double ih = rsq(h2);
    ih = h2 > 1e-60 ? ih : 0.0;
    M3 RN;
    RN.a = rel_r * ir;
    RN.c = h * ih;
    RN.b = cross(RN.c, RN.a);
    AttRef o;
    o.sigma_RN = dcm_to_mrp(RN);
    double rm = r2 * ir, hm = h2 * ih, dfdt = 0., ddfdt2 = 0.;
    if (rm > 1.) {
        dfdt = hm * ir * ir;
        ddfdt2 = -2.0 * dot(rel_v, RN.a) * ir * dfdt;
    }
    o.omega_RN_N = RN.c * dfdt;            // [RN]^T (0, 0, dfdt)
    o.domega_RN_N = RN.c * ddfdt2;
    return o;
}
LEO_HD AttGuid att_tracking_error(V3 sigma_BN, V3 omega_BN_B, const AttRef &ref)
{ // attTrackingError.computeAttitudeError with sigma_R0R = 0 (addMRP with zero is the identity + inner-set map)
    AttGuid g;
    V3 sigma_RN = mrp_inner(ref.sigma_RN);
    g.sigma_BR = mrp_sub(sigma_BN, sigma_RN);
    MrpRot BN = mrp_rot(sigma_BN);
    g.omega_RN_B = rot_BN(BN, sigma_BN, ref.omega_RN_N);
    g.omega_BR_B = omega_BN_B - g.omega_RN_B;
    g.domega_RN_B = rot_BN(BN, sigma_BN, ref.domega_RN_N);
    return g;
}
template <class PA = ParBatch>
LEO_HD V3 mrp_feedback(const LeoParams &P, const AttGuid &g, const double *S, int64_t stride, int64_t e)
{ // MRP_Feedback with Ki < 0 (integral off) and no wheel feed-forward wired (SIM:440-449)
    double buf[9];
    const double *Ifsw = PA::I_fsw(P, S, stride, e, buf);
    V3 w = g.omega_BR_B + g.omega_RN_B;
    V3 Lr = g.omega_BR_B * PA::Pgain(P, S, stride, e) + g.sigma_BR * PA::K(P, S, stride, e);
    Lr = Lr - cross(g.omega_RN_B, mv9(Ifsw, w));
    Lr = Lr - mv9(Ifsw, g.domega_RN_B - cross(w, g.omega_RN_B));
    return -Lr;
}

// thrForceMapping.Update for the on-pulsing octet: minimum-norm impulses, subtract-min, saturation scaling
LEO_HD_NOINLINE void thr_force_mapping(const LeoParams &P, V3 Lr, double (&F)[LEO_NTHR])
{
    double mn = 0.0;
    for (int i = 0; i < LEO_NTHR; i++) {
        F[i] = P.thr_W[i][0] * Lr.x + P.thr_W[i][1] * Lr.y + P.thr_W[i][2] * Lr.z;
        if (F[i] < mn) mn = F[i];
    }
    if (P.thrForceSign > 0)
        for (int i = 0; i < LEO_NTHR; i++) F[i] -= mn;
    // computeTorqueAngErr
    double ang = 0.0;
    if (norm(Lr) > P.tfm_eps) {
        V3 tau = mk(0., 0., 0.);
        for (int i = 0; i < LEO_NTHR; i++) {
            double f = fabs(F[i]) < P.thr_Fmax ? F[i] : P.thr_Fmax * fabs(F[i]) / F[i];
            tau = tau + mk(P.thr_D[0][i], P.thr_D[1][i], P.thr_D[2][i]) * f;
        }
        double c = dot(unit_or_zero(Lr), unit_or_zero(tau));
        if (c < 1.0) ang = clamp_acos(c);
    }
    if (ang > P.tfm_angErrThresh) {
        double mx = 0.0;
        for (int i = 0; i < LEO_NTHR; i++) {
            double fr = fabs(F[i]) / P.thr_Fmax;
            if (fr > mx) mx = fr;
        }
        if (mx > 1.0)
            for (int i = 0; i < LEO_NTHR; i++) F[i] = (1.0 / mx) * F[i];
    }
}

// rwDesatTask = thrMomentumManagement -> thrForceMapping -> thrMomentumDumping (SIM:488-490).
// wheel speeds = the RWSpeed message of the previous dynamics tick (zeros before the first tick).
// Returns 1 when the dumping block ran and left nothing to do: no on-time remaining on any thruster and a zero
// command (the chain is then "quiet": until the next Reset every pass only advances the rest counter and the
// time tag, see fsw_pass).
template <int NRW, class PA = ParBatch>
LEO_HD_NOINLINE int fsw_desat(const LeoParams &P, double *S, int64_t *I, int64_t stride, int64_t e, int64_t now_ns,
                              const double (&ws)[NRW])
{
#define SD(f) S[(int64_t)(f) * stride + e]
#define SI(f) I[(int64_t)(f) * stride + e]
    // thrMomentumManagement: one-shot after Reset
    if (SI(I_INITREQ) == 1) {
        V3 hs = mk(0., 0., 0.);
        for (int i = 0; i < NRW; i++) hs = hs + arr(P.gs[i]) * (P.Js[i] * ws[i]);
        double hm = norm(hs);
        const double hs_min = PA::hs_min(P, S, stride, e);
        V3 dH = (hm < hs_min) ? mk(0., 0., 0.) : hs * (-(hm - hs_min) / hm);
        SD(F_DELTAH) = dH.x; SD(F_DELTAH + 1) = dH.y; SD(F_DELTAH + 2) = dH.z;
        SI(I_DHTIME) = now_ns;
        SI(I_INITREQ) = 0;
    }
    // thrMomentumDumping (thrForceMapping evaluated lazily: its output is only consumed on a new Delta H)
    double tOn[LEO_NTHR];
    for (int k = 0; k < LEO_NTHR; k++) tOn[k] = 0.0;
    int64_t prior = SI(I_DUMPPRIOR);
    if (prior != 0) {
        double dt = t_mul((double)(now_ns - prior), 1e-9);
        if (dt < 0.0) dt = 0.0;
        int64_t tdh = SI(I_DHTIME);
        if (SI(I_LASTDH) != tdh) {
            SI(I_LASTDH) = tdh;
            SI(I_DUMPCNT) = 0;
            double F[LEO_NTHR];
            thr_force_mapping(P, mk(SD(F_DELTAH), SD(F_DELTAH + 1), SD(F_DELTAH + 2)), F);
            for (int k = 0; k < LEO_NTHR; k++) SD(F_THRREM + k) = F[k] / P.thr_Fmax;
        }
        if (SI(I_DUMPCNT) <= 0) {
            for (int k = 0; k < LEO_NTHR; k++) {
                double rem = SD(F_THRREM + k);
                tOn[k] = rem;
                if (rem > 0.0) SD(F_THRREM + k) = t_sub(rem, dt);
            }
            SI(I_DUMPCNT) = P.maxCounterValue;
        } else {
            SI(I_DUMPCNT) -= 1;
        }
        for (int k = 0; k < LEO_NTHR; k++) {
            if (tOn[k] < P.thrMinFireTime) tOn[k] = 0.0;
            if (SD(F_THRREM + k) < 0.0) SD(F_THRREM + k) = 0.0;
            if (tOn[k] >= dt) tOn[k] = dt;
        }
    }
    SI(I_DUMPPRIOR) = now_ns;
    int quiet = prior != 0;
    for (int k = 0; k < LEO_NTHR; k++) {
        SD(F_THRCMD + k) = tOn[k];
        if (tOn[k] != 0.0 || SD(F_THRREM + k) != 0.0) quiet = 0;
    }
    return quiet;
#undef SD
#undef SI
}

// thrusterDynamicEffector.UpdateState on a NEW on-time message (ConfigureThrustRequests)
LEO_HD_NOINLINE int thr_latch(const LeoParams &P, double *S, int64_t *I, int64_t stride, int64_t e, int64_t cmd_ns, int factor)
{
    int any = 0;
    for (int k = 0; k < LEO_NTHR; k++) {
        double cmd = S[(int64_t)(F_THRCMD + k) * stride + e], on;
        bool burning = (factor >> k) & 1;
        if (cmd >= P.thr_MinOnTime) {
            on = cmd;
            if (!burning) I[(int64_t)(I_FIRE + k) * stride + e] += 1;
        } else {
            on = burning ? cmd : 0.0;
        }
        S[(int64_t)(F_THRON + k) * stride + e] = on;
        if (on > 0.0) any = 1;
    }
    S[(int64_t)F_THRSTART * stride + e] = t_mul((double)cmd_ns, 1.0E-9);
    return (any || factor != 0) ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------
// eclipse (conical shadow model) and solar panel, per environment tick
// ------------------------------------------------------------------------------------------------
// eclipse.cpp computePercentShadow, literal form (apparent radii a, b and separation c as angles).  Cold path:
// only used when the small-Sun expansion of penumbra_fraction() below does not apply.
LEO_HD_NOINLINE double percent_shadow_general(double a, double b, double c)
{
    const double PI = 3.14159265358979323846;
    double shadow = 1.0;
    if (c < b - a) {
        shadow = 0.0;
    } else if (c < a - b) {
        double area = PI * a * a - PI * b * b;
        shadow = 1. - area / (PI * a * a);
    } else if (c < a + b) {
        double x = (c * c + a * a - b * b) / (2. * c);
        double y = sqrt(a * a - x * x);
        double area = a * a * clamp_acos(x / a) + b * b * clamp_acos((c - x) / b) - c * y;
        shadow = 1. - area / (PI * a * a);
    }
    return shadow;
}
// asin(t) for |t| <= 0.1 (Maclaurin series through t^13: truncation < 1e-17 relative)
LEO_HD double asin_small(double t)
{
    const double t2 = t * t;
    double p = fmad(t2, 231. / 13312., 63. / 2816.);
    p = fmad(p, t2, 35. / 1152.); p = fmad(p, t2, 5. / 112.); p = fmad(p, t2, 3. / 40.); p = fmad(p, t2, 1. / 6.);
    return fmad(t * t2, p, t);
}
#if defined(__CUDACC__)
// R(z) ~ (asin(sqrt z) / sqrt z - 1) / z on [0, 1/4]: degree-12 Chebyshev interpolant (scripts/gen_asin_poly.py; the error of
// s + s z R(z) against asin(s) on |s| <= 1/2 is 5.8e-17, i.e. the rounding of the result).  In constant memory: see LEO_K.
__constant__ double LEO_ASIN_C[13] = {
    0.16666666666666669, 0.07499999999998433, 0.04464285714635543, 0.030381944138531247, 0.02237217294214989,
    0.017352392720869973, 0.013971212973552933, 0.011479177415184906, 0.01032281435018578, 0.005457506718640358,
    0.01740087944269402, -0.014851887071247204, 0.028757851367421566};
// asin_small() in Estrin form with its coefficients, the planet-segment series, pi/2 (hi, lo) and 1/pi as constant-bank operands
// (a 64-bit literal costs two uniform-register moves per use: the libm-free penumbra was 240 UMOV of 830 instructions)
__constant__ double LEO_PEN_K[14] = {1. / 6., 3. / 40., 5. / 112., 35. / 1152., 63. / 2816., 231. / 13312.,
                                     2. / 3., 1. / 5., 3. / 28., 5. / 72.,
                                     1.57079632679489655800e+00, 6.12323399573676603587e-17, 0.31830988618379067154, 3.14159265358979323846};
#endif
#if defined(__CUDA_ARCH__)
// Device-side inverse trigonometry of the penumbra evaluation.  The penumbra is a rare, divergent path, but a lone warp (small
// batches) pays its full latency: libm's asin / acos / sqrt / divide cost ~2700 cycles per evaluation there, these ~1000.
// No special operands: callers pass finite arguments inside the domain.
LEO_HD double asin_poly(double s, double z)        // asin(s) for |s| <= 1/2, z = s^2 (Estrin form)
{
    const double *c = LEO_ASIN_C;
    const double z2 = z * z, z4 = z2 * z2, z8 = z4 * z4;
    const double p0 = fma(c[1], z, c[0]), p1 = fma(c[3], z, c[2]), p2 = fma(c[5], z, c[4]), p3 = fma(c[7], z, c[6]);
    const double p4 = fma(c[9], z, c[8]), p5 = fma(c[11], z, c[10]);
    const double q0 = fma(p1, z2, p0), q1 = fma(p3, z2, p2), q2 = fma(p5, z2, p4);
    const double r0 = fma(q1, z4, q0), r1 = fma(c[12], z4, q2);
    return fma(s * z, fma(r1, z8, r0), s);
}
LEO_HD double sqrt_pos(double x) { return x > 1e-290 ? x * rsq(x) : 0.0; }      // sqrt of a non-negative operand (~1 ulp)
LEO_HD double asin_small_dev(double t)
{
    const double *k = LEO_PEN_K;
    const double z = t * t, z2 = z * z, z4 = z2 * z2;
    const double p0 = fma(k[1], z, k[0]), p1 = fma(k[3], z, k[2]), p2 = fma(k[5], z, k[4]);
    return fma(t * z, fma(p2, z4, fma(p1, z2, p0)), t);
}
LEO_HD double acos_dev(double q)                   // acos with the argument clamped to [-1, 1] (clamp_acos)
{
    q = fmin(fmax(q, -1.0), 1.0);
    const double aq = fabs(q);
    const bool small = aq <= 0.5;
    const double z = small ? q * q : fma(-0.5, aq, 0.5);       // |q| > 1/2: acos |q| = 2 asin sqrt((1 - |q|) / 2)
    const double sv = small ? q : sqrt_pos(z);
    const double r = asin_poly(sv, z);
    const double pio2_hi = LEO_PEN_K[10], pio2_lo = LEO_PEN_K[11];
    if (small) return pio2_hi - (r - pio2_lo);
    return q > 0. ? 2. * r : (2. * pio2_hi - 2. * r) + 2. * pio2_lo;
}
LEO_HD double asin_dev_hi(double x)                // asin for 1/2 <= x < 1
{
    const double z = fma(-0.5, x, 0.5);
    const double r = asin_poly(sqrt_pos(z), z);
    return (LEO_PEN_K[10] - 2. * r) + LEO_PEN_K[11];
}
#endif
// Fraction of the solar disk left visible inside the penumbra (eclipse.cpp computePercentShadow: overlap of two
// disks of apparent radii a = asin(R_sun/|r_HB|), b = asin(R_p/|s_BP|) whose centres are c apart).
// The Sun's disk is small (a = 4.65e-3 rad) and c is within a of b, so the reference's five inverse
// trigonometric calls reduce to two: a and the offset delta = c - b come from their sines (series; sin(delta)
// = sin c cos b - cos c sin b is formed algebraically, which also avoids the cancellation in c - b), and the
// planet's circular segment b^2 (phi - sin phi cos phi), sin phi = y/b <= a/b, is a short series.  The same
// lens-area formula, regrouped as (Sun segment) + (planet segment); agreement with the literal form is ~1e-13.
//   ir = 1/|s_BP|, id = 1/|r_HB|, rdh = s_BP . r_HB
#if defined(__CUDA_ARCH__) && !defined(LEO_LIBM_PENUMBRA)
// Device form: the same formula; reciprocals, square roots and the inverse trigonometric functions without libm's special-operand
// paths, polynomial coefficients as constant-bank operands, Estrin forms (this rare, divergent path sits on a lone warp's chain
// in the small-batch organisations: 2700 cycles per evaluation with libm, 2000 with the first libm-free form).
LEO_HD_NOINLINE double penumbra_cold(const LeoParams &P, double ta, double tb, double cc)
{
    return percent_shadow_general(clamp_asin(ta), clamp_asin(tb), clamp_acos(cc));
}
LEO_HD_NOINLINE double penumbra_fraction(const LeoParams &P, double ir, double id, double rdh)
{
    const double *k = LEO_PEN_K;
    const double ta = P.R_sun * id, tb = P.R_planet * ir;             // sin a, sin b
    const double cc = -rdh * ir * id;                                  // cos c
    const double sc2 = 1. - cc * cc, cb2 = 1. - tb * tb;
    const double sd = (sc2 > 0. && cb2 > 0.) ? sqrt_pos(sc2) * sqrt_pos(cb2) - cc * tb : 2.0;   // sin(c - b)
    if (!(ta <= 0.05 && fabs(sd) <= 0.1 && tb >= 20. * ta && tb < 1. && tb >= 0.5))    // not a small Sun next to a big, near limb
        return penumbra_cold(P, ta, tb, cc);
    const double a = asin_small_dev(ta), d = asin_small_dev(sd), b = asin_dev_hi(tb);
    if (d < -a) return 0.0;                                            // c < b - a: total
    if (!(d < a)) return 1.0;                                          // c >= a + b: clear   (c < a - b cannot occur: b > a)
    const double c = b + d, a2 = a * a, ia = frcp(a), ib = frcp(b);
    const double x = (a2 + d * (2. * b + d)) * frcp(2. * c);
    double y2 = a2 - x * x;
    if (y2 < 0.) y2 = 0.;
    const double y = sqrt_pos(y2);
    const double u = y * ib, u2 = u * u;
    const double seg = fma(fma(k[9], u2, k[8]), u2 * u2, fma(k[7], u2, k[6]));
    const double area = a2 * acos_dev(x * ia) - x * y + (b * b) * (u * u2) * seg;
    return 1. - area * (ia * ia) * k[12];
}
#else
LEO_HD_NOINLINE double penumbra_fraction(const LeoParams &P, double ir, double id, double rdh)
{
    const double PI = 3.14159265358979323846;
    const double ta = P.R_sun * id, tb = P.R_planet * ir;             // sin a, sin b
    const double cc = -rdh * ir * id;                                  // cos c
    const double sc2 = 1. - cc * cc, cb2 = 1. - tb * tb;
    const double sd = (sc2 > 0. && cb2 > 0.) ? sqrt(sc2) * sqrt(cb2) - cc * tb : 2.0;   // sin(c - b)
    if (!(ta <= 0.05 && fabs(sd) <= 0.1 && tb >= 20. * ta && tb < 1.))                  // not a small Sun next to a big limb
        return percent_shadow_general(clamp_asin(ta), clamp_asin(tb), clamp_acos(cc));
    const double a = asin_small(ta), d = asin_small(sd), b = asin(tb);
    if (d < -a) return 0.0;                                            // c < b - a: total
    if (!(d < a)) return 1.0;                                          // c >= a + b: clear   (c < a - b cannot occur: b > a)
    const double c = b + d;
    const double x = (a * a + d * (2. * b + d)) / (2. * c);
    double y2 = a * a - x * x;
    if (y2 < 0.) y2 = 0.;
    const double y = sqrt(y2);
    const double u = y / b, u2 = u * u;
    double seg = fmad(u2, 5. / 72., 3. / 28.);
    seg = fmad(seg, u2, 1. / 5.); seg = fmad(seg, u2, 2. / 3.);
    const double area = a * a * clamp_acos(x / a) - x * y + (b * b) * (u * u2) * seg;
    return 1. - area / (PI * a * a);
}
#endif
// PARITY BUILD ONLY (-DLEO_LITERAL_ECLIPSE, libbskenv_literal.so; tests/test_gpu_round2.py): the disk overlap exactly as
// eclipse.cpp writes it -- norms by sqrt, apparent radii and separation through asin / acos of quotients, the lens-area
// formula in its original grouping -- so that the deviation of the regrouped production form above from the reference's
// arithmetic is a MEASURED quantity (DESIGN.md section 9, deviation D7), not an asserted one.
LEO_HD_NOINLINE double penumbra_literal(const LeoParams &P, V3 sun_r, V3 r)
{
    const V3 r_HB = sun_r - r;
    const double nh = sqrt(dot(r_HB, r_HB)), ns = sqrt(dot(r, r));
    const double a = clamp_asin(P.R_sun / nh), b = clamp_asin(P.R_planet / ns), c = clamp_acos((-dot(r, r_HB)) / (ns * nh));
    return percent_shadow_general(a, b, c);
}
// Shadow factor of the planet at the origin (zeroBase earth), eclipse.UpdateState + computePercentShadow.
// Full sun / umbra are decided on squared cone radii (no sqrt, no transcendentals); a relative guard band of
// ECL_BAND around both cone surfaces, and the penumbra itself, go through the disk-overlap formula.
// The cone tests and the apparent-disk tests of computePercentShadow describe the same geometry (tangent
// cones of two spheres), so outside the band both give exactly 0.0 or 1.0 (tests/test_hostcore_eclipse.py).
//   s2 = r.r, ir = 1/|r|, r_HB = sun_r - r, hb2 = r_HB.r_HB, id = 1/|r_HB|
#define ECL_BAND 1e-7
// Cone tests only: returns the shadow factor where it is decided by the cones (1.0 lit / outside the gate, 0.0 umbra) and sets
// `penumbra` when the disk-overlap formula has to be evaluated (the rare, divergent part: the tick loop calls it out of line
// AFTER the common-path arithmetic of the tick, so that the cone tests stay in one straight-line block with the rest).
LEO_HD double eclipse_cones(const LeoParams &P, const double (&ec)[6], V3 sun_r, V3 r, double s2, double hb2, bool &penumbra)
{
    const double hp2 = ec[0], inv_hp = ec[1], c1off = ec[2], c2off = ec[3], tan1 = ec[4], tan2 = ec[5];
    const double s0 = -dot(r, sun_r) * inv_hp;
    const double c1 = s0 + c1off, c2 = s0 - c2off;
    const double l2sq = s2 - s0 * s0;                       // l^2
    const double l1 = c1 * tan1, l2 = c2 * tan2;
    const double p2 = l1 * l1, u2 = l2 * l2;                // squared penumbra / umbra cone radii at this depth
    const bool lit = (hb2 < hp2)                            // spacecraft on the sunny side of the planet
                     || (l2sq > p2 * (1. + ECL_BAND) && l2sq > u2 * (1. + ECL_BAND));       // outside both cones
    const bool dark = l2sq < u2 * (1. - ECL_BAND) && c2 < 0. && P.R_sun > P.R_planet;      // inside the umbra, before its apex
    // eclipse.cpp gate `fabs(l) < fabs(l_2) || fabs(l) < fabs(l_1)`, on the squares
    penumbra = !lit && !dark && (l2sq < u2 || l2sq < p2);
    return (lit || !dark) ? 1.0 : 0.0;
}
LEO_HD double eclipse_core(const LeoParams &P, const double (&ec)[6], V3 sun_r, V3 r, double s2, double ir, V3 r_HB, double hb2, double id)
{
    bool pen;
    double f = eclipse_cones(P, ec, sun_r, r, s2, hb2, pen);
    if (pen) f = penumbra_fraction(P, ir, id, dot(r, r_HB));
    return f;
}
LEO_HD double eclipse_factor(const LeoParams &P, const SunLatch &sun, V3 r, double s2, V3 r_HB, double hb2)
{
    const double ec[6] = {sun.hp2, sun.inv_hp, sun.c1off, sun.c2off, sun.tan1, sun.tan2};
    return eclipse_core(P, ec, sun.r, r, s2, rsq(s2), r_HB, hb2, rsq(hb2));
}

// ------------------------------------------------------------------------------------------------
// counter-based RNG for device-side initial conditions (Philox4x32-10)
// ------------------------------------------------------------------------------------------------
LEO_HD void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t (&out)[4])
{
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1, n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
struct IcRng {
    uint64_t seed, env; uint32_t episode, block; uint32_t buf[4]; int have;
    LEO_HD double u01()
    { // 53-bit uniform in [0,1)
        if (have == 0) {
            philox4x32((uint32_t)env, (uint32_t)(env >> 32), episode, block++, (uint32_t)seed, (uint32_t)(seed >> 32), buf);
            have = 2;
        }
        int j = 2 - have;
        have--;
        uint64_t x = ((uint64_t)buf[2 * j + 1] << 32) | buf[2 * j];
        return (double)(x >> 11) * (1.0 / 9007199254740992.0);
    }
    LEO_HD double uniform(double lo, double hi) { return lo + (hi - lo) * u01(); }
};
// Same distributions as the reference's sampler (SURVEY 8a R3/R4): leo_orbit.sampled_400km,
// sc_attitudes.random_tumble(1e-5), set_ICs N(0,1)^3 / U(-800,800)^3 rpm / U(8,20) Wh.
LEO_HD_NOINLINE void sample_ic(const LeoParams &P, int64_t global_env, int64_t episode, double (&ic)[19])
{
    IcRng g; g.seed = P.seed; g.env = (uint64_t)global_env; g.episode = (uint32_t)episode; g.block = 0; g.have = 0;
    const double PI = 3.14159265358979323846, D2R = PI / 180.0;
    double a = 6371 * 1000.0 + 500. * 1000;
    double ecc = g.uniform(0, 0.05), inc = g.uniform(-90 * D2R, 90 * D2R);
    double Om = g.uniform(0 * D2R, 360 * D2R), om = g.uniform(0 * D2R, 360 * D2R), f = g.uniform(0 * D2R, 360 * D2R);
    { // orbitalMotion.elem2rv, non-rectilinear branch
        double mu = P.mu_c, p = a * (1.0 - ecc * ecc), r = p / (1.0 + ecc * cos(f)), th = om + f, h = sqrt(mu * p);
        ic[0] = r * (cos(th) * cos(Om) - cos(inc) * sin(th) * sin(Om));
        ic[1] = r * (cos(th) * sin(Om) + cos(inc) * sin(th) * cos(Om));
        ic[2] = r * (sin(th) * sin(inc));
        ic[3] = -mu / h * (cos(Om) * (ecc * sin(om) + sin(th)) + cos(inc) * (ecc * cos(om) + cos(th)) * sin(Om));
        ic[4] = -mu / h * (sin(Om) * (ecc * sin(om) + sin(th)) - cos(inc) * (ecc * cos(om) + cos(th)) * cos(Om));
        ic[5] = mu / h * (ecc * cos(om) + cos(th)) * sin(inc);
    }
    for (int k = 0; k < 3; k++) ic[6 + k] = g.uniform(0, 1.0);
    for (int k = 0; k < 3; k++) ic[9 + k] = g.uniform(-0.00001, 0.00001);
    { // three standard normals by Box-Muller (the fourth is discarded)
        double u1 = 1.0 - g.u01(), u2 = g.u01(), u3 = 1.0 - g.u01(), u4 = g.u01();
        double r1 = sqrt(-2.0 * log(u1)), r2 = sqrt(-2.0 * log(u3));
        ic[12] = r1 * cos(2. * PI * u2); ic[13] = r1 * sin(2. * PI * u2); ic[14] = r2 * cos(2. * PI * u4);
    }
    for (int k = 0; k < 3; k++) ic[15 + k] = g.uniform(-800, 800);
    ic[18] = g.uniform(8. * 3600., 20. * 3600.);
}

// ------------------------------------------------------------------------------------------------
// reset: LEOPowerAttitudeSimulator.__init__ (SIM:67-117) + InitializeSimulationAndDiscover, and the
// initial observation of leoPowerAttEnv.reset (ENV:188-190)
// ------------------------------------------------------------------------------------------------
// rw_set 1: the fourth wheel starts at the mean speed of the three sampled ones [RPM]
LEO_HD double ic_w4(const double (&ic)[19]) { return (ic[15] + ic[16] + ic[17]) / 3.0; }
// The initial observation of a reset from its ICs (w4 = ic_w4(ic), taken by the caller before it writes the state: the
// stores may alias `ic` for all the compiler knows): SIM:347-351 (wheel speeds in RPM, un-converted: SIM:306) then
// ENV:189-190.  Also what bskenv_restore returns for an env fresh from a reset.
LEO_HD void reset_obs(const LeoParams &P, const double (&ic)[19], double w4, double *obs)
{
    obs[0] = sqrt(ic[6] * ic[6] + ic[7] * ic[7] + ic[8] * ic[8]);
    obs[1] = sqrt(ic[9] * ic[9] + ic[10] * ic[10] + ic[11] * ic[11]);
    obs[2] = sqrt(ic[15] * ic[15] + ic[16] * ic[16] + ic[17] * ic[17] + (P.nrw == 4 ? w4 * w4 : 0.0)) / P.wheel_limit;
    obs[3] = ic[18] / 3600.0 / P.power_max;
    obs[4] = 0.0;
}

template <class PA = ParBatch>
LEO_HD void leo_reset_env(const LeoParams &P, double *S, int64_t *I, int64_t stride, int64_t e, const double (&ic)[19],
                          double *obs /* 5, may be null */)
{
#define SD(f) S[(int64_t)(f) * stride + e]
#define SI(f) I[(int64_t)(f) * stride + e]
    for (int f = 0; f < LEO_ND; f++) SD(f) = 0.0;
    int64_t episode = SI(I_EPISODE);
    for (int f = 0; f < LEO_NI; f++) SI(f) = 0;
    SI(I_EPISODE) = episode;
    for (int k = 0; k < 12; k++) SD(F_R + k) = ic[k];
    const double dist_mag = PA::dist_mag(P, S, stride, e);
    for (int k = 0; k < 3; k++) SD(F_LDIST + k) = dist_mag * ic[12 + k];               // SIM:295 (quirk Q4: raw vector)
    for (int k = 0; k < 3; k++) SD(F_WHL + k) = ic[15 + k] * P.wheel_rpm2rad;       // SIM:303-305
    const double w4 = ic_w4(ic);
    if (P.nrw == 4) SD(F_WHL + 3) = w4 * P.wheel_rpm2rad;
    SD(F_E) = ic[18];
    SI(I_TICK) = -1;
    SI(I_MASK) = LEO_TASK_ALL;       // every task starts enabled
    SI(I_INITREQ) = 1;               // Reset_thrMomentumManagement
    if (obs) reset_obs(P, ic, w4, obs);
#undef SD
#undef SI
}

// ------------------------------------------------------------------------------------------------
// one decision interval of one environment
// ------------------------------------------------------------------------------------------------
struct StepOut { double ob[5]; double reward; int done; int reason; };

// Per-thread "message bus": the flight-software messages, the Sun latch and the data of the rare paths live in
// SHARED memory for the duration of the launch ([field][thread], conflict-free, immediate-offset LDS/STS), so
// that none of it occupies registers in the tick loop and none of it costs address arithmetic.  Fields M_GUID..
// M_RWCMD+3 mirror the persistent state fields F_GUID..F_RWCMD+3 (loaded at entry, written back at exit); the
// rest is scratch.  On the host (tests/hostcore) the bus is a plain array.
enum LeoMField : int {
    M_GUID = 0,      // att_guidance (12)
    M_REF = 12,      // att_reference (9)
    M_LR = 21,       // commandedControlTorque (3)
    M_RWCMD = 24,    // rwTorqueCommand (4)
    M_SUNR = 28,     // Sun latch: position (3), velocity (3)
    M_SUNV = 31,
    M_ECL = 34,      // eclipse constants of the latch: |s_HP|^2, 1/|s_HP|, R_p/sin f1, R_p/sin f2, tan f1, tan f2
    M_LEXT = 40,     // extForceTorque torque (3)
    M_FM = 43,       // held thruster force / mass, body frame (3)
    M_U = 46,        // latched wheel motor torques u_current (4)
    M_LTHR = 50,     // held thruster torque (3), zero outside burns
    M_TNEXT = 53,    // earliest expiry of a burning thruster
    LEO_NM = 54,     // (battery charge and shadow factor are carried in registers)
    // only allocated by the planet-fixed gravity variant (J2 == 2):
    M_PFIX = 54,     // J20002Pfix of the last SPICE message (9, row-major)
    M_PFIXD = 63,    // J20002Pfix_dot (9)
    LEO_NM_PFIX = 72,
    // only allocated by the per-env parameter kernel (ParEnv): the stage-rate parameters PE_INV_MASS..PE_DRAGKA+2
    M_PE = 54,
    LEO_NM_PENV = 64
};
#define LEO_M_MIRROR 28          // number of leading bus fields that mirror state fields starting at F_GUID
struct MBus {
    uint32_t a;      // device: shared-window byte address of this thread's column
    double *p;       // host (tests/hostcore): plain array of LEO_NM doubles
};
LEO_HD double mld(MBus m, int f)
{
#ifdef __CUDA_ARCH__
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(m.a + (uint32_t)f * (uint32_t)(LEO_BLOCK * 8)) : "memory");
    return v;
#else
    return m.p[f];
#endif
}
LEO_HD void mst(MBus m, int f, double v)
{
#ifdef __CUDA_ARCH__
    asm volatile("st.shared.f64 [%0], %1;" : : "r"(m.a + (uint32_t)f * (uint32_t)(LEO_BLOCK * 8)), "d"(v) : "memory");
#else
    m.p[f] = v;
#endif
}
LEO_HD V3 mld3(MBus m, int f) { return mk(mld(m, f), mld(m, f + 1), mld(m, f + 2)); }
LEO_HD void mst3(MBus m, int f, V3 v) { mst(m, f, v.x); mst(m, f + 1, v.y); mst(m, f + 2, v.z); }

// ------------------------------------------------------------------------------------------------
// per-spacecraft parameters (see ParBatch above)
// ------------------------------------------------------------------------------------------------
struct PAt { MBus m; const double *S; int64_t stride, e; };   // an env's bus column and state column
struct ParBatch {
    // read at every RK stage
    LEO_HD static void load_bus(const LeoParams &, const PAt &) {}
    LEO_HD static double inv_mass(const LeoParams &P, const PAt &) { return P.inv_mass; }
    LEO_HD static double D(const LeoParams &P, const PAt &, int k) { return P.D[4 * k]; }          // diagonal (DIAG path)
    LEO_HD static double Dinv(const LeoParams &P, const PAt &, int k) { return P.Dinv[4 * k]; }
    LEO_HD static double dragKa(const LeoParams &P, const PAt &, int k) { return P.dragKa[k]; }
    // read once per dynamics tick, per flight-software pass or per reset
    LEO_HD static double rho0(const LeoParams &P, const double *, int64_t, int64_t) { return P.rho0; }
    LEO_HD static double inv_H(const LeoParams &P, const double *, int64_t, int64_t) { return P.inv_H; }
    LEO_HD static double panel_coef(const LeoParams &P, const double *, int64_t, int64_t) { return P.panel_coef; }
    LEO_HD static double sink_power(const LeoParams &P, const double *, int64_t, int64_t) { return P.sink_power; }
    LEO_HD static double capacity(const LeoParams &P, const double *, int64_t, int64_t) { return P.capacity; }
    LEO_HD static double K(const LeoParams &P, const double *, int64_t, int64_t) { return P.K; }
    LEO_HD static double Pgain(const LeoParams &P, const double *, int64_t, int64_t) { return P.P; }
    LEO_HD static const double *I_fsw(const LeoParams &P, const double *, int64_t, int64_t, double *) { return P.I_fsw; }
    LEO_HD static double hs_min(const LeoParams &P, const double *, int64_t, int64_t) { return P.hs_min; }
    LEO_HD static double dist_mag(const LeoParams &P, const double *, int64_t, int64_t) { return P.dist_mag; }
};
// The env's own values: the LEO_NPD block behind the state fields (leo_params.h: LeoPField).  The stage-rate values are
// copied into this thread's bus column once per call of leo_step_env (load_bus) and read from shared memory at every
// stage; the others are read from global memory where they are used.  LEO_PENV_GLOBAL (measurement builds, DESIGN.md
// section 12) reads the stage-rate values from global memory as well.  Only the DIAG path reads D / Dinv through here.
struct ParEnv {
    LEO_HD static double g(const double *S, int64_t stride, int64_t e, int f) { return S[(int64_t)(LEO_ND + f) * stride + e]; }
#ifdef LEO_PENV_GLOBAL
    LEO_HD static void load_bus(const LeoParams &, const PAt &) {}
    LEO_HD static double st(const PAt &at, int f) { return g(at.S, at.stride, at.e, f); }
#else
    LEO_HD static void load_bus(const LeoParams &, const PAt &at)
    {
#pragma unroll
        for (int f = PE_INV_MASS; f <= PE_DRAGKA + 2; f++) mst(at.m, M_PE + f, g(at.S, at.stride, at.e, f));
    }
    LEO_HD static double st(const PAt &at, int f) { return mld(at.m, M_PE + f); }
#endif
    LEO_HD static double inv_mass(const LeoParams &, const PAt &at) { return st(at, PE_INV_MASS); }
    LEO_HD static double D(const LeoParams &, const PAt &at, int k) { return st(at, PE_D + k); }
    LEO_HD static double Dinv(const LeoParams &, const PAt &at, int k) { return st(at, PE_DINV + k); }
    LEO_HD static double dragKa(const LeoParams &, const PAt &at, int k) { return st(at, PE_DRAGKA + k); }
    LEO_HD static double rho0(const LeoParams &, const double *S, int64_t s, int64_t e) { return g(S, s, e, PE_RHO0); }
    LEO_HD static double inv_H(const LeoParams &, const double *S, int64_t s, int64_t e) { return g(S, s, e, PE_INV_H); }
    LEO_HD static double panel_coef(const LeoParams &, const double *S, int64_t s, int64_t e) { return g(S, s, e, PE_PANEL); }
    LEO_HD static double sink_power(const LeoParams &, const double *S, int64_t s, int64_t e) { return g(S, s, e, PE_SINK); }
    LEO_HD static double capacity(const LeoParams &, const double *S, int64_t s, int64_t e) { return g(S, s, e, PE_CAP); }
    LEO_HD static double K(const LeoParams &, const double *S, int64_t s, int64_t e) { return g(S, s, e, PE_K); }
    LEO_HD static double Pgain(const LeoParams &, const double *S, int64_t s, int64_t e) { return g(S, s, e, PE_P); }
    LEO_HD static const double *I_fsw(const LeoParams &, const double *S, int64_t s, int64_t e, double *buf)
    { // the same 3x3 product as the batch path (its off-diagonal zeros included): identical arithmetic for a default row
        for (int k = 0; k < 9; k++) buf[k] = 0.0;
        for (int k = 0; k < 3; k++) buf[4 * k] = g(S, s, e, PE_IFSW + k);
        return buf;
    }
    LEO_HD static double hs_min(const LeoParams &, const double *S, int64_t s, int64_t e) { return g(S, s, e, PE_HSMIN); }
    LEO_HD static double dist_mag(const LeoParams &, const double *S, int64_t s, int64_t e) { return g(S, s, e, PE_DIST); }
};

// Pool row of an env at a reset.  BY_INDEX: global env index mod n_rows.  PER_EPISODE: one Philox4x32-10 block keyed like
// the IC stream, (seed, global env, episode), at counter word 0xFFFFFFFF, which the IC sampler (blocks 0, 1, ...) never
// reaches: the IC draws are those of a run without a pool, and neither depends on the sharding.
LEO_HD int64_t pool_row(const LeoPool &pool, uint64_t seed, int64_t global_env, int64_t episode)
{
    if (pool.assign == LEO_POOL_BY_INDEX) return global_env % pool.n_rows;
    uint32_t o[4];
    philox4x32((uint32_t)global_env, (uint32_t)((uint64_t)global_env >> 32), (uint32_t)episode, 0xFFFFFFFFu, (uint32_t)seed,
               (uint32_t)(seed >> 32), o);
    return (int64_t)((((uint64_t)o[1] << 32) | o[0]) % (uint64_t)pool.n_rows);
}
// Copy a derived pool row into the env's parameter block
LEO_HD void pool_assign(const LeoPool &pool, double *S, int64_t stride, int64_t e, int64_t row)
{
    for (int f = 0; f < LEO_NPD; f++) S[(int64_t)(LEO_ND + f) * stride + e] = pool.rows[(int64_t)f * pool.n_rows + row];
}

// Initial-condition pool row of an env at a reset (LEO and opNav).  BY_INDEX: global env index mod n_rows.  PARAM_ROW: the
// env's parameter-pool row of the same reset.  PER_EPISODE: one Philox4x32-10 block keyed like the IC stream, (seed, global
// env, episode), at counter word 0xFFFFFFFE.  No other stream reaches that word: the IC samplers use blocks 0, 1, ... (a few
// dozen at most), the parameter pool 0xFFFFFFFF, and the opNav noise streams (stream << 16 | block) with stream 1 or 2 and
// block < 4 -- those run under the key seed_hi ^ episode, which is the IC key at episode 0, so only the counter word keeps
// them apart, and it does.  The ICs a run samples, its parameter rows and its noise are therefore those of a run without an
// IC pool, and none of them depends on the sharding.
LEO_HD int64_t ic_pool_row(const IcPool &pool, uint64_t seed, int64_t global_env, int64_t episode, int64_t param_row)
{
    if (pool.assign == IC_POOL_BY_INDEX) return global_env % pool.n_rows;
    if (pool.assign == IC_POOL_PARAM_ROW) return param_row;
    uint32_t o[4];
    philox4x32((uint32_t)global_env, (uint32_t)((uint64_t)global_env >> 32), (uint32_t)episode, 0xFFFFFFFEu, (uint32_t)seed,
               (uint32_t)(seed >> 32), o);
    return (int64_t)((((uint64_t)o[1] << 32) | o[0]) % (uint64_t)pool.n_rows);
}

LEO_HD_NOINLINE void sun_latch_to_bus(const LeoParams &P, MBus m, int64_t msg_ns)
{
    SunLatch s = sun_latch(P, msg_ns);
    mst3(m, M_SUNR, s.r); mst3(m, M_SUNV, s.v);
    mst(m, M_ECL, s.hp2); mst(m, M_ECL + 1, s.inv_hp); mst(m, M_ECL + 2, s.c1off);
    mst(m, M_ECL + 3, s.c2off); mst(m, M_ECL + 4, s.tan1); mst(m, M_ECL + 5, s.tan2);
}

// Earth orientation at a SPICE message time (SURVEY 8(f)-4; spice_interface with computeOrient): J2000 -> planet-fixed
// DCM P = R3(W) R1(pi/2 - DEC) R3(pi/2 + RA) and its time derivative (pxform_c / sxform_c).  Angles from the
// orientation table when one is loaded, else the IAU rotation model of the SPICE text kernel pck00010.tpc
// (BODY399_POLE_RA = 0 - 0.641 T, POLE_DEC = 90 - 0.557 T, PM = 190.147 + 360.9856235 d).
LEO_HD_NOINLINE void pfix_latch_to_bus(const LeoParams &P, MBus m, int64_t msg_ns)
{
    const double D2R = 3.14159265358979323846 / 180.0, HPI = 0.5 * 3.14159265358979323846;
    const double t = ns2sec(msg_ns);
    V3 ang, rate;
    if (P.eph_orient.nseg > 0) {
        cheb_eval(P.eph_orient, t, ang, rate);
    } else {
        const double d = P.epoch_days + t / 86400.0, T = d / 36525.0;
        ang = mk((0.0 - 0.641 * T) * D2R, (90.0 - 0.557 * T) * D2R, (190.147 + 360.9856235 * d) * D2R);
        rate = mk(-0.641 / 36525.0 / 86400.0 * D2R, -0.557 / 36525.0 / 86400.0 * D2R, 360.9856235 / 86400.0 * D2R);
    }
    const double th = HPI - ang.y, ph = HPI + ang.x, thd = -rate.y, phd = rate.x, Wd = rate.z;
    const double cw = cos(ang.z), sw = sin(ang.z), ct = cos(th), st = sin(th), cp = cos(ph), sp = sin(ph);
    // A = R1(th) R3(ph) and its derivative
    const V3 A0 = mk(cp, sp, 0.), A1 = mk(-ct * sp, ct * cp, st), A2 = mk(st * sp, -st * cp, ct);
    const V3 dA0 = mk(-sp * phd, cp * phd, 0.);
    const V3 dA1 = mk(st * sp * thd - ct * cp * phd, -st * cp * thd - ct * sp * phd, ct * thd);
    const V3 dA2 = mk(ct * sp * thd + st * cp * phd, -ct * cp * thd + st * sp * phd, -st * thd);
    const V3 P0 = A0 * cw + A1 * sw, P1 = A1 * cw - A0 * sw;
    mst3(m, M_PFIX, P0); mst3(m, M_PFIX + 3, P1); mst3(m, M_PFIX + 6, A2);
    mst3(m, M_PFIXD, P1 * Wd + dA0 * cw + dA1 * sw);
    mst3(m, M_PFIXD + 3, dA1 * cw - dA0 * sw - P0 * Wd);
    mst3(m, M_PFIXD + 6, dA2);
}

// One flight-software pass at time now_ns (the priority 100/50 tasks run before DynTask at equal times).
// nav = state written by the previous dynamics tick (zeros before tick 0: messages never written).
// Out of line: it runs once per ticks_per_fsw dynamics ticks and must not bloat the hot tick loop.
// Returns the state of the desat chain: 0 did not run; 1 full pass; 3 full pass that left the chain quiet (to be
// confirmed by the thruster latch); 4 quiet pass (all on-times and commands are zero and stay zero: only
// thrMomentumDumping's rest counter and time tag advance).
template <int NRW, class PA = ParBatch>
LEO_HD_NOINLINE int fsw_pass(const LeoParams &P, double *S, int64_t *I, int64_t stride, int64_t e, MBus m, int mask,
                             int64_t n, int64_t now_ns, Dyn x, const double (&W)[NRW], int64_t sun_ns, int desat_quiet)
{
    V3 nr = x.r, nv = x.v, ns = x.s, nw = x.w;
    double ws[NRW];
#pragma unroll
    for (int i = 0; i < NRW; i++) ws[i] = W[i];
    if (n == 0) {
        nr = nv = ns = nw = mk(0., 0., 0.);
#pragma unroll
        for (int i = 0; i < NRW; i++) ws[i] = 0.0;
    }
    AttRef ref;
    if (mask & LEO_TASK_NADIR) {                     // hillPoint
        V3 cr = mk(0., 0., 0.), cv = mk(0., 0., 0.);
        // SURVEY Q3: r_BdyZero_N aliases {J2000Current, 0, 0} of the Sun message in force
        if (P.hill_cel_pun) cr.x = P.epoch_days * 86400.0 + ns2sec(sun_ns);
        ref = hill_point(nr, nv, cr, cv);
    } else if (mask & LEO_TASK_SUN) {                // inertial3D
        ref.sigma_RN = arr(P.sigma_R0N);
        ref.omega_RN_N = mk(0., 0., 0.); ref.domega_RN_N = mk(0., 0., 0.);
    } else {                                         // no guidance task enabled: the last message stays in force
        ref.sigma_RN = mld3(m, M_REF); ref.omega_RN_N = mld3(m, M_REF + 3); ref.domega_RN_N = mld3(m, M_REF + 6);
    }
    if (mask & (LEO_TASK_SUN | LEO_TASK_NADIR)) {
        mst3(m, M_REF, ref.sigma_RN); mst3(m, M_REF + 3, ref.omega_RN_N); mst3(m, M_REF + 6, ref.domega_RN_N);
    }
    int desat_ran = 0;
    if (mask & LEO_TASK_DESAT) {
        if (desat_quiet) {
            const int64_t cnt = I[(int64_t)I_DUMPCNT * stride + e];
            I[(int64_t)I_DUMPCNT * stride + e] = cnt <= 0 ? (int64_t)P.maxCounterValue : cnt - 1;
            I[(int64_t)I_DUMPPRIOR * stride + e] = now_ns;
            desat_ran = 4;
        } else {
            desat_ran = 1 | (fsw_desat<NRW, PA>(P, S, I, stride, e, now_ns, ws) << 1);
        }
    }
    if (mask & LEO_TASK_MRP) {
        // quirk Q1: MRP_Feedback runs BEFORE attTrackingError -> uses last pass's att_guidance
        AttGuid g;
        g.sigma_BR = mld3(m, M_GUID); g.omega_BR_B = mld3(m, M_GUID + 3);
        g.omega_RN_B = mld3(m, M_GUID + 6); g.domega_RN_B = mld3(m, M_GUID + 9);
        V3 Lr = mrp_feedback<PA>(P, g, S, stride, e);
        mst3(m, M_LR, Lr);
        g = att_tracking_error(ns, nw, ref);
        mst3(m, M_GUID, g.sigma_BR); mst3(m, M_GUID + 3, g.omega_BR_B);
        mst3(m, M_GUID + 6, g.omega_RN_B); mst3(m, M_GUID + 9, g.domega_RN_B);
        // rwMotorTorque: us = Umap (-Lr)
        V3 mLr = -Lr;
#pragma unroll
        for (int i = 0; i < NRW; i++) mst(m, M_RWCMD + i, P.Umap[i][0] * mLr.x + P.Umap[i][1] * mLr.y + P.Umap[i][2] * mLr.z);
    }
    return desat_ran;
}

LEO_HD V3 add_cross(V3 p, V3 u, V3 v)     // p + u x v, six fused operations
{
    return mk(fmad(u.y, v.z, fmad(-u.z, v.y, p.x)), fmad(u.z, v.x, fmad(-u.x, v.z, p.y)), fmad(u.x, v.y, fmad(-u.y, v.x, p.z)));
}
LEO_HD V3 sub_cross(V3 p, V3 u, V3 v)     // p - u x v
{
    return mk(fmad(-u.y, v.z, fmad(u.z, v.y, p.x)), fmad(-u.z, v.x, fmad(u.x, v.z, p.y)), fmad(-u.x, v.y, fmad(u.y, v.x, p.z)));
}

// Sun third-body acceleration of the gravityEffector (direct + indirect term) at spacecraft position r, Sun at rs
LEO_HD V3 sun_accel(const LeoParams &P, V3 rs, V3 r)
{
    V3 d = r - rs;
    double is = rsq(dot(rs, rs)), id = rsq(dot(d, d));
    return rs * (-P.mu_sun * (is * is * is)) + d * (-P.mu_sun * (id * id * id));
}

// The Sun third-body acceleration HELD over a window of w dynamics ticks (one flight-software period): evaluated once, at the
// window's mid time and the position predicted for it from the state at the window's start (time offset dt0 from the Sun
// message in force; the first tick of the window has length h_first, the others dyn_s).  The term is a tide of 2.8e-7 m/s^2
// that turns with the orbit (rate of change ~5e-10 m/s^3): held at the midpoint of a 1 s window the first-order error
// cancels over the window and the second-order one leaves ~5e-14 m/s of velocity per window.  MEASURED against the oracle,
// which evaluates the Sun at every RK stage (tests/test_gpu_round2.py, long-horizon test, up to 61 intervals = 3 h without
// re-synchronisation): position / velocity 9.6e-12 relative (2.2e-12 with the term evaluated every tick; a second-order
// position prediction changes nothing), growing quadratically -- 2e-10 after a full 270-interval episode; per decision
// interval < 1e-13.  Steps in which a thruster may switch, and the step whose Sun clock wraps, evaluate the Sun at every
// stage (rk4_general).  DESIGN.md section 9b, D14.
LEO_HD V3 sun_window(const LeoParams &P, MBus m, const Dyn &x, double dt0, double h_first, int w, double dyn_s)
{
    const double half = 0.5 * (h_first + (double)(w - 1) * dyn_s);
    return sun_accel(P, mld3(m, M_SUNR) + mld3(m, M_SUNV) * (dt0 + half), x.r + x.v * half);
}

// What one RK4 step needs besides the parameter block and the integrated state.
struct StageIn {
    V3 Lc;                         // held body torque: extForceTorque (+ thrusters) - wheel motor torque on the hub
    V3 gsun;                       // Sun third-body acceleration
    V3 HB, tau_u;                  // wheel momentum invariant at the start of the step and motor torque sum_i g_i u_i (see Dyn)
    double rho, h;
    double dtp;                    // planet-fixed gravity only: time since the SPICE message that carries the orientation
};

// One evaluation of SpacecraftPlus::equationsOfMotion for the scenario's effector set at stage time t0 + ct.
//   DIAG   fast path of the reference configuration: diagonal hub inertia, three wheels along the body axes
//          (AP:20-37) and drag facets located on their own normal axis (SIM:274-281) -- the same arithmetic
//          with the structural zeros dropped
template <int J2, bool DIAG, class PA = ParBatch>
LEO_HD void eom(const LeoParams &P, const Dyn &x, Dyn &k, const StageIn &a, double ct, bool thr_on, MBus m,
                const double *S = nullptr, int64_t stride = 0, int64_t e = 0)
{
    const PAt at = {m, S, stride, e};
    // gravity: central point mass (+J2) + Sun third body (gravityEffector)
    V3 g;
    {
        double ir = rsq(dot(x.r, x.r));
        double ir3 = ir * ir * ir;
        g = a.gsun + x.r * (-P.mu_c * ir3);
        if (J2 == 2) {
            // degree-2 field in the planet-fixed frame (GravBodyData::computeGravityInertial with spherical harmonics):
            // dcm_PfixN = J20002Pfix + J20002Pfix_dot dt, g_N += dcm^T grad U_2(dcm r), with the closed-form gradient of
            // U_2 = (r^T M r) / |r|^5:  grad U_2 = 2 M r / |r|^5 - 5 (r^T M r) r / |r|^7   (gm2 = mu Req^2 M)
            const V3 D0 = mld3(m, M_PFIX) + mld3(m, M_PFIXD) * a.dtp;
            const V3 D1 = mld3(m, M_PFIX + 3) + mld3(m, M_PFIXD + 3) * a.dtp;
            const V3 D2 = mld3(m, M_PFIX + 6) + mld3(m, M_PFIXD + 6) * a.dtp;
            const V3 rp = mk(dot(D0, x.r), dot(D1, x.r), dot(D2, x.r));
            const double ip = rsq(dot(rp, rp)), ip2 = ip * ip, ip5 = ip2 * ip2 * ip;
            const V3 Mr = mk(P.gm2[0] * rp.x + P.gm2[3] * rp.y + P.gm2[4] * rp.z,
                             P.gm2[3] * rp.x + P.gm2[1] * rp.y + P.gm2[5] * rp.z,
                             P.gm2[4] * rp.x + P.gm2[5] * rp.y + P.gm2[2] * rp.z);
            const double q5 = -5. * dot(rp, Mr) * ip5 * ip2;
            const V3 gp = Mr * (2. * ip5) + rp * q5;
            g = g + D0 * gp.x + D1 * gp.y + D2 * gp.z;
        } else if (J2) {
            double ir2 = ir * ir, z2 = 5. * x.r.z * x.r.z * ir2, kk = -P.j2k * ir3 * ir2;
            g = g + mk(kk * x.r.x * (1. - z2), kk * x.r.y * (1. - z2), kk * x.r.z * (3. - z2));
        }
    }
    // facet drag with axis-aligned facets: F_B = -rho * S' * v_B (parallel to v_B, so [NB] F_B = -rho S' v_N),
    // L_B = -rho * (M' x v_B).  A facet contributes when its normal has a positive component along v_B:
    // K(sign v) |v| = Ka |v| + Kd v with Ka/Kd the half sum / half difference of the +/- facets.
    MrpRot R = mrp_rot(x.s);
    V3 vB = rot_BN(R, x.s, x.v);
    V3 Mp;
    double Sp;
    {
        double ax = fabs(vB.x), ay = fabs(vB.y), az = fabs(vB.z);
        // DIAG also means equal + / - facet areas on every axis (SIM:274-281: 0.06 / 0.06, 2.02 / 2.02, 0.03 / 0.03): Kd = 0
        Sp = PA::dragKa(P, at, 0) * ax + PA::dragKa(P, at, 1) * ay + PA::dragKa(P, at, 2) * az;
        if (!DIAG) Sp += P.dragKd[0] * vB.x + P.dragKd[1] * vB.y + P.dragKd[2] * vB.z;
        if (DIAG) {
            Mp = mk(P.dragMa[0][0] * ax + P.dragMd[0][0] * vB.x, P.dragMa[1][1] * ay + P.dragMd[1][1] * vB.y,
                    P.dragMa[2][2] * az + P.dragMd[2][2] * vB.z);
        } else {
            Mp = arr(P.dragMa[0]) * ax + arr(P.dragMa[1]) * ay + arr(P.dragMa[2]) * az
               + arr(P.dragMd[0]) * vB.x + arr(P.dragMd[1]) * vB.y + arr(P.dragMd[2]) * vB.z;
        }
    }
    const double mrho = -a.rho;
    k.v = g + x.v * (mrho * Sp);                    // dragKa/Kd carry the 1/mass
    if (thr_on) k.v = k.v + rot_NB(R, x.s, mld3(m, M_FM));
    k.r = x.v;
    // rotational EOM with balanced wheels (back-substitution, D constant; wheel momentum from the invariant):
    //   D wdot = -w x (D w + HB + ct tau_u) - sum g u + L
    V3 rot = add_cross(a.Lc, Mp * mrho, vB);
    const V3 hw = a.HB + a.tau_u * ct;
    if (DIAG) {
        V3 h = mk(fmad(PA::D(P, at, 0), x.w.x, hw.x), fmad(PA::D(P, at, 1), x.w.y, hw.y), fmad(PA::D(P, at, 2), x.w.z, hw.z));
        rot = sub_cross(rot, x.w, h);
        k.w = mk(rot.x * PA::Dinv(P, at, 0), rot.y * PA::Dinv(P, at, 1), rot.z * PA::Dinv(P, at, 2));
    } else {
        V3 h = mv9(P.D, x.w) + hw;
        rot = sub_cross(rot, x.w, h);
        k.w = mv9(P.Dinv, rot);
    }
    { // sigma_dot = 1/4 [B(sigma)] omega
        double sw = dot(x.s, x.w);
        k.s = x.w * (0.25 * R.oms2) + cross(x.s, x.w) * 0.5 + x.s * (0.5 * sw);
    }
}

// Classical RK4 over one dynamics tick.  The four stages run as ONE rolled loop whose body is a single block of
// FP64 arithmetic small enough to stay resident in the SM sub-partition's L0 instruction cache (a fully
// unrolled step streams ~20 KB of code per tick and the kernel becomes instruction-fetch bound: ncu
// stall_no_instruction, profiles/).  No register copies cross the back edge: the stage input is rebuilt from
// the tick-start state and the previous slope (xs = x + c k, with k = 0 before the first stage), and the
// weighted slopes are summed separately and added once.
// The Sun's third-body acceleration is held (evaluated by the caller once per flight-software period at the period's mid
// time and predicted mid position, see sun_window()); the thrust is constant over the step.  Steps in which a thruster may
// switch, and the step whose Sun clock wraps, go through rk4_general().
template <int J2, bool DIAG, class PA = ParBatch>
LEO_HD Dyn rk4_step(const LeoParams &P, const Dyn &x, const StageIn &a, bool thr_on, MBus m,
                    const double *S = nullptr, int64_t stride = 0, int64_t e = 0)
{
    const double h = a.h, hh = 0.5 * h, h6 = h * (1.0 / 6.0), h3 = h * (1.0 / 3.0);
    Dyn k, acc;
    k.r = k.v = k.s = k.w = acc.r = acc.v = acc.s = acc.w = mk(0., 0., 0.);
    double c = 0.;
#if LEO_UNROLL_STAGES == 2
#pragma unroll 2
#elif LEO_UNROLL_STAGES
#pragma unroll
#else
#pragma unroll 1
#endif
    for (int st = 0; st < 4; st++) {
        Dyn xs;
        xs.r = x.r + k.r * c; xs.v = x.v + k.v * c; xs.s = x.s + k.s * c; xs.w = x.w + k.w * c;
        eom<J2, DIAG, PA>(P, xs, k, a, c, thr_on, m, S, stride, e);
        const double wo = (st == 0 || st == 3) ? h6 : h3;
        acc.r = acc.r + k.r * wo; acc.v = acc.v + k.v * wo; acc.s = acc.s + k.s * wo; acc.w = acc.w + k.w * wo;
        c = (st == 2) ? h : hh;
    }
    Dyn xo;
    xo.r = x.r + acc.r; xo.v = x.v + acc.v; xo.s = x.s + acc.s; xo.w = x.w + acc.w;
    return xo;
}

// The same RK4 step with the Sun evaluated at every stage time and position, and with
// thrusterDynamicEffector::computeForceTorque evaluated at every stage time: used for the steps in which a
// thruster may start or stop burning (a new on-time command was just latched, or a commanded burn expires
// within the step) and for the step whose Sun clock wraps (quirk Q18: the stage clocks are not on a line,
// stage 4 may land exactly on the message time while stages 1-3 are 2^64 ns away).  Out of line; classical
// accumulation order.
struct SunDt { double d0, dm, d1; };
struct ThrEventOut { Dyn x; int factor, active; };
template <int J2, bool DIAG, class PA = ParBatch>
LEO_HD_NOINLINE ThrEventOut rk4_general(const LeoParams &P, const double *S, int64_t stride, int64_t e, MBus m, Dyn x,
                                        StageIn a, SunDt dts, double tBefore, double tauPrev, int thr_factor, int thr_active)
{
    const double h = a.h, hh = 0.5 * h, h6 = h * (1.0 / 6.0), h3 = h * (1.0 / 3.0);
    const V3 sun_r = mld3(m, M_SUNR), sun_v = mld3(m, M_SUNV), L_ext = mld3(m, M_LEXT);
    Dyn xs = x, xo = x, k;
    ThrCmd tc = {};
    if (thr_active) tc = thr_cmd_load(S, stride, e);
#pragma unroll 1
    for (int st = 0; st < 4; st++) {
        const double dt = (st == 0) ? dts.d0 : (st == 3 ? dts.d1 : dts.dm);
        const double ct = (st == 0) ? 0.0 : (st == 3 ? h : hh);
        a.gsun = sun_accel(P, sun_r + sun_v * dt, xs.r);
        a.dtp = dt;
        V3 Fm = mk(0., 0., 0.), Lx = L_ext;
        const bool thr_on = thr_active != 0;
        if (thr_on) {
            const double tau = t_add(tBefore, (st == 0) ? 0.0 : (st == 3 ? h : t_mul(h, 0.5)));
            ThrOut to = thr_stage(P, tc, tau, t_sub(tau, tauPrev), thr_factor);
            thr_factor = to.factor; thr_active = to.active;
            Fm = to.F * PA::inv_mass(P, PAt{m, S, stride, e}); Lx = Lx + to.L;
            tauPrev = tau;
        }
        a.Lc = Lx - a.tau_u;
        mst3(m, M_FM, Fm);
        eom<J2, DIAG, PA>(P, xs, k, a, ct, thr_on, m, S, stride, e);
        const double wo = (st == 0 || st == 3) ? h6 : h3;
        const double cn = (st == 2) ? h : hh;
        xo.r = xo.r + k.r * wo; xo.v = xo.v + k.v * wo; xo.s = xo.s + k.s * wo; xo.w = xo.w + k.w * wo;
        if (st < 3) { xs.r = x.r + k.r * cn; xs.v = x.v + k.v * cn; xs.s = x.s + k.s * cn; xs.w = x.w + k.w * cn; }
    }
    ThrEventOut o;
    o.x = xo; o.factor = thr_factor; o.active = thr_active;
    return o;
}

// Force / torque of the thrusters that are burning (bit mask `factor`) and the earliest time at which one of
// them stops: until then computeForceTorque returns the same sums at every stage (expiry is monotone in
// time and the commanded on-times only change at the next command latch).  Publishes the held thrust on the
// bus and rebuilds the held body torque.
struct ThrRefresh { V3 Lc, L_thr; double t_next; };
template <class PA = ParBatch>
LEO_HD_NOINLINE ThrRefresh thr_refresh(const LeoParams &P, const double *S, int64_t stride, int64_t e, MBus m, int factor, V3 tau_u)
{
    ThrRefresh o;
    V3 F = mk(0., 0., 0.);
    o.L_thr = mk(0., 0., 0.); o.t_next = 1e300;
    double start = S[(int64_t)F_THRSTART * stride + e];
    for (int k = 0; k < LEO_NTHR; k++) {
        if (!((factor >> k) & 1)) continue;
        V3 f = arr(P.thr_dir[k]) * (P.thr_Fmax * 1.0);
        F = f + F;
        o.L_thr = cross(arr(P.thr_loc[k]), f) + o.L_thr;
        double t_off = t_add(S[(int64_t)(F_THRON + k) * stride + e], start);
        if (t_off < o.t_next) o.t_next = t_off;
    }
    mst3(m, M_FM, F * PA::inv_mass(P, PAt{m, S, stride, e}));
    o.Lc = (mld3(m, M_LEXT) + o.L_thr) - tau_u;
    return o;
}

// Stage clocks of the step whose Sun message is newer than the integration time (quirk Q18): Basilisk's
// unsigned (systemClock - WriteClockNanos) wraps.  Replicated (last tick of every decision interval).
LEO_HD_NOINLINE SunDt sun_dt_wrapped(double prev_ns_d, double sun_ns_d, double tBefore, double prevTime, double h)
{
    SunDt o;
    uint64_t sun_ns = (uint64_t)sun_ns_d;
    uint64_t s0 = (uint64_t)t_add(prev_ns_d, t_div(t_sub(tBefore, prevTime), 1e-9));
    uint64_t sm = (uint64_t)t_add(prev_ns_d, t_div(t_sub(t_add(tBefore, t_mul(h, 0.5)), prevTime), 1e-9));
    uint64_t s1 = (uint64_t)t_add(prev_ns_d, t_div(t_sub(t_add(tBefore, h), prevTime), 1e-9));
    o.d0 = t_mul((double)(s0 - sun_ns), 1e-9);
    o.dm = t_mul((double)(sm - sun_ns), 1e-9);
    o.d1 = t_mul((double)(s1 - sun_ns), 1e-9);
    return o;
}

// The rare events after a dynamics tick, in task order:
//  * reactionWheelStateEffector.UpdateState: latch the motor torque command (torque and speed saturation) when
//    the command is new or a speed limit is in play;
//  * thrusterDynamicEffector.UpdateState: only a NEW on-time message re-configures the thrusters.
// Rebuilds the held body torque.  Returns the new thr_active (or -1 when no thruster message arrived).
template <int NRW>
struct PostOut { double uJ[NRW]; V3 Lc, tau_u; int thr_active, quiet; };
// reactionWheelStateEffector.UpdateState: torque saturation, dead band and speed limit of every wheel; rebuilds the held torque
template <int NRW>
LEO_HD void wheel_latch(const LeoParams &P, MBus m, const double (&W)[NRW], V3 L_thr, double (&uJ)[NRW], V3 &Lc, V3 &tau_u_out)
{
    V3 tau_u = mk(0., 0., 0.);
#pragma unroll
    for (int i = 0; i < NRW; i++) {
        double uc = mld(m, M_RWCMD + i);
        if (P.u_max[i] > 0.) { if (uc > P.u_max[i]) uc = P.u_max[i]; else if (uc < -P.u_max[i]) uc = -P.u_max[i]; }
        if (fabs(uc) < P.u_min[i]) uc = 0.0;
        if (fabs(W[i]) >= P.Om_max[i] && P.Om_max[i] > 0.0 && W[i] * uc >= 0.0) uc = 0.0;
        mst(m, M_U + i, uc);
        uJ[i] = uc * P.invJs[i];
        tau_u = tau_u + arr(P.gs[i]) * uc;
    }
    tau_u_out = tau_u;
    Lc = (mld3(m, M_LEXT) + L_thr) - tau_u;
}
template <int NRW>
LEO_HD_NOINLINE PostOut<NRW> post_tick_events(const LeoParams &P, double *S, int64_t *I, int64_t stride, int64_t e, MBus m,
                                              const double (&W)[NRW], V3 L_thr, int desat_ran, int64_t now_ns, int thr_factor)
{
    PostOut<NRW> o;
    wheel_latch<NRW>(P, m, W, L_thr, o.uJ, o.Lc, o.tau_u);
    o.thr_active = -1; o.quiet = 0;
    if (desat_ran & 1) {
        o.thr_active = thr_latch(P, S, I, stride, e, now_ns, thr_factor);
        o.quiet = (desat_ran & 2) && o.thr_active == 0;          // nothing commanded, nothing burning
    } else if (desat_ran & 4) {                                 // quiet: the latch would rewrite zeros; keep the time tag
        S[(int64_t)F_THRSTART * stride + e] = t_mul((double)now_ns, 1.0E-9);
        o.quiet = 1;
    }
    return o;
}

// Margin [s] by which a burning thruster's expiry must lie beyond the end of a step for the step to take the
// constant-thrust path (the exact test has a tolerance of 1e-9 * stage spacing around the expiry time).
#define LEO_THR_MARGIN 1e-6

// Wheel speeds from the momentum invariant (see Dyn): Omega_i = C_i - g_i.omega
template <int NRW, bool DIAG>
LEO_HD void wheel_speeds(const LeoParams &P, V3 HB, const double (&C)[NRW], V3 w, double (&W)[NRW])
{
    if (DIAG) {
        W[0] = fmad(HB.x, P.invJs[0], -w.x); W[1] = fmad(HB.y, P.invJs[1], -w.y); W[2] = fmad(HB.z, P.invJs[2], -w.z);
    } else {
#pragma unroll
        for (int i = 0; i < NRW; i++) W[i] = C[i] - dot(arr(P.gs[i]), w);
    }
}

#if defined(__CUDACC__)
// 64-bit literals of the per-tick code live in constant memory: an FP64 instruction takes a constant-bank operand for free,
// whereas a literal that does not fit the 32-bit immediate form costs two uniform-register moves (two issue slots) per use.
__constant__ double LEO_K[16] = {
    1.4426950408889634, 6755399441055744.0, -6.93147180369123816490e-01, -1.90821492927058770002e-10,    // exp: log2 e, 2^52 + 2^51, -ln2 hi / lo
    1. / 6., 1. / 24., 1. / 120., 1. / 720., 1. / 5040., 1. / 40320., 1. / 362880., 1. / 3628800., 1. / 39916800.,
    1. / 479001600., 1. / 6227020800.,                                                                   // exp: Taylor 1/3! .. 1/13!
    1e-9};                                                                                               // NANO2SEC
#endif
#if defined(__CUDA_ARCH__)
#define LEO_NANO2SEC LEO_K[15]
#else
#define LEO_NANO2SEC 1e-9
#endif
// exp(x) for |x| <= 700 without special-operand handling (the atmosphere's argument): Cody-Waite reduction by
// ln 2, degree-13 Taylor polynomial on |r| <= ln2/2 in Estrin form (truncation 4e-18), exponent patched in.
LEO_HD double exp_bounded(double x)
{
#ifdef __CUDA_ARCH__
    x = fmin(fmax(x, -700.0), 700.0);
    const double t = fma(x, LEO_K[0], LEO_K[1]);
    const int kk = __double2loint(t);
    const double kd = t - LEO_K[1];
    double r = fma(kd, LEO_K[2], x);
    r = fma(kd, LEO_K[3], r);
    const double r2 = r * r, r4 = r2 * r2, r8 = r4 * r4;
    const double a0 = r + 1.0, a1 = fma(r, LEO_K[4], 0.5), a2 = fma(r, LEO_K[6], LEO_K[5]), a3 = fma(r, LEO_K[8], LEO_K[7]);
    const double a4 = fma(r, LEO_K[10], LEO_K[9]), a5 = fma(r, LEO_K[12], LEO_K[11]);
    const double a6 = fma(r, LEO_K[14], LEO_K[13]);
    const double b0 = fma(a1, r2, a0), b1 = fma(a3, r2, a2), b2 = fma(a5, r2, a4);
    const double d0 = fma(b1, r4, b0), d1 = fma(a6, r4, b2);
    const double p = fma(d1, r8, d0);
    return __hiloint2double(__double2hiint(p) + (kk << 20), __double2loint(p));
#else
    return exp(x);
#endif
}

}  // namespace leo
#include "leo_f32.cuh"      // mixed-precision tick (BASELINE config 5); needs everything above
namespace leo {

// F32 = false: the FP64 kernel (the reference's arithmetic; every parity claim).  F32 = true: mixed precision, see leo_f32.cuh.
// PA = ParEnv: the env's own spacecraft parameters (bskenv_set_param_pool; DIAG, FP64 only).
template <int NRW, int J2, bool DIAG, bool F32 = false, class PA = ParBatch>
// `chunk` / `n_chunks`: the decision interval may be executed as n_chunks consecutive calls of ticks/n_chunks dynamics
// ticks each (chunk 0 applies the mode switch, the last chunk samples the observation and does the gym bookkeeping); the
// persistent state carries everything across a chunk boundary exactly as it does across a decision boundary, and the
// Sun / orientation latch keeps the time of the interval's SPICE message.  The kernel uses this to cut one launch into
// finer work items (bskenv.cu: smaller tail); leo_host::step_chunks() fixes the split as a function of the rates only.
LEO_HD void leo_step_env(const LeoParams &P, double *__restrict__ S, int64_t *__restrict__ I, int64_t stride, int64_t e,
                         MBus m, int action, StepOut &out, const LeoParamsF &PF = LeoParamsF(), int chunk = 0, int n_chunks = 1)
{
#define SD(f) S[(int64_t)(f) * stride + e]
#define SI(f) I[(int64_t)(f) * stride + e]
    // ---------------- load ----------------
    Dyn x;
    StageIn a;
    x.r = mk(SD(F_R), SD(F_R + 1), SD(F_R + 2));
    x.v = mk(SD(F_V), SD(F_V + 1), SD(F_V + 2));
    x.s = mk(SD(F_SIG), SD(F_SIG + 1), SD(F_SIG + 2));
    x.w = mk(SD(F_OMG), SD(F_OMG + 1), SD(F_OMG + 2));
    PA::load_bus(P, PAt{m, S, stride, e});
    double C[NRW], uJ[NRW];                                     // wheel invariants / motor torque over Js (general path)
    a.tau_u = mk(0., 0., 0.); a.HB = mk(0., 0., 0.);
#pragma unroll
    for (int i = 0; i < NRW; i++) {
        const double u = SD(F_UCUR + i);
        mst(m, M_U + i, u);
        uJ[i] = u * P.invJs[i];
        C[i] = SD(F_WHL + i) + dot(arr(P.gs[i]), x.w);
        a.tau_u = a.tau_u + arr(P.gs[i]) * u;
        a.HB = a.HB + arr(P.gs[i]) * (P.Js[i] * C[i]);
    }
    for (int f = 0; f < LEO_M_MIRROR; f++) mst(m, f, SD(F_GUID + f));
    a.rho = SD(F_RHO);
    {
        const V3 L_ext = mk(SD(F_LDIST), SD(F_LDIST + 1), SD(F_LDIST + 2));
        mst3(m, M_LEXT, L_ext); mst3(m, M_FM, mk(0., 0., 0.));
        a.Lc = L_ext - a.tau_u;
    }
    mst3(m, M_LTHR, mk(0., 0., 0.));                            // held thruster torque (zero outside burns)
    const int64_t tick = SI(I_TICK);
    int mask = (int)SI(I_MASK);
    int thr_factor = (int)SI(I_THRFACTOR), thr_active = (int)SI(I_THRACTIVE), rw_sat = (int)SI(I_RWSAT);
    int nswitch = 0;

    // ---------------- mode switch (SIM:543-588); modeRequest = str(action) ----------------
    if (chunk > 0) {}                                          // the mode was switched by chunk 0 (mask is persistent)
    else if (action == 0) mask = LEO_TASK_NADIR | LEO_TASK_MRP;
    else if (action == 1) mask = LEO_TASK_SUN | LEO_TASK_MRP;
    else if (action == 2) {
        mask = LEO_TASK_SUN | LEO_TASK_MRP | LEO_TASK_DESAT;
        SI(I_INITREQ) = 1;                                   // thrDesatControlWrap.Reset (SIM:580)
        SI(I_DUMPPRIOR) = 0; SI(I_DUMPCNT) = 0; SI(I_LASTDH) = 0;   // thrDumpWrap.Reset (SIM:581)
        for (int k = 0; k < LEO_NTHR; k++) SD(F_THRREM + k) = 0.0;
    }
    // thrusters: the burning set is re-derived by an exact step before the constant-thrust path is trusted
    mst(m, M_TNEXT, -1.0);

    // ---------------- clock: all tick times are integers below 2^53 ns, held exactly in doubles ----------------
    const bool first = tick < 0;                               // tick 0 (t = 0, h = 0) only runs right after a reset
    const int tpf = P.ticks_per_fsw;
    const int ticks_step = tpf * P.fsw_per_step;               // dynamics ticks of a decision interval
    const int ticks = ticks_step / n_chunks;                   // ... of this call
    const int64_t n_base = (first ? 0 : tick) + 1;             // loop index j executes tick n = n_base + j
    const int64_t n_step0 = ((n_base - 1) / ticks_step) * ticks_step;   // tick at which this decision interval started
    const int64_t n_end = n_step0 + ticks_step;                // last tick of the interval, inclusive (ConfigureStopTime is inclusive)
    const double dyn_d = (double)P.dyn_ns;
    double sun_d = (double)(n_step0 * P.dyn_ns);               // write time of the Sun message in force
    sun_latch_to_bus(P, m, n_step0 * P.dyn_ns);
    if (J2 == 2) pfix_latch_to_bus(P, m, n_step0 * P.dyn_ns);
    a.dtp = 0.;
    // FP32 shadows of the Sun latch and its eclipse constants (mixed-precision variant only)
    V3f sunr_f = mkf(0.f, 0.f, 0.f), sunv_f = mkf(0.f, 0.f, 0.f);
    float ecf[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (F32) {
        sunr_f = tof(mld3(m, M_SUNR)); sunv_f = tof(mld3(m, M_SUNV));
#pragma unroll
        for (int q = 0; q < 6; q++) ecf[q] = (float)mld(m, M_ECL + q);
    }
    // ---------------- the tick loop ----------------
    // Layout for latency: a tick is [flight software, every ticks_per_fsw-th tick, out of line] -> [RK4: one rolled loop of four
    // stages] -> ONE straight-line block with everything else that runs every tick -- wheel invariant, MRP switch (as a
    // select), |r|, atmosphere, wheel-limit flags, eclipse cone tests, panel geometry, and the clock and Sun third-body
    // term of the NEXT tick -- -> [rare, out of line: command latches; penumbra] -> battery.  The independent dependency
    // chains of the block (rsqrt / exp / rcp seeds, cone tests, rotations) are interleaved by the instruction scheduler,
    // which cannot move code across the branches that used to separate them; a single resident warp (small batches)
    // otherwise waits out every chain in turn.  Battery charge and shadow factor live in registers.
    const int j0 = first ? -1 : 0;                             // tick 0 (t = 0, h = 0) only runs right after a reset
    int phase = (int)((n_base + j0) % tpf);                    // (n mod ticks_per_fsw) of the tick about to run
    double now_d = (double)((n_base + j0) * P.dyn_ns);         // exact: n * dyn_ns
    int desat_ran = 0, desat_quiet = 0;                        // the chain's quiet state is re-established once per launch
    double charge = SD(F_E), shadow = SD(F_SHADOW);
    // clock of the first tick: CurrentSimNanos * NANO2SEC of this and of the previous tick (tick 0 integrates over an empty
    // interval); for the later ticks prevTime is the previous newTime
    double newTime = t_mul(now_d, LEO_NANO2SEC);
    double prevTime = j0 < 0 ? 0.0 : t_mul(now_d - dyn_d, 1e-9);
    double h = t_sub(newTime, prevTime);
    // Sun at the step's mid time: dt = (systemClock - WriteClockNanos) * 1e-9 at the second/third stage
    double dtsm = t_mul((j0 < 0 ? 0.0 : now_d - dyn_d) - sun_d, LEO_NANO2SEC) + 0.5 * h;
    // Sun third body: held per flight-software period (sun_window); here for the ticks up to the next pass
    const double dyn_s = t_mul(dyn_d, LEO_NANO2SEC);
    if (!F32) a.gsun = sun_window(P, m, x, dtsm - 0.5 * h, h, tpf - phase, dyn_s);

#pragma unroll 1
    for (int j = j0; j < ticks; j++) {
        bool wrapped = false;
        // ================= flight software every ticks_per_fsw-th tick =================
        if (LEO_RARE(phase == 0)) {
            const int64_t n = n_base + j;
            double W[NRW];
            wheel_speeds<NRW, DIAG>(P, a.HB, C, x.w, W);
#ifndef LEO_EXP_NOFSW       // (LEO_EXP_*: measurement switches -- compile a block out to read its cost off the clock, DESIGN.md 5b / 6)
            desat_ran = fsw_pass<NRW, PA>(P, S, I, stride, e, m, mask, n, n * P.dyn_ns, x, W, (int64_t)sun_d, desat_quiet);
            rw_sat |= 2;
#endif    // a (possibly) new wheel command: re-latch after this tick's integration
            // SpiceTask was queued for this time long before DynTask -> runs first (scheduler FIFO rule); the
            // message is then newer than the start of this integration step (quirk Q18)
            if (n > 0 && n == n_end) {
                sun_d = now_d; sun_latch_to_bus(P, m, n * P.dyn_ns); wrapped = true;
                if (J2 == 2) pfix_latch_to_bus(P, m, n * P.dyn_ns);
                if (F32) {
                    sunr_f = tof(mld3(m, M_SUNR)); sunv_f = tof(mld3(m, M_SUNV));
#pragma unroll
                    for (int q = 0; q < 6; q++) ecf[q] = (float)mld(m, M_ECL + q);
                }
            }
            // Sun third body of the ticks up to the next pass
            if (!F32) a.gsun = sun_window(P, m, x, t_mul((j < 0 ? 0.0 : now_d - dyn_d) - sun_d, LEO_NANO2SEC), h, tpf, dyn_s);
        }
        // ================= DynTask: spacecraftPlus.UpdateState (RK4 over [t-h, t]) =================
        a.h = h;
        if (LEO_RARE(wrapped || (thr_active && !(newTime + LEO_THR_MARGIN <= mld(m, M_TNEXT))))) {
            // a thruster may switch within this step (exact per-stage evaluation, then refresh the held thrust),
            // or the Sun clock wraps: every stage gets its own Sun position
            const double prev_d = j < 0 ? 0.0 : now_d - dyn_d;
            const double tBefore = t_sub(newTime, h);
            SunDt dts;
            dts.d0 = t_mul(prev_d - sun_d, 1e-9); dts.dm = dts.d0 + 0.5 * h; dts.d1 = dts.d0 + h;
            if (wrapped) dts = sun_dt_wrapped(prev_d, sun_d, tBefore, prevTime, h);
            double tauPrev = 0.0;          // time of the previous equationsOfMotion call = last stage of the previous tick
            if (j >= 0) {
                const double ppT = (n_base + j > 1) ? t_mul(prev_d - dyn_d, 1e-9) : 0.0;
                const double ph = t_sub(prevTime, ppT);
                tauPrev = t_add(t_sub(prevTime, ph), ph);
            }
            ThrEventOut o = rk4_general<J2, DIAG, PA>(P, S, stride, e, m, x, a, dts, tBefore, tauPrev, thr_factor, thr_active);
            x = o.x; thr_factor = o.factor; thr_active = o.active;
            ThrRefresh th = thr_refresh<PA>(P, S, stride, e, m, thr_active ? thr_factor : 0, a.tau_u);
            a.Lc = th.Lc; mst3(m, M_LTHR, th.L_thr); mst(m, M_TNEXT, th.t_next);
        } else if (F32) {
            StageInF af;
            af.h = (float)h; af.rho = (float)a.rho;
            af.Lc = tof(a.Lc); af.HB = tof(a.HB); af.tau_u = tof(a.tau_u);
            af.gsun = sun_accelf(PF, sunr_f + sunv_f * (float)dtsm, tof(x.r) + tof(x.v) * (0.5f * af.h));
            const bool thr_on = thr_active != 0;
            x = rk4_step_mixed<(J2 != 0), DIAG>(PF, x, af, thr_on, thr_on ? tof(mld3(m, M_FM)) : mkf(0.f, 0.f, 0.f));
        } else {
            if (J2 == 2) a.dtp = dtsm;     // orientation held at the step's mid time, like the Sun
            x = rk4_step<J2, DIAG, PA>(P, x, a, thr_active != 0, m, S, stride, e);
        }
        // ================= everything else that runs every tick: one straight-line block =================
        // the wheel invariant advances with the motor torque held over the step
        a.HB = a.HB + a.tau_u * h;
        if (!DIAG) {
#pragma unroll
            for (int i = 0; i < NRW; i++) C[i] = fmad(uJ[i], h, C[i]);
        }
        // HubEffector::modifyStates -- MRP shadow-set switch: |sigma| > 1 with the correctly rounded norm, i.e.
        // sigma.sigma > 1 + 2^-52 (sqrt(1 + 2^-52) rounds to 1).  A select, not a branch.
        {
            const double s2 = dot(x.s, x.s);
            const bool sw = s2 > 1.0000000000000002;
            const double f = -frcp(sw ? s2 : 1.0);
            x.s = mk(sw ? x.s.x * f : x.s.x, sw ? x.s.y * f : x.s.y, sw ? x.s.z * f : x.s.z);
            nswitch += sw ? 1 : 0;
        }
        // |r| of the new state: shared by the atmosphere, the eclipse model and the solar panel
        double r2 = 0., ir = 0., id = 0., rdh = 0., pgeo = 0.;
        bool penumbra = false;
        float shf = 0.f, panel_f = 0.f;
        V3f xr_f = mkf(0.f, 0.f, 0.f);
        if (F32) {
            xr_f = tof(x.r);
            const float r2f = dot(xr_f, xr_f);
            a.rho = (double)(PF.rho0 * expf(-(r2f * rsqf(r2f) - PF.Rp_atmo) * PF.inv_H));
            // EnvTask in FP32: eclipse cone tests, panel projection
            const V3f r_SBf = sunr_f - xr_f;
            const float d2f = dot(r_SBf, r_SBf), idf = rsqf(d2f);
            shf = eclipse_coref(PF, ecf, sunr_f, xr_f, r2f, d2f);
            penumbra = shf < 0.f;                              // cone-surface band / penumbra: the FP64 evaluation below
            const V3f sf = tof(x.s);
            MrpRotF R = mrp_rotf(sf);
            V3f n_N = rot_NBf(R, sf, arrf(PF.nHat_B));
            float proj = dot(n_N, r_SBf) * idf;
            if (proj < 0.f) proj = 0.f;
            panel_f = PF.panel_coef * proj * (idf * idf);
        } else {
            r2 = dot(x.r, x.r); ir = rsq(r2);
            // exponentialAtmosphere (density latched for the NEXT step, zero-order hold)
            a.rho = PA::rho0(P, S, stride, e) * exp_bounded(-(r2 * ir - P.Rp_atmo) * PA::inv_H(P, S, stride, e));
        }
        // wheel-limit flags (the latch itself is a rare event, below)
        double W[NRW];
        wheel_speeds<NRW, DIAG>(P, a.HB, C, x.w, W);
        int lim = 0;
#pragma unroll
        for (int i = 0; i < NRW; i++) lim |= (fabs(W[i]) >= P.Om_max[i] && P.Om_max[i] > 0.0) ? 1 : 0;
#ifndef LEO_EXP_NOENV
        if (!F32) {
            // EnvTask: eclipse cone tests and solar-panel geometry
            const V3 sun_r = mld3(m, M_SUNR);
            const V3 r_SB = sun_r - x.r;                       // spacecraft -> Sun
            const double d2 = dot(r_SB, r_SB);
            id = rsq(d2);
            const double ec[6] = {mld(m, M_ECL), mld(m, M_ECL + 1), mld(m, M_ECL + 2), mld(m, M_ECL + 3), mld(m, M_ECL + 4), mld(m, M_ECL + 5)};
            shadow = eclipse_cones(P, ec, sun_r, x.r, r2, d2, penumbra);
            rdh = dot(x.r, r_SB);
            MrpRot R = mrp_rot(x.s);
            V3 n_N = rot_NB(R, x.s, arr(P.nHat_B));            // panel normal in the inertial frame
            double proj = dot(n_N, r_SB) * id;                 // sHat_B . nHat_B
            if (proj < 0.) proj = 0.;
            pgeo = PA::panel_coef(P, S, stride, e) * proj * (id * id);
        }
#endif
        // clock of the NEXT tick
        const double h_this = h;
        now_d += dyn_d;
        phase = (phase + 1 == tpf) ? 0 : phase + 1;
        prevTime = newTime;
        newTime = t_mul(now_d, LEO_NANO2SEC);
        h = t_sub(newTime, prevTime);
        dtsm = t_mul((now_d - dyn_d) - sun_d, LEO_NANO2SEC) + 0.5 * h;      // (mixed precision / planet-fixed gravity only)
        // ================= rare, out of line =================
        // wheel command latch (new command, or a wheel at its speed limit) and thruster command latch
        if (LEO_RARE(rw_sat | lim | desat_ran)) {
            PostOut<NRW> po = post_tick_events<NRW>(P, S, I, stride, e, m, W, mld3(m, M_LTHR), desat_ran, (int64_t)(now_d - dyn_d), thr_factor);
#pragma unroll
            for (int i = 0; i < NRW; i++) uJ[i] = po.uJ[i];
            a.Lc = po.Lc; a.tau_u = po.tau_u;
            rw_sat = lim;
            if (po.thr_active >= 0) { thr_active = po.thr_active; mst(m, M_TNEXT, -1.0); }   // burning set: re-derive exactly
            if (desat_ran) desat_quiet = po.quiet;
            desat_ran = 0;
        }
        // penumbra / cone-surface band: the disk-overlap formula
        if (LEO_RARE(penumbra)) {
            if (F32) {
                const V3 sun_r = mld3(m, M_SUNR);
                const V3 r_SB = sun_r - x.r;
                const double r2d = dot(x.r, x.r), d2 = dot(r_SB, r_SB);
                const double ec[6] = {mld(m, M_ECL), mld(m, M_ECL + 1), mld(m, M_ECL + 2), mld(m, M_ECL + 3), mld(m, M_ECL + 4), mld(m, M_ECL + 5)};
                shadow = eclipse_core(P, ec, sun_r, x.r, r2d, rsq(r2d), r_SB, d2, rsq(d2));
                shf = (float)shadow;
            } else {
#ifdef LEO_LITERAL_ECLIPSE
                shadow = penumbra_literal(P, mld3(m, M_SUNR), x.r);
#else
                shadow = penumbra_fraction(P, ir, id, rdh);
#endif
            }
        } else if (F32) {
            shadow = (double)shf;
        }
        // ================= battery (quirk Q2: the sink message does not exist at tick 0) =================
        {
            const double panel = F32 ? (double)(panel_f * shf) : pgeo * shadow;
            const double capacity = PA::capacity(P, S, stride, e);
            double E = charge + (panel + PA::sink_power(P, S, stride, e)) * h_this;
            if (E > capacity) E = capacity;
            if (E < 0.) E = 0.;
            charge = j >= 0 ? E : charge;
        }
    }
    for (int f = 0; f < LEO_M_MIRROR; f++) SD(F_GUID + f) = mld(m, f);
    double W[NRW];
    wheel_speeds<NRW, DIAG>(P, a.HB, C, x.w, W);
    if (chunk + 1 < n_chunks) {
        // ---------------- chunk boundary inside the interval: persist the state, nothing else ----------------
        SD(F_R) = x.r.x; SD(F_R + 1) = x.r.y; SD(F_R + 2) = x.r.z;
        SD(F_V) = x.v.x; SD(F_V + 1) = x.v.y; SD(F_V + 2) = x.v.z;
        SD(F_SIG) = x.s.x; SD(F_SIG + 1) = x.s.y; SD(F_SIG + 2) = x.s.z;
        SD(F_OMG) = x.w.x; SD(F_OMG + 1) = x.w.y; SD(F_OMG + 2) = x.w.z;
#pragma unroll
        for (int i = 0; i < NRW; i++) { SD(F_WHL + i) = W[i]; SD(F_UCUR + i) = mld(m, M_U + i); }
        SD(F_RHO) = a.rho; SD(F_E) = charge; SD(F_SHADOW) = shadow;
        SI(I_TICK) = n_base - 1 + ticks; SI(I_MASK) = mask; SI(I_SWITCH) = SI(I_SWITCH) + nswitch;
        SI(I_THRFACTOR) = thr_factor; SI(I_THRACTIVE) = thr_active; SI(I_RWSAT) = rw_sat;
        out.done = 0; out.reason = 0; out.reward = 0.;
        return;
    }
    // ---------------- observation sampling (SIM:598-642) + gym bookkeeping (ENV:98-145) ----------------
    double ob0 = norm(mld3(m, M_GUID));
    double ob1 = norm(x.w);
    double wn = 0.;
#pragma unroll
    for (int i = 0; i < NRW; i++) wn += W[i] * W[i];
    const double E = charge;
    double ob2 = sqrt(wn), ob3 = E / 3600., ob4 = shadow;
    int sim_over = norm(x.r) < P.decay_radius;
    int64_t curr_step = SI(I_STEP);
    int over = (int)SI(I_OVER), reason = 0;
    if (curr_step >= P.max_length) { over = 1; reason |= 1; }
    double reward = 0.;
    if (action == 0) reward = fabs(P.reward_mult / (1. + ob0 * ob0));
    double ret = SD(F_EPRET) + reward;
    SD(F_OBS) = ob0; SD(F_OBS + 1) = ob1; SD(F_OBS + 2) = ob2; SD(F_OBS + 3) = ob3; SD(F_OBS + 4) = ob4;
    ob2 = ob2 / P.wheel_limit;
    ob3 = ob3 / P.power_max;
    if (ob2 > 1.) { over = 1; reward -= P.failure_penalty; ret -= P.failure_penalty; reason |= 2; }
    if (ob3 == 0.) { over = 1; reward -= P.failure_penalty; ret -= P.failure_penalty; reason |= 4; }
    if (sim_over) { over = 1; reason |= 8; }
    out.ob[0] = ob0; out.ob[1] = ob1; out.ob[2] = ob2; out.ob[3] = ob3; out.ob[4] = ob4;
    out.reward = reward; out.done = over; out.reason = reason;

    // ---------------- store ----------------
    SD(F_R) = x.r.x; SD(F_R + 1) = x.r.y; SD(F_R + 2) = x.r.z;
    SD(F_V) = x.v.x; SD(F_V + 1) = x.v.y; SD(F_V + 2) = x.v.z;
    SD(F_SIG) = x.s.x; SD(F_SIG + 1) = x.s.y; SD(F_SIG + 2) = x.s.z;
    SD(F_OMG) = x.w.x; SD(F_OMG + 1) = x.w.y; SD(F_OMG + 2) = x.w.z;
#pragma unroll
    for (int i = 0; i < NRW; i++) { SD(F_WHL + i) = W[i]; SD(F_UCUR + i) = mld(m, M_U + i); }
    SD(F_RHO) = a.rho; SD(F_E) = E; SD(F_SHADOW) = shadow; SD(F_EPRET) = ret;
    SI(I_TICK) = n_end; SI(I_STEP) = curr_step + 1; SI(I_MASK) = mask; SI(I_SWITCH) = SI(I_SWITCH) + nswitch;
    SI(I_THRFACTOR) = thr_factor; SI(I_THRACTIVE) = thr_active; SI(I_OVER) = over; SI(I_RWSAT) = rw_sat;
#undef SD
#undef SI
}

}  // namespace leo
