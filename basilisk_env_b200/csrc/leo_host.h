// leo_host.h -- host-side derivation of the kernel parameter block from bskenv_config.
// This is where the reference's scenario wiring (set_dynamics / set_fsw,
// /root/reference/basilisk_env/simulators/leoPowerAttitudeSimulator.py:195-490, cited SIM:line, and
// actuatorPrimatives.py, cited AP:line) turns into numbers; Basilisk factory values are cited [BSK].
#pragma once
#include <math.h>
#include <string.h>
#include <string>
#include "../../include/bskenv.h"
#include "leo_params.h"

namespace leo_host {

static inline bool inv3(const double m[9], double out[9])
{
    double det = m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6]);
    if (fabs(det) < 1e-300) return false;
    out[0] = (m[4] * m[8] - m[5] * m[7]) / det; out[1] = (m[2] * m[7] - m[1] * m[8]) / det; out[2] = (m[1] * m[5] - m[2] * m[4]) / det;
    out[3] = (m[5] * m[6] - m[3] * m[8]) / det; out[4] = (m[0] * m[8] - m[2] * m[6]) / det; out[5] = (m[2] * m[3] - m[0] * m[5]) / det;
    out[6] = (m[3] * m[7] - m[4] * m[6]) / det; out[7] = (m[1] * m[6] - m[0] * m[7]) / det; out[8] = (m[0] * m[4] - m[1] * m[3]) / det;
    return true;
}
static inline int64_t sec2nano(double s) { return (int64_t)(s * 1e9 + 0.5); }   // [BSK: macros.sec2nano]

static inline void default_config(bskenv_config *c)
{
    memset(c, 0, sizeof(*c));
    c->abi_version = BSKENV_ABI_VERSION;
    c->dynRate = 0.1; c->fswRate = 1.0; c->step_duration = 180.;            // ENV:185, ENV:40
    c->mass = 330; c->width = 1.38; c->depth = 1.04; c->height = 1.58;        // SIM:129,137-139
    c->planetRadius = 6378.1366 * 1000.; c->baseDensity = 1.22; c->scaleHeight = 8e3;   // SIM:146-148
    c->disturbance_magnitude = 2e-4;                                           // SIM:151
    c->nHat_B[0] = 0; c->nHat_B[1] = -1; c->nHat_B[2] = 0;                      // SIM:158
    c->panelArea = 0.2 * 0.3; c->panelEfficiency = 0.20;                       // SIM:159-160
    c->powerDraw = -5.0; c->storageCapacity = 20.0 * 3600.;                    // SIM:163,166
    c->sigma_R0N[0] = 1; c->sigma_R0N[1] = 0; c->sigma_R0N[2] = 0;             // SIM:170
    c->K = 7; c->Ki = -1.0; c->P = 35;                                         // SIM:178-180
    c->hs_min = 4.; c->thrForceSign = 1; c->maxCounterValue = 4; c->thrMinFireTime = 0.002;  // SIM:183-190
    c->max_length = 3 * 180;                                                   // ENV:25
    c->wheel_limit_rpm = 3000; c->power_max = 20.0; c->failure_penalty = 1;    // ENV:36-42
}

// returns "" on success, else an error message
static inline std::string build_params(const bskenv_config &c, LeoParams &p)
{
    memset(&p, 0, sizeof(p));
    if (c.abi_version != BSKENV_ABI_VERSION) return "bskenv_config.abi_version mismatch";
    if (!(c.dynRate > 0) || !(c.fswRate > 0) || !(c.step_duration > 0)) return "rates must be positive";
    p.dyn_ns = sec2nano(c.dynRate); p.fsw_ns = sec2nano(c.fswRate); p.step_ns = sec2nano(c.step_duration);
    if (p.fsw_ns % p.dyn_ns || p.step_ns % p.fsw_ns) return "fswRate must be a multiple of dynRate and step_duration a multiple of fswRate";
    p.ticks_per_fsw = (int32_t)(p.fsw_ns / p.dyn_ns); p.fsw_per_step = (int32_t)(p.step_ns / p.fsw_ns);
    if (c.Ki >= 0) return "integral feedback (Ki >= 0) is not on the reference path";
    if (c.thrForceSign <= 0) return "only on-pulsing thrusters (thrForceSign = +1) are on the reference path";
    if (c.max_length < 0 || c.mass <= 0) return "bad mass / max_length";
    const double RPM = 0.10471975511965977;                      // [BSK: macros.RPM]
    // hub: solid cuboid inertia (SIM:245-250)
    p.inv_mass = 1.0 / c.mass;
    p.I[0] = 1. / 12. * c.mass * (pow(c.width, 2.) + pow(c.depth, 2.));
    p.I[4] = 1. / 12. * c.mass * (pow(c.depth, 2.) + pow(c.height, 2.));
    p.I[8] = 1. / 12. * c.mass * (pow(c.width, 2.) + pow(c.height, 2.));
    memcpy(p.I_fsw, p.I, sizeof(p.I));                           // same inertia in FSW (SIM:392-403)
    // gravity (SIM:227-232): Earth central + Sun third body; NO J2 in the reference (SURVEY M1)
    p.mu_c = 0.3986004415e15; p.mu_sun = 1.32712440018e20;       // [BSK: simIncludeGravBody]
    p.j2k = 1.5 * 1.08262668355e-3 * p.mu_c * (6378136.6 * 6378136.6);
    p.hill_cel_pun = c.hill_cel_pun; p.use_j2 = c.use_j2 ? 1 : 0;
    if (c.precision != 0 && c.precision != 1) return "precision must be 0 (FP64) or 1 (mixed: FP32 stages, FP64 accumulation)";
    p.mixed = c.precision;
    // Honeywell HR16 at 50 Nms ([BSK: simIncludeRW.Honeywell_HR16]): three along the body axes (AP:20-37), or the
    // four-wheel pyramid of the opNav spacecraft (opNav_models/BSK_OpNavDynamics.py:269-293:
    // gsHat = M3(-az) M2(el) e_x = (cos el cos az, cos el sin az, sin el))
    if (c.rw_set != 0 && c.rw_set != 1) return "rw_set must be 0 (triad) or 1 (four-wheel pyramid)";
    p.nrw = c.rw_set == 1 ? 4 : 3;
    for (int i = 0; i < p.nrw; i++) {
        if (c.rw_set == 1) {
            const double D2R = 3.14159265358979323846 / 180.0, el = 40.0 * D2R, az = (45.0 + 90.0 * i) * D2R;
            p.gs[i][0] = cos(el) * cos(az); p.gs[i][1] = cos(el) * sin(az); p.gs[i][2] = sin(el);
        } else {
            p.gs[i][i] = 1.0;
        }
        p.Om_max[i] = 6000.0 * RPM; p.u_max[i] = 0.200; p.u_min[i] = 0.0;
        p.Js[i] = 50. / p.Om_max[i]; p.invJs[i] = 1.0 / p.Js[i];
    }
    double D[9];
    memcpy(D, p.I, sizeof(D));
    for (int i = 0; i < p.nrw; i++)
        for (int a = 0; a < 3; a++)
            for (int b = 0; b < 3; b++) D[3 * a + b] -= p.Js[i] * p.gs[i][a] * p.gs[i][b];
    memcpy(p.D, D, sizeof(D));
    if (!inv3(D, p.Dinv)) return "singular back-substitution matrix";
    { // structural fast path: diagonal inertia and wheel i along body axis i
        bool diag = p.nrw == 3;
        for (int a = 0; a < 3 && diag; a++)
            for (int b = 0; b < 3; b++)
                if (a != b && (p.I[3 * a + b] != 0.0 || p.gs[a][b] != 0.0)) diag = false;
        for (int a = 0; a < 3 && diag; a++) if (p.gs[a][a] != 1.0) diag = false;
        p.diag = diag ? 1 : 0;
    }
    { // rwMotorTorque map with controlAxes_B = identity (SIM:173-175): Umap = Gs^T (Gs Gs^T)^-1
        double M[9] = {0}, Mi[9];
        for (int a = 0; a < 3; a++)
            for (int b = 0; b < 3; b++)
                for (int i = 0; i < p.nrw; i++) M[3 * a + b] += p.gs[i][a] * p.gs[i][b];
        if (!inv3(M, Mi)) return "wheel set does not span the control axes";
        for (int i = 0; i < p.nrw; i++)
            for (int b = 0; b < 3; b++)
                for (int a = 0; a < 3; a++) p.Umap[i][b] += p.gs[i][a] * Mi[3 * a + b];
    }
    { // eight drag facets (SIM:274-281), all with axis-aligned normals -> collapsed per axis/sign
        const double A[8] = {0.2 * 0.3, 0.2 * 0.3, 0.1 * 0.2, 0.1 * 0.2, 0.1 * 0.3, 0.1 * 0.3, 1. * 2., 1. * 2.};
        const int axis[8] = {0, 0, 1, 1, 2, 2, 1, 1}, sign[8] = {0, 1, 0, 1, 0, 1, 0, 1};   // 0:+ 1:-
        const double Lc[8][3] = {{0.05, 0, 0}, {0.05, 0, 0}, {0, 0.15, 0}, {0, -0.15, 0}, {0, 0, 0.1}, {0, 0, -0.1}, {0, 2., 0}, {0, 2., 0}};
        const double Cd = 2.2;
        double K[3][2] = {{0}}, M[3][2][3] = {{{0}}};
        for (int f = 0; f < 8; f++) {
            double k = 0.5 * Cd * A[f];
            K[axis[f]][sign[f]] += k;
            for (int j = 0; j < 3; j++) M[axis[f]][sign[f]][j] += k * Lc[f][j];
        }
        for (int ax = 0; ax < 3; ax++) {
            p.dragKa[ax] = 0.5 * (K[ax][0] + K[ax][1]) * p.inv_mass; p.dragKd[ax] = 0.5 * (K[ax][0] - K[ax][1]) * p.inv_mass;
            if (p.dragKd[ax] != 0.0) p.diag = 0;        // the fast path drops the Kd terms (equal + / - facet areas)
            for (int j = 0; j < 3; j++) {
                p.dragMa[ax][j] = 0.5 * (M[ax][0][j] + M[ax][1][j]); p.dragMd[ax][j] = 0.5 * (M[ax][0][j] - M[ax][1][j]);
                if (ax != j && (p.dragMa[ax][j] != 0.0 || p.dragMd[ax][j] != 0.0)) p.diag = 0;
            }
        }
    }
    p.dist_mag = c.disturbance_magnitude;
    p.rho0 = c.baseDensity; p.inv_H = 1.0 / c.scaleHeight; p.Rp_atmo = c.planetRadius;
    p.R_sun = 695000.0 * 1000; p.R_planet = 6378.1366 * 1000;    // [BSK: astroConstants REQ_SUN, REQ_EARTH]
    for (int k = 0; k < 3; k++) p.nHat_B[k] = c.nHat_B[k];
    const double AUm = 149597870.693 * 1000.;
    p.panel_coef = c.panelEfficiency * 1372.5398 * c.panelArea * AUm * AUm;     // [BSK: SOLAR_FLUX_EARTH]
    p.sink_power = c.powerDraw; p.capacity = c.storageCapacity;
    p.K = c.K; p.P = c.P; p.Ki = c.Ki;
    for (int k = 0; k < 3; k++) p.sigma_R0N[k] = c.sigma_R0N[k];
    p.hs_min = c.hs_min;
    { // MOOG Monarc-1 octet (AP:73-156, [BSK: simIncludeThruster.MOOG_Monarc_1])
        const double loc[8][3] = {
            {3.874945160902288e-2, -1.206182747348013, 0.85245}, {3.874945160902288e-2, -1.206182747348013, -0.85245},
            {-3.8749451609022656e-2, -1.206182747348013, 0.85245}, {-3.8749451609022656e-2, -1.206182747348013, -0.85245},
            {-3.874945160902288e-2, 1.206182747348013, 0.85245}, {-3.874945160902288e-2, 1.206182747348013, -0.85245},
            {3.8749451609022656e-2, 1.206182747348013, 0.85245}, {3.8749451609022656e-2, 1.206182747348013, -0.85245}};
        const double dir[8][3] = {
            {-0.7071067811865476, 0.7071067811865475, 0.0}, {-0.7071067811865476, 0.7071067811865475, 0.0},
            {0.7071067811865475, 0.7071067811865476, 0.0}, {0.7071067811865475, 0.7071067811865476, 0.0},
            {0.7071067811865476, -0.7071067811865475, 0.0}, {0.7071067811865476, -0.7071067811865475, 0.0},
            {-0.7071067811865475, -0.7071067811865476, 0.0}, {-0.7071067811865475, -0.7071067811865476, 0.0}};
        double DDT[9] = {0}, DDTi[9];
        for (int i = 0; i < 8; i++) {
            for (int k = 0; k < 3; k++) { p.thr_loc[i][k] = loc[i][k]; p.thr_dir[i][k] = dir[i][k]; }
            p.thr_D[0][i] = loc[i][1] * dir[i][2] - loc[i][2] * dir[i][1];
            p.thr_D[1][i] = loc[i][2] * dir[i][0] - loc[i][0] * dir[i][2];
            p.thr_D[2][i] = loc[i][0] * dir[i][1] - loc[i][1] * dir[i][0];
        }
        for (int a = 0; a < 3; a++)
            for (int b = 0; b < 3; b++)
                for (int i = 0; i < 8; i++) DDT[3 * a + b] += p.thr_D[a][i] * p.thr_D[b][i];
        if (!inv3(DDT, DDTi)) return "thruster set does not span the control axes";
        for (int i = 0; i < 8; i++)
            for (int b = 0; b < 3; b++)
                for (int a = 0; a < 3; a++) p.thr_W[i][b] += p.thr_D[a][i] * DDTi[3 * a + b];
        p.thr_Fmax = 0.9; p.thr_MinOnTime = 0.020;
    }
    p.thrMinFireTime = c.thrMinFireTime; p.thrForceSign = c.thrForceSign; p.maxCounterValue = c.maxCounterValue;
    p.tfm_eps = 0.0; p.tfm_angErrThresh = 0.0;                   // zero-initialised thrForceMappingConfig
    p.wheel_rpm2rad = RPM;
    p.wheel_limit = c.wheel_limit_rpm * RPM;                     // ENV:36
    p.power_max = c.power_max;
    p.reward_mult = c.max_length > 0 ? 1. / c.max_length : 0.0;  // ENV:41
    p.failure_penalty = c.failure_penalty;
    p.decay_radius = 6378.1366 / 1000.;                          // SIM:641 (quirk Q6: km/1000 compared with metres)
    p.max_length = c.max_length; p.auto_reset = c.auto_reset;
    // '2021 MAY 04 07:47:48.965 (UTC)' (SIM:219) as days of TT from J2000: JD 2459338.5 + UTC seconds + 69.184 s
    p.epoch_days = 7793.5 + (28068.965 + 69.184) / 86400.0;
    return "";
}

// ---- per-env parameter pools (bskenv_set_param_pool): BSKENV_PARAM_DIM reference values per row ----
static inline void param_row_get(const bskenv_config &c, double r[BSKENV_PARAM_DIM])
{
    const double v[BSKENV_PARAM_DIM] = {c.mass, c.width, c.depth, c.height, c.baseDensity, c.scaleHeight, c.disturbance_magnitude,
                                        c.panelArea, c.panelEfficiency, c.powerDraw, c.storageCapacity, c.K, c.P, c.hs_min};
    memcpy(r, v, sizeof(v));
}
static inline void param_row_set(bskenv_config &c, const double r[BSKENV_PARAM_DIM])
{
    c.mass = r[0]; c.width = r[1]; c.depth = r[2]; c.height = r[3]; c.baseDensity = r[4]; c.scaleHeight = r[5];
    c.disturbance_magnitude = r[6]; c.panelArea = r[7]; c.panelEfficiency = r[8]; c.powerDraw = r[9]; c.storageCapacity = r[10];
    c.K = r[11]; c.P = r[12]; c.hs_min = r[13];
}
// The values a row puts into an env's parameter block (leo_params.h: LeoPField), taken from the parameter block that
// build_params derived for the configuration with the row's values: the device never re-derives them.
static inline void param_row_derive(const LeoParams &p, const double raw[BSKENV_PARAM_DIM], double row, double out[LEO_NPD])
{
    out[PE_INV_MASS] = p.inv_mass;
    for (int k = 0; k < 3; k++) {
        out[PE_D + k] = p.D[4 * k]; out[PE_DINV + k] = p.Dinv[4 * k]; out[PE_DRAGKA + k] = p.dragKa[k]; out[PE_IFSW + k] = p.I_fsw[4 * k];
    }
    out[PE_RHO0] = p.rho0; out[PE_INV_H] = p.inv_H; out[PE_PANEL] = p.panel_coef; out[PE_SINK] = p.sink_power;
    out[PE_CAP] = p.capacity; out[PE_K] = p.K; out[PE_P] = p.P; out[PE_HSMIN] = p.hs_min; out[PE_DIST] = p.dist_mag;
    out[PE_ROW] = row;
    for (int k = 0; k < BSKENV_PARAM_DIM; k++) out[PE_RAW + k] = raw[k];
}
// Checks a row against the configuration it is applied to and derives it; returns "" or an error message.
static inline std::string param_row_build(const bskenv_config &base, const double raw[BSKENV_PARAM_DIM], double row, double out[LEO_NPD])
{
    for (int k = 0; k < BSKENV_PARAM_DIM; k++)
        if (!isfinite(raw[k])) return "non-finite value";
    if (!(raw[0] > 0) || !(raw[1] > 0) || !(raw[2] > 0) || !(raw[3] > 0)) return "mass, width, depth and height must be positive";
    if (!(raw[5] > 0)) return "scaleHeight must be positive";
    if (!(raw[10] > 0)) return "storageCapacity must be positive";
    bskenv_config c = base;
    param_row_set(c, raw);
    LeoParams p;
    const std::string err = build_params(c, p);
    if (!err.empty()) return err;
    param_row_derive(p, raw, row, out);
    return "";
}

// Checks one initial-condition pool row of `dim` doubles whose first three are the position rN (LEO: BSKENV_IC_DIM, opNav:
// BSKENV_OPNAV_IC_DIM); returns "" or an error message.
static inline std::string ic_row_check(const double *row, int dim)
{
    for (int k = 0; k < dim; k++)
        if (!isfinite(row[k])) return "non-finite value in column " + std::to_string(k);
    if (row[0] == 0.0 && row[1] == 0.0 && row[2] == 0.0) return "zero position vector rN";
    return "";
}

// SURVEY 8(f)-4: normalised degree-2 coefficients (C20, C21, S21, C22, S22; the form gravity-model files carry and
// Basilisk's loadGravFromFile reads) -> mu Req^2 [M] of the closed-form gradient used by the kernel.
// Un-normalisation: C_nm = Cbar_nm sqrt((2 - delta_0m)(2n + 1)(n - m)!/(n + m)!).
static inline void set_degree2(LeoParams &p, const double cbar[5])
{
    static const double ggm03s[5] = {-4.8416537173459064e-04, -2.0661550900e-10, 1.3844138138e-09, 2.4393836573e-06, -1.4002737040e-06};
    if (!cbar) cbar = ggm03s;
    const double C20 = cbar[0] * sqrt(5.0), C21 = cbar[1] * sqrt(5.0 / 3.0), S21 = cbar[2] * sqrt(5.0 / 3.0);
    const double C22 = cbar[3] * sqrt(5.0 / 12.0), S22 = cbar[4] * sqrt(5.0 / 12.0);
    const double k = p.mu_c * (6378136.6 * 6378136.6);
    p.gm2[0] = k * (-0.5 * C20 + 3.0 * C22); p.gm2[1] = k * (-0.5 * C20 - 3.0 * C22); p.gm2[2] = k * C20;
    p.gm2[3] = k * 3.0 * S22; p.gm2[4] = k * 1.5 * C21; p.gm2[5] = k * 1.5 * S21;
    p.grav_pfix = 1;
}

// Number of chunks a decision interval is executed in (leo_step_env): a function of the task rates only, so that a
// trajectory never depends on the batch size, the sharding or the entry point.  Six chunks of 300 ticks at the reference
// rates; one when the interval does not split into whole flight-software periods.
#ifndef LEO_STEP_CHUNKS
#define LEO_STEP_CHUNKS 6
#endif
static inline int step_chunks(const LeoParams &p)
{
    const int c = LEO_STEP_CHUNKS;
    return (c > 1 && p.fsw_per_step % c == 0) ? c : 1;
}

static inline void build_params_f(const LeoParams &p, LeoParamsF &f)
{
    memset(&f, 0, sizeof(f));
    f.mu_c = (float)p.mu_c; f.mu_sun = (float)p.mu_sun; f.j2k = (float)p.j2k;
    for (int i = 0; i < 9; i++) { f.D[i] = (float)p.D[i]; f.Dinv[i] = (float)p.Dinv[i]; }
    for (int a = 0; a < 3; a++) {
        f.dragKa[a] = (float)p.dragKa[a]; f.dragKd[a] = (float)p.dragKd[a]; f.nHat_B[a] = (float)p.nHat_B[a];
        for (int b = 0; b < 3; b++) { f.dragMa[a][b] = (float)p.dragMa[a][b]; f.dragMd[a][b] = (float)p.dragMd[a][b]; }
    }
    f.rho0 = (float)p.rho0; f.inv_H = (float)p.inv_H; f.Rp_atmo = (float)p.Rp_atmo;
    f.R_sun = (float)p.R_sun; f.R_planet = (float)p.R_planet; f.panel_coef = (float)p.panel_coef;
}

// FP64 flop per env-decision-step of the step kernel AS BUILT (DESIGN.md "Flop model"): FMA = 2, add/mul = 1,
// one per MUFU seed; counted from the operation list of leo_core.cuh for modes 0/1 and cross-checked against the
// executed instruction counters of ncu (2 DFMA + DMUL + DADD thread instructions per env: 2.074e6 for the
// reference configuration, profiles/ncu_r01c.md; this formula gives 2.0736e6).  It is the work the kernel performs,
// not the larger count of the un-fused Basilisk formulation (SURVEY 8(d): 4.29e6), so the roofline fraction built
// on it is the fraction of the FP64 pipe's flop rate actually delivered.
//   per RK stage   gravity 22, MRP rotation set-up 17, [BN] v 30, collapsed drag 21 (equal + / - facet areas: no Kd terms), torque/gyro/inverse
//                  inertia 42, MRP kinematics 31                                                   = 163 (diagonal path)
//   RK4 per tick   stage inputs 96, weighted slope sums 96, final update 12                          = 204
//   per tick       Sun third body 55, invariant/|r| 30, MRP switch as a select (reciprocal + 3 products, every tick) 10,
//                  atmosphere 40, wheel test 6, eclipse + panel + battery 105                          = 246
//   FSW pass       hillPoint 130, attTrackingError 146, MRP_Feedback 69, rwMotorTorque 15           = 360
static inline double flops_per_step(const LeoParams &p)
{
    double F_eom = 163.0;
    const double F_rk4 = 204.0, F_tick = 246.0;
    double F_fsw = 360.0;
    if (!p.diag) F_eom += 42.0 + 8.0 * (p.nrw - 3);        // full 3x3 D / Dinv / drag moment arms, wheel invariants
    if (p.grav_pfix) F_eom += 92.0;      // DCM Euler step 18, r_Pfix 15, |r|^-5/-7 9, M r + quadratic form 29, g_Pfix 9, back-rotation 15 (- point-mass share 3)
    else if (p.use_j2) F_eom += 14.0;
    if (p.nrw == 4) F_fsw += 5.0;
    double ticks = (double)p.ticks_per_fsw * p.fsw_per_step;
    // the Sun third-body term (55 flop + 6 for its mid-step position and time) is evaluated once per flight-software period,
    // not per tick (leo_core.cuh: sun_window); matched to ncu's executed count (profiles/ncu_leo_r02c.md: 1.9483e6 per env-step)
    return ticks * (4 * F_eom + F_rk4 + (F_tick - 61.0)) + p.fsw_per_step * (F_fsw + 59.0);
}

}  // namespace leo_host
