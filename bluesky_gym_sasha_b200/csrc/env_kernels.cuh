// env_kernels.cuh -- K1/K3/K4/K5/K6: the batched BlueSky-Gym step as one kernel launch.
//
// One group of G lanes (G = 1, 8, 16 or 32; lane = aircraft slot) owns one env instance; aircraft
// state lives in registers for all n_sub simulator substeps of an env step and is read / written
// once per step as coalesced float4 / double2 (slot index fastest, so a warp touches 512 contiguous
// bytes per array).  Inside a substep: autopilot (select modes, LNAV/FMS for MergeEnv's routes) ->
// in-group all-pairs state-based CD (records staged in shared memory, broadcast LDS.128; K3) ->
// OpenAP-lite limits -> airspeed / heading / vertical-speed response -> flat-earth lat/lon
// integration in float64 (K1).  Then observation + reward + termination (K4), the TimeLimit cap and
// vector autoreset with a Philox-keyed scenario generator (K5).
//
// Replaces, per env step: Env.step of the reference (e.g. horizontal_cr_env.py:103-125 ->
// n_sub x bs.sim.step() -> _get_obs :150-213 -> _get_reward :225-270), i.e. upstream
// Simulation.step / Traffic.update / Autopilot.update / perfoap.limits / StateBased.detect as
// restated in oracle/traffic.py, oracle/perf.py, oracle/statebased.py, oracle/envs.py.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "bsg_internal.h"
#include "bsg_math.cuh"
#include "cd_pair.cuh"
#include "rng.cuh"

namespace bsg {

constexpr int kEnvThreads = 128;
constexpr int kEnvBlocksPerSm = 7;      // 28 warps per SM: what 72 registers per thread allow
constexpr uint32_t kFlAlive = 1u, kFlLnav = 2u, kFlLastWp = 4u, kFlTgt = 8u /* aux.w caches allow_tas */, kFlWpShift = 8u;
enum { kModeStep = 0, kModeReset = 1, kModeTraf = 2 };

// bluesky.traffic.performance.openap.phase constants
enum { PH_NA = 0, PH_TO = 1, PH_IC = 2, PH_CL = 3, PH_CR = 4, PH_DE = 5, PH_AP = 6, PH_LD = 7, PH_GD = 8 };

struct EnvParams {
    int env_type, E, n_int, cd_enabled, autoreset, max_steps, hdg_random, n_sub, fms_rel_freq, mode;
    int obs_dim, act_dim, info_dim;
    int fc_slot;                  // which of final_count[0..1] counts this launch's finished envs (the other is zeroed for the next)
    float simdt, R2, hpz, dtlook, rpz, init_alt, inv_axmax_gd, inv_axmax_air;
    double init_tas0;             // TAS the scenario generator creates aircraft with (fixed altitude / CAS envs), host-evaluated
    double fix_lat, fix_lon;      // MergeEnv FIX (merge_env.py:43-46), evaluated on the host in double
    uint64_t seed;
    long long gid0;
    bsg_perf perf;
    double2* pos; float4* kin; float4* cmd; float4* aux; uint32_t* flags;
    float* tcpamax; uint8_t* inconf;
    double* ef64; float* ef32; int32_t* ei32; double* poly;
    float* obs; float* final_obs; int32_t* final_ids; int32_t* final_count; float* reward; uint8_t* term; uint8_t* trunc; float* info;
    const float* actions; const uint8_t* reset_mask;
    uint32_t* cd_pairs; float* cd_attr; int cd_pair_cap;      // in-sim ASAS pair lists of the last substep (may be null)
    // WindFieldWrapper (bsg_set_wind): wind_n == 0 <=> no wind
    int wind_n, wind_nalt, wind_obs, sector_uniform;
    float wind_altstep;
    const float* wind_lat; const float* wind_lon; const float* wind_vn; const float* wind_ve;
    float2* gsv;
};

struct Ac {
    double lat, lon;
    float alt, tas, hdg, vs;
    float selspd, selalt, selvs, aptrk;
    float ax, curlegdir, cas;
    float tgt;                // allow_tas of the last launch's targets (valid with kFlTgt; see env_kernel)
    uint32_t flags;
    float gsn, gse;           // cached tas*cos(hdg), tas*sin(hdg) of the last groundspeed update
    float coslat;             // cached cos(lat) of the last position update
    float tcpamax; bool inconf;
};

struct EnvS {
    double wpt_lat, wpt_lon, target_alt, poly_area;
    float total_reward, drift_sum, final_alt, last_wdist, last_drift;
    float step_reward; int step_done;      // StaticObstacle: outcome of the per-substep checks (not persisted)
    int step, episode, simk, wpt_reach, drift_n, intrusions, num_ac, nvert, needs_reset, faf, nconf, nlos, rflags;
};

// ---- MergeEnv constants: merge_env.py:40-46 (FIX = get_point_at_distance(RWY, 200 km, 0 deg)) ----
constexpr double kRwyLat = 52.36239301495972, kRwyLon = 4.713195734579777;
constexpr double kSectorLat0 = 51.990426702297746, kSectorLon0 = 4.376124857109851;   // sector_cr_env.py:16

// ---- float64 helpers used only by the (rare) scenario generators -----------------------------------
__device__ inline void d_atmos(double h, double& p, double& rho, double& T) {
    T = fmax(288.15 - 0.0065 * h, 216.65);
    double rhotrop = 1.225 * pow(T / 288.15, 4.256848030018761);
    rho = rhotrop * exp(-fmax(0.0, h - 11000.0) / 6341.552161);
    p = rho * 287.05287 * T;
}
// (the _at forms take the pressure and density at the altitude: the host evaluates them once when the altitude is a
// configuration constant, which keeps the double-precision pow / exp of d_atmos out of that env's kernel)
__device__ inline double d_cas2tas_at(double cas, double p, double rho) {
    double q = 101325.0 * (pow(1.0 + 1.225 * cas * cas / (7.0 * 101325.0), 3.5) - 1.0);
    double t = sqrt(7.0 * p / rho * (pow(q / p + 1.0, 2.0 / 7.0) - 1.0));
    return cas < 0 ? -t : t;
}
__device__ inline double d_tas2cas_at(double tas, double p, double rho) {
    double q = p * (pow(1.0 + rho * tas * tas / (7.0 * p), 3.5) - 1.0);
    double c = sqrt(7.0 * 101325.0 / 1.225 * (pow(q / 101325.0 + 1.0, 2.0 / 7.0) - 1.0));
    return tas < 0 ? -c : c;
}
__device__ inline double d_cas2tas(double cas, double h) {
    double p, rho, T;
    d_atmos(h, p, rho, T);
    return d_cas2tas_at(cas, p, rho);
}
__device__ inline double d_tas2cas(double tas, double h) {
    double p, rho, T;
    d_atmos(h, p, rho, T);
    return d_tas2cas_at(tas, p, rho);
}
// functions.py:24-42
__device__ inline void d_point_at_distance(double lat1, double lon1, double d_km, double brg, double& lat2, double& lon2) {
    double la = lat1 * kDeg2RadD, lo = lon1 * kDeg2RadD, a = brg * kDeg2RadD, ang = d_km / 6371.0;
    double l2 = asin(sin(la) * cos(ang) + cos(la) * sin(ang) * cos(a));
    double o2 = lo + atan2(sin(a) * sin(ang) * cos(la), cos(ang) - sin(la) * sin(l2));
    lat2 = l2 * kRad2DegD; lon2 = o2 * kRad2DegD;
}

// Traffic.cre with SI arguments (oracle/traffic.py::Traffic.cre)
__device__ inline void ac_create_tas(Ac& a, double lat, double lon, double hdg, double alt, double cas_cmd, double tas) {
    a.lat = lat; a.lon = lon > 180.0 ? lon - 360.0 : (lon < -180.0 ? lon + 360.0 : lon);
    a.alt = (float)alt; a.tas = (float)tas; a.hdg = (float)hdg; a.vs = 0.0f;
    a.selspd = (float)cas_cmd; a.selalt = (float)alt; a.selvs = 0.0f; a.aptrk = (float)hdg;
    a.ax = 0.0f; a.curlegdir = -999.0f; a.cas = (float)cas_cmd; a.tgt = 0.0f;
    a.flags = kFlAlive;
    double hr = hdg * kDeg2RadD;
    a.gsn = (float)(tas * cos(hr)); a.gse = (float)(tas * sin(hr));
    a.coslat = (float)cos(a.lat * kDeg2RadD);
    a.tcpamax = 0.0f; a.inconf = false;
}
// same with the cosine / sine of the heading at hand (the generator just computed them)
__device__ inline void ac_create_dir(Ac& a, double lat, double lon, double hdg, double alt, double cas_cmd, double tas,
                                     double ch, double sh) {
    a.lat = lat; a.lon = lon > 180.0 ? lon - 360.0 : (lon < -180.0 ? lon + 360.0 : lon);
    a.alt = (float)alt; a.tas = (float)tas; a.hdg = (float)hdg; a.vs = 0.0f;
    a.selspd = (float)cas_cmd; a.selalt = (float)alt; a.selvs = 0.0f; a.aptrk = (float)hdg;
    a.ax = 0.0f; a.curlegdir = -999.0f; a.cas = (float)cas_cmd; a.tgt = 0.0f;
    a.flags = kFlAlive;
    a.gsn = (float)(tas * ch); a.gse = (float)(tas * sh);
    a.coslat = __cosf((float)a.lat * kDeg2Rad);                // (the expression ac_load rebuilds it with)
    a.tcpamax = 0.0f; a.inconf = false;
}
__device__ inline void ac_create(Ac& a, double lat, double lon, double hdg, double alt, double cas_cmd) {
    ac_create_tas(a, lat, lon, hdg, alt, cas_cmd, d_cas2tas(cas_cmd, alt));     // the reference never passes a Mach number to cre
}
__device__ inline void ac_clear(Ac& a) {
    a.lat = 0.0; a.lon = 0.0; a.alt = 0.0f; a.tas = 0.0f; a.hdg = 0.0f; a.vs = 0.0f;
    a.selspd = 0.0f; a.selalt = 0.0f; a.selvs = 0.0f; a.aptrk = 0.0f; a.ax = 0.0f; a.curlegdir = -999.0f;
    a.cas = 0.0f; a.tgt = 0.0f; a.flags = 0u; a.gsn = 0.0f; a.gse = 0.0f; a.coslat = 1.0f; a.tcpamax = 0.0f; a.inconf = false;
}

// ---- wind field: upstream windfield.py::getdata (oracle/windfield.py) -------------------------------
// inverse-distance-squared weights on the flat-earth metric in degrees (longitude scaled by the cosine of the
// mean latitude), linear interpolation between the two bracketing altitude rows
__device__ __forceinline__ void wind_at(const EnvParams& P, double latd, double lond, float alt, float& vn, float& ve) {
    const int n = P.wind_n;
    int ia = 0;
    float fa = 0.0f;
    if (P.wind_nalt > 1) {
        float idx = fmaxf(0.0f, fminf(P.wind_altstep * (float)(P.wind_nalt - 1), alt) / P.wind_altstep);
        ia = min((int)floorf(idx), P.wind_nalt - 2);
        fa = idx - (float)ia;
    }
    float wsum = 0.0f, sn = 0.0f, se = 0.0f;
    for (int k = 0; k < n; ++k) {
        const float plat = P.wind_lat[k], plon = P.wind_lon[k];
        const float dy = (float)(latd - (double)plat), dxl = (float)(lond - (double)plon);
        const float cav = __cosf(0.5f * ((float)latd + plat) * kDeg2Rad);
        const float dx = cav * dxl;
        const float w = 1.0f / fmaxf(fmaf(dx, dx, dy * dy), 1e-20f);
        float vnk = P.wind_vn[ia * n + k], vek = P.wind_ve[ia * n + k];
        if (P.wind_nalt > 1) {
            vnk = fmaf(fa, P.wind_vn[(ia + 1) * n + k] - vnk, vnk);
            vek = fmaf(fa, P.wind_ve[(ia + 1) * n + k] - vek, vek);
        }
        wsum += w; sn = fmaf(w, vnk, sn); se = fmaf(w, vek, se);
    }
    vn = n ? sn / wsum : 0.0f;
    ve = n ? se / wsum : 0.0f;
}
// bs.traf.gs: equals tas without wind (and below 50 ft)
__device__ __forceinline__ float ac_gs(const Ac& a, const EnvParams& P) {
    return P.wind_n > 0 ? sqrtf(fmaf(a.gsn, a.gsn, a.gse * a.gse)) : a.tas;
}
__device__ __forceinline__ float ac_trk(const Ac& a, const EnvParams& P) {
    return P.wind_n > 0 ? mod360(kRad2Deg * atan2f(a.gse, a.gsn)) : a.hdg;
}

// ---- state I/O (coalesced: consecutive lanes -> consecutive float4 / double2) ----------------------
__device__ __forceinline__ void ac_load(Ac& a, const EnvParams& P, long long idx) {
    // (loads only: nothing here waits for the data, see ac_finish_load)
    double2 p = P.pos[idx];
    float4 k = P.kin[idx], c = P.cmd[idx], x = P.aux[idx];
    a.lat = p.x; a.lon = p.y;
    a.alt = k.x; a.tas = k.y; a.hdg = k.z; a.vs = k.w;
    a.selspd = c.x; a.selalt = c.y; a.selvs = c.z; a.aptrk = c.w;
    a.ax = x.x; a.curlegdir = x.y; a.cas = x.z; a.tgt = x.w;
    a.flags = P.flags[idx];
    a.gsn = 0.0f; a.gse = 0.0f;
    if (P.gsv) { float2 g = P.gsv[idx]; a.gsn = g.x; a.gse = g.y; }      // with wind the ground speed is state
    a.tcpamax = 0.0f; a.inconf = false;
}
__device__ __forceinline__ void ac_finish_load(Ac& a, const EnvParams& P) {
    // the cached ground-speed components and cos(lat) are rebuilt with the very expressions of ac_kinematics, so a launch
    // continues bit for bit where the previous one stopped (n substeps in one launch == the same n split over launches)
    if (!P.gsv) {
        float s, co;
        __sincosf((a.hdg - 180.0f) * kDeg2Rad, &s, &co);
        a.gsn = -a.tas * co; a.gse = -a.tas * s;
    }
    a.coslat = __cosf((float)a.lat * kDeg2Rad);
}
__device__ __forceinline__ void ac_store(const Ac& a, const EnvParams& P, long long idx) {
    P.pos[idx] = make_double2(a.lat, a.lon);
    P.kin[idx] = make_float4(a.alt, a.tas, a.hdg, a.vs);
    P.cmd[idx] = make_float4(a.selspd, a.selalt, a.selvs, a.aptrk);
    P.aux[idx] = make_float4(a.ax, a.curlegdir, a.cas, a.tgt);
    P.flags[idx] = a.flags;
    if (P.gsv) P.gsv[idx] = make_float2(a.gsn, a.gse);
    if (P.cd_enabled) {
        P.tcpamax[idx] = a.tcpamax;
        P.inconf[idx] = a.inconf ? 1 : 0;
    }
}
__device__ __forceinline__ void env_load(EnvS& s, const EnvParams& P, long long e) {
    const double* d = P.ef64 + e * BSG_F64_COUNT;
    const float* f = P.ef32 + e * BSG_F32_COUNT;
    const int32_t* i = P.ei32 + e * BSG_I32_COUNT;
    s.wpt_lat = d[BSG_F64_WPT_LAT]; s.wpt_lon = d[BSG_F64_WPT_LON]; s.target_alt = d[BSG_F64_TARGET_ALT];
    s.poly_area = d[BSG_F64_POLY_AREA];
    s.total_reward = f[BSG_F32_TOTAL_REWARD]; s.drift_sum = f[BSG_F32_DRIFT_SUM]; s.final_alt = f[BSG_F32_FINAL_ALT];
    s.last_wdist = f[BSG_F32_LAST_WDIST]; s.last_drift = f[BSG_F32_LAST_DRIFT]; s.step_reward = 0.0f; s.step_done = 0;
    s.step = i[BSG_I32_STEP]; s.episode = i[BSG_I32_EPISODE]; s.simk = i[BSG_I32_SIMK];
    s.wpt_reach = i[BSG_I32_WPT_REACH]; s.drift_n = i[BSG_I32_DRIFT_N]; s.intrusions = i[BSG_I32_INTRUSIONS];
    s.num_ac = i[BSG_I32_NUM_AC]; s.nvert = i[BSG_I32_NVERT]; s.needs_reset = i[BSG_I32_NEEDS_RESET];
    s.faf = i[BSG_I32_FAF]; s.nconf = i[BSG_I32_NCONF]; s.nlos = i[BSG_I32_NLOS]; s.rflags = i[BSG_I32_RESET_FLAGS];
}
// the few fields the substep loop needs; the rest is fetched after the loop to keep registers free
__device__ __forceinline__ void env_load_pre(EnvS& s, const EnvParams& P, long long e) {
    const int32_t* i = P.ei32 + e * BSG_I32_COUNT;
    s.episode = i[BSG_I32_EPISODE]; s.simk = i[BSG_I32_SIMK]; s.num_ac = i[BSG_I32_NUM_AC];
    s.needs_reset = i[BSG_I32_NEEDS_RESET]; s.nconf = i[BSG_I32_NCONF]; s.nlos = i[BSG_I32_NLOS];
    s.nvert = i[BSG_I32_NVERT]; s.rflags = i[BSG_I32_RESET_FLAGS];
    s.wpt_lat = 0.0; s.wpt_lon = 0.0; s.target_alt = 0.0; s.poly_area = 0.0;
    s.total_reward = 0.0f; s.drift_sum = 0.0f; s.final_alt = 0.0f; s.last_wdist = 0.0f; s.last_drift = 0.0f;
    s.step_reward = 0.0f; s.step_done = 0;
    s.step = 0; s.wpt_reach = 0; s.drift_n = 0; s.intrusions = 0; s.faf = 0;
}
__device__ __forceinline__ void env_load_post(EnvS& s, const EnvParams& P, long long e) {
    const double* d = P.ef64 + e * BSG_F64_COUNT;
    const float* f = P.ef32 + e * BSG_F32_COUNT;
    const int32_t* i = P.ei32 + e * BSG_I32_COUNT;
    s.wpt_lat = d[BSG_F64_WPT_LAT]; s.wpt_lon = d[BSG_F64_WPT_LON]; s.target_alt = d[BSG_F64_TARGET_ALT];
    s.poly_area = d[BSG_F64_POLY_AREA];
    s.total_reward = f[BSG_F32_TOTAL_REWARD]; s.drift_sum = f[BSG_F32_DRIFT_SUM]; s.final_alt = f[BSG_F32_FINAL_ALT];
    s.last_wdist = f[BSG_F32_LAST_WDIST]; s.last_drift = f[BSG_F32_LAST_DRIFT];
    s.step = i[BSG_I32_STEP]; s.wpt_reach = i[BSG_I32_WPT_REACH]; s.drift_n = i[BSG_I32_DRIFT_N];
    s.intrusions = i[BSG_I32_INTRUSIONS]; s.faf = i[BSG_I32_FAF];
}
__device__ __forceinline__ void env_store_pre(const EnvS& s, const EnvParams& P, long long e) {
    int32_t* i = P.ei32 + e * BSG_I32_COUNT;
    i[BSG_I32_SIMK] = s.simk; i[BSG_I32_NCONF] = s.nconf; i[BSG_I32_NLOS] = s.nlos;
}
__device__ __forceinline__ void env_store(const EnvS& s, const EnvParams& P, long long e) {
    double* d = P.ef64 + e * BSG_F64_COUNT;
    float* f = P.ef32 + e * BSG_F32_COUNT;
    int32_t* i = P.ei32 + e * BSG_I32_COUNT;
    d[BSG_F64_WPT_LAT] = s.wpt_lat; d[BSG_F64_WPT_LON] = s.wpt_lon; d[BSG_F64_TARGET_ALT] = s.target_alt;
    d[BSG_F64_POLY_AREA] = s.poly_area;
    f[BSG_F32_TOTAL_REWARD] = s.total_reward; f[BSG_F32_DRIFT_SUM] = s.drift_sum; f[BSG_F32_FINAL_ALT] = s.final_alt;
    f[BSG_F32_LAST_WDIST] = s.last_wdist; f[BSG_F32_LAST_DRIFT] = s.last_drift;
    i[BSG_I32_STEP] = s.step; i[BSG_I32_EPISODE] = s.episode; i[BSG_I32_SIMK] = s.simk;
    i[BSG_I32_WPT_REACH] = s.wpt_reach; i[BSG_I32_DRIFT_N] = s.drift_n; i[BSG_I32_INTRUSIONS] = s.intrusions;
    i[BSG_I32_NUM_AC] = s.num_ac; i[BSG_I32_NVERT] = s.nvert; i[BSG_I32_NEEDS_RESET] = s.needs_reset;
    i[BSG_I32_FAF] = s.faf; i[BSG_I32_NCONF] = s.nconf; i[BSG_I32_NLOS] = s.nlos; i[BSG_I32_RESET_FLAGS] = s.rflags;
}

// ====================================================================================================
// K1: one simulator substep of one aircraft (Traffic.update minus ASAS).  oracle/traffic.py::update
// ====================================================================================================

// Everything in a substep that depends only on (alt, vs, selspd, selalt): ISA state, the autopilot's TAS
// target, flight phase and the performance-limited commands.  In level flight with a constant speed
// command these inputs do not change from substep to substep, so the result is cached and recomputed
// only when alt or vs moved (bit-identical inputs => identical outputs; selspd / selalt change only
// between env steps).  This removes 7 of the 9 pow-type evaluations from the steady-state substep.
struct Targets {
    Atmos at;               // atmosphere at the aircraft altitude
    float allow_tas, allow_h, amax, inv_amax;
    float k_alt, k_vs;      // inputs the cache was computed for
    int ph;
};

// `cached`: a.tgt holds allow_tas for exactly these inputs (env_kernel's targets cache): only the cheap parts are redone;
// ATMOS: the caller needs T.at afterwards either way.
template <bool ATMOS>
__device__ __forceinline__ void compute_targets(const Ac& a, const EnvParams& P, Targets& T, const bool cached) {
    const bsg_perf& pf = P.perf;
    T.k_alt = a.alt; T.k_vs = a.vs;
    if (ATMOS || !cached) T.at = vatmos(a.alt);
    else { T.at.p = 0.0f; T.at.rho = 0.0f; T.at.T = 0.0f; }
    // ---- perfoap.update: phase.get (later assignments overwrite earlier ones)
    float alt_ft = a.alt * (1.0f / kFt), roc = a.vs * (1.0f / kFpm);
    int ph = PH_NA;
    if (alt_ft <= 75.0f) ph = PH_GD;
    if (alt_ft >= 75.0f && alt_ft <= 1000.0f && roc >= 150.0f) ph = PH_IC;
    if (alt_ft >= 75.0f && alt_ft <= 1000.0f && roc <= -150.0f) ph = PH_AP;
    if (alt_ft >= 1000.0f && roc >= 150.0f) ph = PH_CL;
    if (alt_ft >= 1000.0f && roc <= -150.0f) ph = PH_DE;
    if (alt_ft >= 10000.0f && roc <= 150.0f && roc >= -150.0f) ph = PH_CR;
    T.ph = ph;
    float vmin = pf.vminer, vmax = pf.vmaxer;
    if (ph == PH_AP) { vmin = pf.vminap; vmax = pf.vmaxap; }
    if (ph == PH_GD) { vmin = 0.0f; vmax = pf.vmaxic; }
    T.amax = (ph == PH_GD) ? pf.axmax_gd : pf.axmax_air;
    T.inv_amax = (ph == PH_GD) ? P.inv_axmax_gd : P.inv_axmax_air;       // (1 / amax, evaluated on the host)
    // ---- perfoap.limits (CAS round trip evaluated at the allowed commanded altitude)
    T.allow_h = a.selalt > pf.hmax ? pf.hmax : a.selalt;
    if (cached) { T.allow_tas = a.tgt; return; }
    const bool level = T.allow_h == a.alt;
    Atmos ah = level ? T.at : vatmos(T.allow_h);
    float allow_tas = 0.0f, cas_c = a.selspd;
    bool convert = true;
    if (level && fabsf(a.selspd) >= 1.0f) {
        // a CAS command held at the commanded altitude: vtas2cas(vcas2tas(selspd)) is selspd itself, so the clamp applies
        // to the command and ONE CAS -> TAS conversion is left (same bits as the general path, minus 4 pow's)
        if (cas_c < vmin) cas_c = vmin;
        if (cas_c > vmax) cas_c = vmax;
    } else {
        float ap_tas = casormach2tas(a.selspd, T.at);      // Autopilot.update: ap.tas = vcasormach2tas(selspd, alt)
        float intent_cas = tas2cas(ap_tas, ah);
        allow_tas = ap_tas;                             // vcas2tas(vtas2cas(x)) == x when not clamped
        convert = false;
        if (intent_cas < vmin) { cas_c = vmin; convert = true; }
        if (intent_cas > vmax) { cas_c = vmax; convert = true; }
    }
    if (convert) allow_tas = cas2tas(cas_c, ah);
    float snd = vsound(ah);
    if (allow_tas > pf.mmo * snd) allow_tas = pf.mmo * snd;
    T.allow_tas = allow_tas;
}

template <int ENV>
__device__ __forceinline__ void ac_autopilot(Ac& a, const EnvParams& P, bool fms_ready) {
    if (ENV == BSG_ENV_MERGE) {
        if (a.flags & kFlLnav) {         // Autopilot.update LNAV + update_fms (2-waypoint route FIX -> RWY)
            double wlat, wlon;
            int iwp = (int)(a.flags >> kFlWpShift);
            if (iwp == 0) { wlat = P.fix_lat; wlon = P.fix_lon; } else { wlat = kRwyLat; wlon = kRwyLon; }
            float qdr, dist;
            qdrdist_wgs(a.lat, a.lon, wlat, wlon, qdr, dist, fms_ready);
            if (fms_ready) {
                // ActiveWaypoint.reached: next_qdr is -999 for both legs of this route => turndist = 0
                bool close2wp = dist / fmaxf(0.0001f, fabsf(ac_gs(a, P))) < 4.0f;
                bool tooclose = close2wp && fabsf(degto180(mod360(ac_trk(a, P)) - mod360(qdr))) > 90.0f;
                bool passed = fabsf(degto180(qdr - a.curlegdir)) > 90.0f;
                if (tooclose || passed) {
                    if ((a.flags & kFlLastWp) || iwp >= 1) {
                        a.flags &= ~kFlLnav;
                    } else {
                        a.flags = (a.flags & 0xffu) | (1u << kFlWpShift) | kFlLastWp;
                        qdrdist_wgs(a.lat, a.lon, kRwyLat, kRwyLon, qdr, dist);
                        a.curlegdir = qdr;
                    }
                }
            }
            if (a.flags & kFlLnav) a.aptrk = mod360(qdr);
        }
    }
}

// EXT (single-airspace traffic, traf_airspace.cu): the commanded track and vertical speed come from the caller -- VNAV or
// the ASAS resolution may be in command (APorASAS.update) -- instead of the select modes; the env kernels never set it.
template <bool WIND, bool EXT = false>
__device__ __forceinline__ void ac_kinematics(Ac& a, const EnvParams& P, const Targets& T, const float ext_trk = 0.0f,
                                              const float ext_vs = 0.0f) {
    const float dt = P.simdt;
    const bsg_perf& pf = P.perf;
    // ---- Autopilot select modes + APorASAS.update (resolution off)
    float selvs_eff = fabsf(a.selvs) > 0.1f ? a.selvs : kVsDef;
    float p_vs = fabsf(selvs_eff);
    float p_hdg = mod360(a.aptrk);
    if (EXT) { p_vs = fabsf(ext_vs); p_hdg = mod360(ext_trk); }
    float wn = 0.0f, we = 0.0f;
    if (WIND) {
        // APorASAS.update with wind: the heading that makes good the commanded track (crab angle), from the
        // wind at the aircraft's position before this substep's update_pos
        wind_at(P, a.lat, a.lon, a.alt, wn, we);
        const float vw = sqrtf(fmaf(wn, wn, we * we));
        const float drift = a.aptrk * kDeg2Rad - atan2f(we, wn);
        const float steer = asinf(fminf(1.0f, fmaxf(-1.0f, vw * sinf(drift) / fmaxf(0.001f, a.tas))));
        p_hdg = mod360(a.aptrk + kRad2Deg * steer);
        if (!(a.alt > 50.0f * kFt)) { wn = 0.0f; we = 0.0f; }       // update_groundspeed: wind only when airborne
    }
    const float amax = T.amax, allow_tas = T.allow_tas, allow_h = T.allow_h;
    float vs_max_acc = (1.0f - a.ax * T.inv_amax) * pf.vsmax;
    float allow_vs = p_vs;
    if (p_vs > 0.0f && p_vs > pf.vsmax) allow_vs = vs_max_acc;
    if (p_vs < 0.0f && p_vs < pf.vsmin) allow_vs = vs_max_acc;
    if (T.ph == PH_GD && a.tas < pf.vminto) allow_vs = 0.0f;
    // ---- update_airspeed
    float dspd = allow_tas - a.tas;
    bool need_ax = fabsf(dspd) > fabsf(dt * amax);
    a.ax = need_ax ? copysignf(amax, dspd) : 0.0f;
    a.tas = need_ax ? a.tas + a.ax * dt : allow_tas;
    float turnrate = (kRad2Deg * (kG0 * kTanBankDef)) * rcp_approx(fmaxf(a.tas, 0.01f));
    float delhdg = degto180(p_hdg - a.hdg);
    bool swhdgsel = fabsf(delhdg) > fabsf(dt * turnrate);
    a.hdg = mod360(swhdgsel ? a.hdg + copysignf(dt * turnrate, delhdg) : p_hdg);
    float delta_alt = allow_h - a.alt;
    bool swaltsel = fabsf(delta_alt) > 1.05f * fmaxf(fabsf(dt * allow_vs), fabsf(dt * a.vs));
    float target_vs = swaltsel ? copysignf(fabsf(allow_vs), delta_alt) : 0.0f;
    float delta_vs = target_vs - a.vs;
    bool need_az = fabsf(delta_vs) > kAzMax;
    a.vs = need_az ? a.vs + copysignf(kAzMax, delta_vs) * dt : target_vs;
    if (!isfinite(a.vs)) a.vs = 0.0f;
    // ---- update_groundspeed (no wind: gs = tas, trk = hdg; WIND: + the wind vector when above 50 ft)
    // hdg is in [0, 360): evaluate at hdg - 180 in [-pi, pi) where the MUFU sin/cos are accurate to ~5e-7,
    // and flip the signs (sin(x + pi) = -sin x, cos(x + pi) = -cos x)
    float sh, ch;
    __sincosf((a.hdg - 180.0f) * kDeg2Rad, &sh, &ch);
    a.gsn = -a.tas * ch; a.gse = -a.tas * sh;
    if (WIND) { a.gsn += wn; a.gse += we; }
    // ---- update_pos (lat/lon accumulate in float64)
    a.alt = swaltsel ? a.alt + a.vs * dt : allow_h;
    a.lat += (double)(kRad2Deg * (dt * a.gsn * (1.0f / kRearth)));
    a.coslat = __cosf((float)a.lat * kDeg2Rad);          // |lat| <= 90 deg: MUFU.COS is accurate to ~3e-7 here
    a.lon += (double)(kRad2Deg * (dt * a.gse * rcp_approx(a.coslat) * (1.0f / kRearth)));
}

// ====================================================================================================
// K3: in-group all-pairs CD in two phases.
//   Hot phase: three conditions every conflict or LoS needs, none of which takes a division:
//     dcpa < R                 |d x w| < R |w|
//     not past the zone        d . w < R |w|       (moving apart and more than R beyond the closest point: touthor < 0,
//                                                   and dist >= d . w / |w| > R)
//     zone within reach        dist < R + |w| dtlook   (the distance shrinks by at most |w| per second, so tinhor >= dtlook
//                                                   otherwise; this also settles the co-moving pairs whose |w|^2 upstream
//                                                   clamps to 1e-6: they can only be flagged when dist < R + 0.3 m)
//   each inflated by 2e-4, so the filter is a superset of what the exact routine accepts (a few % of the pairs of a
//   HorizontalCR-20 env pass early in an episode, almost none later).
//     (A) pairs with slot 0 -- the only aircraft the agent steers, in every env of the reference -- are filtered
//         every substep, one pair per lane.
//     (B) pairs among the other aircraft (a ring of m = n - 1 members; lane r tests the offsets 1 .. m/2, two per
//         iteration in packed f32x2, records staged as a structure of arrays written twice, m apart, so that
//         (r + k) mod m is a plain offset) are filtered when the env step starts and again only after one of them
//         moved its ground-speed vector by more than kCdVelTol.  With w(t) = w0 + eps(t), |eps| <= dw,
//         d x w and d . w - t |w0|^2 stay within dw (|d0| + 2 t |w0| + t dw) of their values at the filter pass, plus
//         the flat-earth terms -- cos(mean lat) and the longitude rate drift as the pair moves in latitude -- which
//         change dcpa by at most  kappa (|dx| + |dy| + d0),  kappa = 1.5 T vmax tan(lat_max) / Re,  d0 = (4 vmax + 1) T,
//         over the T seconds left in the env step.  The (B) pass tests with |w0| + dw for |w|, R + kappa (...) for R,
//         dtlook + T for dtlook and adds dw (|dx| + |dy| + d0): its candidate list stays a superset for every remaining
//         substep and is kept in shared memory.  (HorizontalCR / SectorCR intruders fly straight: one pass per env step;
//         MergeEnv's follow a great-circle bearing that creeps by ~0.01 m/s per substep -- scripts/merge_vel_probe.py --
//         which kCdVelTol = 0.15 m/s covers for a whole env step; an aircraft turning at a waypoint forces a new pass.)
//   Exact phase, every substep: the candidates (i, j) sit in a per-group queue in shared memory ((B) entries first,
//   (A) entries appended), are spread over the lanes and evaluated by cd_pair_sym() -- the same routine as
//   evaluating every pair, so results are bit-identical -- with per-aircraft results scattered through
//   shared-memory atomics that only fire for conflicting pairs.
// ====================================================================================================
enum { HX = 0, HY = 1, HCH = 2, HSH = 3, HU = 4, HV = 5, kHotFields = 6 };
constexpr int kQueuePerThread = 16;      // queue entries per lane: (B) <= (G-1)(G-2)/2 plus (A) <= G-1 < 16 G for G <= 32
constexpr float kCdVelTol = 0.15f;       // [m/s] |du| + |dv| an aircraft may drift from the velocity of the kept (B) pass
constexpr float kCdAbsEps = 1.0f;        // [m^2/s] rounding slack of the |d x w|, d . w tests at |w| ~ 0

constexpr int kSmallPairs = 8 * 7 / 2;
// pair p (ordered by j, then i < j) -> (i, j); the first n(n-1)/2 entries cover exactly the aircraft < n
__device__ __forceinline__ void build_pair_table(uint16_t* s_pairs) {
    for (int p = threadIdx.x; p < kSmallPairs; p += blockDim.x) {
        int j = (int)((1.0f + sqrtf(1.0f + 8.0f * (float)p)) * 0.5f);
        while (j * (j - 1) / 2 > p) --j;
        while ((j + 1) * j / 2 <= p) ++j;
        int i = p - j * (j - 1) / 2;
        s_pairs[p] = (uint16_t)((i << 8) | j);
    }
}

__device__ __forceinline__ u64 abs2(u64 v) { return v & 0x7fffffff7fffffffULL; }
__device__ __forceinline__ u64 neg2(u64 v) { return v ^ 0x8000000080000000ULL; }

// Shared memory of ONE group (env): every array the in-group CD touches sits at a compile-time offset from one base
// address, so a thread needs a single address register (derived once from its index) for all of them.
template <int G>
struct __align__(16) GroupSmem {
    float4 rec[2 * G];                                       // CD records: (x, y, ch, sh), (u, v, alt, vs) per slot
    float hot[(G > 8) ? 2 * G * kHotFields : 4];            // (B) ring, structure of arrays written twice
    uint16_t queue[(G > 8) ? G * kQueuePerThread : 8];      // candidate pairs: (B) entries first, (A) entries appended
    int tmax[G];                                             // per-slot max tcpa of the slot's conflicts (float bits)
    int cnt, nb, np, pad;                                    // compaction cursor | kept (B) entries (-1: none) | list entries
};

// `horizon`: simulated seconds between this substep and the last one of the env step (what a kept (B) list must cover)
// `emit`: this is the last substep of the launch and the caller bound pair lists: the exact phase also appends every
// conflicting / LoS pair to the env's list (entry format in include/bsg.h), count left in S.np for the caller.
// `lane_moved`: this aircraft's ground-speed vector changed in the last kinematics update.  TOL (MergeEnv: LNAV bearings
// creep every substep) keeps a (B) list while every ring aircraft stays within kCdVelTol of the velocity the list was built
// with; otherwise the list is rebuilt as soon as any ring aircraft moved at all (the intruders of HorizontalCR / SectorCR
// never do).  Rebuilding more often never changes results: every list is a superset of what the exact phase accepts.
template <int G, bool TOL>
__device__ __forceinline__ void group_cd(GroupSmem<G>& S, const int lane_g, Ac& a, bool alive, int nac, const EnvParams& P, float horizon,
                                         const uint16_t* s_pairs, int& nconf_env, int& nlos_env, const bool emit, const int e,
                                         const bool lane_moved, const double lat_ref, const double lon_ref) {
    const int lane = threadIdx.x & 31;
    const int wbase = lane - lane_g;                  // first lane of this group in the warp
    // cos / sin of lat/2 from the cached cos(lat): half-angle identities (absolute error ~1e-7); sign of lat from its high word
    const float ch = sqrt_approx(fmaf(0.5f, a.coslat, 0.5f));
    const float sh = __int_as_float((__float_as_int(sqrt_approx(fmaxf(fmaf(-0.5f, a.coslat, 0.5f), 0.0f))) & 0x7fffffff) |
                                    (__double2hiint(a.lat) & 0x80000000));
    // metres of arc east / north of the env's reference point (the envs live within a few hundred km of it, far from the
    // antimeridian: no +-180 fold)
    // (the difference in float64, the scaling in float32: 2 cm at 300 km from the origin)
    const float x = (kRearth * kDeg2Rad) * (float)(a.lon - lon_ref), y = (kRearth * kDeg2Rad) * (float)(a.lat - lat_ref);
    S.rec[2 * lane_g] = make_float4(x, y, ch, sh);
    S.rec[2 * lane_g + 1] = make_float4(a.gse, a.gsn, a.alt, a.vs);
    S.tmax[lane_g] = 0;
    if (emit && lane_g == 0) S.np = 0;
    unsigned confmask = 0u;       // bit = warp lane of an aircraft that is in conflict (this lane's pairs only)
    int counts = 0;               // ordered conflict pairs (low half) / ordered LoS pairs (high half) found by this lane
    bool found = true;
    auto exact_pair = [&](int i, int j) {
        CdSym r = cd_pair_sym(S.rec[2 * i], S.rec[2 * i + 1], S.rec[2 * j], S.rec[2 * j + 1], P.R2, P.hpz, P.dtlook);
        counts += (r.conf_ij ? 1 : 0) + (r.conf_ji ? 1 : 0) + (r.los ? (2 << 16) : 0);
        confmask |= (r.conf_ij ? 1u << (wbase + i) : 0u) | (r.conf_ji ? 1u << (wbase + j) : 0u);
        if (r.conf_ij | r.conf_ji) {               // tcpamax = max over the row of tcpa * swconfl (>= 0)
            const int tb = __float_as_int(fmaxf(r.tcpa, 0.0f));
            if (r.conf_ij) atomicMax(&S.tmax[i], tb);
            if (r.conf_ji) atomicMax(&S.tmax[j], tb);
        }
        if (emit && (r.conf_ij | r.conf_ji | r.los)) {        // rare: the pair goes to the env's list
            const int k = atomicAdd(&S.np, 1);
            if (k < P.cd_pair_cap) {
                const long long o = (long long)e * P.cd_pair_cap + k;
                P.cd_pairs[o] = (uint32_t)i | ((uint32_t)j << 8) | (r.conf_ij ? (uint32_t)BSG_PAIR_CONF_IJ : 0u) |
                                (r.conf_ji ? (uint32_t)BSG_PAIR_CONF_JI : 0u) | (r.los ? (uint32_t)BSG_PAIR_LOS : 0u);
                if (P.cd_attr) {
                    float* q = P.cd_attr + o * BSG_PAIR_ATTR_COUNT;
                    q[BSG_PAIR_ATTR_QDR] = mod360(kRad2Deg * atan2f(r.dx, r.dy));
                    q[BSG_PAIR_ATTR_DIST] = sqrtf(r.dist2);
                    q[BSG_PAIR_ATTR_DCPA] = sqrtf(r.dcpa2);
                    q[BSG_PAIR_ATTR_TCPA] = r.tcpa;
                    q[BSG_PAIR_ATTR_TINCONF_IJ] = r.tin_ij;
                    q[BSG_PAIR_ATTR_TINCONF_JI] = r.tin_ji;
                }
            }
        }
    };
    if (G <= 8) {
        // small groups (<= 8 aircraft, <= 28 pairs): the filter + queue cost more than they save; the
        // unordered pairs are dealt to the lanes from a table (pair p -> lane p % G) and evaluated exactly
        __syncwarp(group_mask<G>());
        const int npairs = nac * (nac - 1) / 2;
        for (int p = lane_g; p < npairs; p += G) {
            const unsigned ij = s_pairs[p];
            exact_pair((int)(ij >> 8), (int)(ij & 0xffu));
        }
    } else {
    const unsigned gm = group_mask<G>();
    const int m = nac - 1, r = lane_g - 1;            // ring of the aircraft the agent does not steer
    const bool ring = lane_g >= 1 && lane_g < nac;
    const int kmax = m >> 1;
    float* hot = S.hot;                               // [field][2G] for this group
    uint16_t* queue = S.queue;
    const float Rh = P.rpz * 1.0002f, Lh = P.dtlook * 1.0002f;
    // ---- is the kept (B) list still good?  (hot[HU], hot[HV] hold the velocities it was computed from)
    int nb = S.nb;
    bool moved;
    if (TOL) moved = ring && (fabsf(a.gse - hot[HU * 2 * G + (lane_g - 1)]) + fabsf(a.gsn - hot[HV * 2 * G + (lane_g - 1)]) > kCdVelTol);
    else moved = ring && lane_moved;
    const bool eval_b = P.cd_enabled == 2 || nb < 0 || __any_sync(gm, moved);
    u64 KAP = 0, RR = 0, D0 = 0, DW = 0, LH = 0;
    if (eval_b) {
        if (ring) {
            float* w = hot + r;
            w[HX * 2 * G] = -x; w[HY * 2 * G] = y;  w[HCH * 2 * G] = ch;      // (x is stored negated: see crs below)
            w[HSH * 2 * G] = sh; w[HU * 2 * G] = a.gse; w[HV * 2 * G] = a.gsn;
            w += m;
            w[HX * 2 * G] = -x; w[HY * 2 * G] = y;  w[HCH * 2 * G] = ch;
            w[HSH * 2 * G] = sh; w[HU * 2 * G] = a.gse; w[HV * 2 * G] = a.gsn;
        }
        if (lane_g == 0) S.cnt = 0;
        // allowances for keeping the list over `horizon` seconds (see the header comment)
        float kap = 0.0f, d0 = 0.0f, dw = 0.0f;
        if (P.cd_enabled != 2 && horizon > 0.0f) {
            const bool in = lane_g < nac;
            const float spd = in ? sqrtf(fmaf(a.gse, a.gse, a.gsn * a.gsn)) : 0.0f;
            // tan |lat| from the cached cos(lat) (capped near the poles like tan(89 deg))
            const float cl = fmaxf(a.coslat, 0.0175f);
            const float tl = in ? sqrt_approx(fmaxf(fmaf(-cl, cl, 1.0f), 0.0f)) * rcp_approx(cl) * 1.0001f : 0.0f;
            const float vmax = __uint_as_float(__reduce_max_sync(gm, __float_as_uint(spd))) + kCdVelTol;
            const float tmax = __uint_as_float(__reduce_max_sync(gm, __float_as_uint(tl)));
            kap = 1.5f * horizon * vmax * tmax * (1.0f / kRearth);
            d0 = (4.0f * vmax + 1.0f) * horizon;
            dw = TOL ? 2.0f * kCdVelTol : 0.0f;              // (without TOL any change of velocity rebuilds the list)
        }
        KAP = pk2(kap, kap); RR = pk2(fmaf(kap, d0, Rh), fmaf(kap, d0, Rh)); D0 = pk2(d0, d0); DW = pk2(dw, dw);
        const float lh = P.cd_enabled != 2 ? Lh + horizon * 1.0002f : Lh;
        LH = pk2(lh, lh);
    }
    __syncwarp(gm);
    if (eval_b) {
        // ---- (B) hot phase ---------------------------------------------------------------------------
        unsigned cand = 0u;
        {
            const u64 pX = pk2(x, x), nY = pk2(-y, -y), CH = pk2(ch, ch), nSH = pk2(-sh, -sh);
            const u64 nU = pk2(-a.gse, -a.gse), nV = pk2(-a.gsn, -a.gsn);
            const u64 EPS = pk2(kCdAbsEps, kCdAbsEps);
            const float* q = hot + r + 1;
#pragma unroll 1
            for (int kk = 0; kk < kmax; kk += 2, q += 2) {        // offsets k = kk + 1 and kk + 2
                const u64 nX = pk2(q[HX * 2 * G], q[HX * 2 * G + 1]);
                const u64 Y = pk2(q[HY * 2 * G], q[HY * 2 * G + 1]);
                const u64 CHc = pk2(q[HCH * 2 * G], q[HCH * 2 * G + 1]);
                const u64 SHc = pk2(q[HSH * 2 * G], q[HSH * 2 * G + 1]);
                const u64 U = pk2(q[HU * 2 * G], q[HU * 2 * G + 1]);
                const u64 V = pk2(q[HV * 2 * G], q[HV * 2 * G + 1]);
                const u64 dy = add2(Y, nY);
                const u64 cav = fma2(SHc, nSH, mul2(CHc, CH));
                const u64 ndxl = add2(nX, pX);
                const u64 ndx = mul2(ndxl, cav);                      // -(x_j - x_i) cos(mean lat)
                const u64 du = add2(U, nU), dv = add2(V, nV);
                const u64 dv2 = fma2(du, du, mul2(dv, dv));
                const u64 crs = fma2(ndx, dv, mul2(dy, du));          // -(dx dv - dy du): only its magnitude is used
                const u64 dot = fma2(neg2(du), ndx, mul2(dv, dy));    // d . w (same rounding as cd_pair_sym's)
                float w0, w1;
                up2(dv2, w0, w1);
                const u64 W = add2(pk2(sqrt_approx(w0), sqrt_approx(w1)), DW);        // |w| + what it may still change by
                const u64 l1 = add2(abs2(ndxl), abs2(dy));                            // |dx| + |dy| >= separation
                const u64 rm = fma2(KAP, l1, RR);                                     // R + flat-earth allowance
                const u64 t0 = fma2(W, rm, fma2(add2(l1, D0), DW, EPS));              // bound on |d x w| and on d . w
                const u64 reach = fma2(W, LH, rm);                                    // zone entry before the look-ahead ends
                float c0, c1, d0, d1, a0, a1, s0, s1, f0, f1;
                up2(abs2(crs), c0, c1);
                up2(dot, d0, d1);
                up2(t0, a0, a1);
                up2(fma2(ndx, ndx, mul2(dy, dy)), s0, s1);
                up2(mul2(reach, reach), f0, f1);
                // kept: dcpa < R, not yet out of the zone for good (d . w < R |w|), and close enough to enter the zone
                // before the look-ahead runs out (dist < R + |w| (dtlook + horizon)) -- each with its allowance
                cand |= (((c0 < a0 && d0 < a0 && s0 < f0) ? 1u : 0u) | ((c1 < a1 && d1 < a1 && s1 < f1) ? 2u : 0u)) << kk;
            }
            // offsets 1 .. m/2 only; for even m the offset m/2 names each pair twice: the lower half keeps it
            unsigned valid = (1u << kmax) - 1u;
            if (!(m & 1) && r >= kmax) valid >>= 1;
            cand = ring ? (cand & valid) : 0u;
        }
        // ---- (B) compaction: (i, j) slot pairs into the group's queue (rare path: kept simple) ----------
        if (__any_sync(gm, cand != 0u)) {
            const int cnt = __popc(cand);
            int pos = 0;
            if (cnt) pos = atomicAdd(&S.cnt, cnt);
            uint16_t* qp = queue + pos;
#pragma unroll 1
            for (unsigned c = cand; c; c &= c - 1u) {
                int rj = r + __ffs(c);                            // offset k = (bit index) + 1
                rj = rj >= m ? rj - m : rj;
                *qp++ = (uint16_t)((lane_g << 8) | (rj + 1));
            }
            __syncwarp(gm);
            nb = S.cnt;
        } else {
            nb = 0;
        }
        if (lane_g == 0) S.nb = nb;
    }
    // ---- (A) pairs with slot 0, every substep ----------------------------------------------------------------
    int ncand;
    {
        const float4 A0 = S.rec[0], B0 = S.rec[1];
        const float cav = fmaf(-A0.w, sh, A0.z * ch);
        const float dx = (x - A0.x) * cav, dy = y - A0.y;
        const float du = a.gse - B0.x, dv = a.gsn - B0.y;
        const float dv2 = fmaf(du, du, dv * dv);
        const float crs = fmaf(dx, dv, -dy * du);
        const float dot = fmaf(du, dx, dv * dy);
        const float w = sqrt_approx(dv2);
        const float t0 = fmaf(w, Rh, kCdAbsEps), reach = fmaf(w, Lh, Rh);
        const bool pass = ring && fabsf(crs) < t0 && dot < t0 && fmaf(dx, dx, dy * dy) < reach * reach;
        const unsigned bm = (G >= 32) ? __ballot_sync(gm, pass) : ((__ballot_sync(gm, pass) >> wbase) & ((1u << (G & 31)) - 1u));
        if (pass) queue[nb + __popc(bm & ((1u << lane_g) - 1u))] = (uint16_t)lane_g;      // (i, j) = (0, lane_g)
        ncand = nb + __popc(bm);
        __syncwarp(gm);
    }
    // ---- exact phase -------------------------------------------------------------------------------
    for (int p = lane_g; p < ncand; p += G) {
        const unsigned en = queue[p];
        exact_pair((int)(en >> 8), (int)(en & 0xffu));
    }
    found = ncand > 0;
    }
    // one REDUX.OR over the group merges every lane's findings; each aircraft then reads its own bit
    if (found) {                                      // (group-uniform)
        confmask = __reduce_or_sync(group_mask<G>(), confmask);
        counts = (int)__reduce_add_sync(group_mask<G>(), (unsigned)counts);
    }
    a.inconf = alive && ((confmask >> lane) & 1u);
    a.tcpamax = __int_as_float(S.tmax[lane_g]);
    nconf_env = counts & 0xffff;
    nlos_env = counts >> 16;
    __syncwarp(group_mask<G>());
}

}  // namespace bsg
