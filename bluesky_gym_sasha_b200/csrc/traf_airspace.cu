// traf_airspace.cu -- one airspace of N aircraft with routes, VNAV and ASAS conflict resolution (SURVEY 8f-4).
//
// Per simulator substep the caller runs  traf_pack_kernel -> K2 (cd_tiled.cu, with pair lists) -> bsg_traf_substep, which
// first indexes K2's unordered conflict list by own aircraft (count, allocate, scatter: three small kernels, no sort) and
// then launches traf_substep_kernel.  The substep kernel owns one aircraft per thread and fuses what
// upstream spreads over Autopilot.update, ConflictResolution.update, APorASAS.update, perfoap.update / limits and
// Traffic.update_airspeed / groundspeed / pos (bluesky/traffic/{autopilot,route,aporasas,traffic}.py,
// asas/{resolution,mvp}.py, performance/openap/perfoap.py as restated in oracle/traffic_ext.py, which it is checked
// against).  An aircraft only ever WRITES its own records; everything it needs from other aircraft -- the intruders of
// its conflicts and of its resopairs -- it reads from the CD records of this substep, an immutable snapshot of the state
// the detection saw, so the update is in place and free of ordering effects.  An aircraft's conflicts sit in one
// contiguous run of the index and are visited in ascending intruder order: the MVP velocity changes are summed in
// upstream's order (confpairs is row-major), deterministically, whatever order K2 emitted them in.
//
// Bound: HBM.  Algorithmic bytes per aircraft-substep: the nine state records read and written (2 x 148 B) plus its
// 32 B CD record = 328 B; the route table is only touched at a waypoint switch.
#include <cuda_runtime.h>
#include <stdint.h>

#include "cd_record.cuh"
#include "env_kernels.cuh"

namespace bsg {

constexpr float kSteepness = 3000.0f * kFt / (10.0f * kNm);        // Autopilot.steepness

struct TrafParams {
    long long n, row0;          // row0: global index (in the CD records and pair lists) of this block's aircraft 0
    int W, reso, reso_mode, fms_ready;
    float simdt, rpz, hpz, dtlook, resofach, resofacv;
    bsg_perf perf;
    double lat0, lon0;
    double2* pos; float4* kin; float4* cmd; float4* aux; double2* actwp; float4* vn1; float4* vn2; float4* asas;
    uint32_t* flags; int32_t* partners;
    const double2* rt_pos; const float4* rt_con; const float* rt_dir; uint32_t* counters;
    const float* rec;
    const int2* pairs; const float* attr; const unsigned long long* npairs; long long cap;      // K2's conflict list
    const unsigned long long* nconf_all;     // conflicts in the whole airspace (== npairs unless the airspace is sharded)
    int* count; int* offs; int* len; int* total; int* seg;     // index of that list by own aircraft: rows seg[offs[i] .. offs[i] + len[i])
};

// registers of one aircraft beyond the kinematic state (struct Ac)
struct TrafAc {
    double wlat, wlon;
    float next_qdr, turndist;
    float nextaltco, xtoalt, actwp_vs, dist2vs;
    float actwp_spd, nextspd, spdcon, vnavvs;
    float asas_trk, asas_tas, asas_vs, asas_alt;
    float ap_alt;                 // Autopilot.alt of this substep (ComputeVNAV may dial it in)
    uint32_t f;                   // BSG_TF_*
};

// Autopilot.ComputeVNAV (swtod = swtoc = True, no RTA): once per leg.  dist2wp [m] to the active waypoint.
__device__ __forceinline__ void compute_vnav(Ac& a, TrafAc& x, const float toalt, const float xtoalt, const float dist2wp) {
    if (toalt < 0.0f || !(x.f & BSG_TF_VNAV)) { x.dist2vs = -999999.0f; return; }
    const float gs = a.tas;
    if (a.alt > toalt + 2.0f * kFt) {
        if (a.vs > 0.0001f) { x.vnavvs = 0.0f; x.ap_alt = a.alt; a.selalt = a.alt; }      // stop a climb first
        x.nextaltco = toalt; x.xtoalt = xtoalt;
        const float descdist = fabsf(a.alt - toalt) / kSteepness;
        x.dist2vs = descdist - xtoalt;
        if (dist2wp - 1.02f * x.turndist < x.dist2vs) {                                  // late: use what is left of the leg
            x.ap_alt = x.nextaltco;
            const float t2go = dist2wp / fmaxf(0.01f, gs);
            x.actwp_vs = (x.nextaltco - a.alt) / fmaxf(0.01f, t2go);
        } else if (xtoalt < descdist) {                                                  // top of descent on this leg
            x.actwp_vs = -kSteepness * (gs + (gs < 0.2f * a.tas ? a.tas : 0.0f));
        } else {
            x.actwp_vs = 0.0f;
        }
    } else if (a.alt < toalt - 10.0f * kFt) {                                            // climb as soon as possible
        if (a.vs < -0.0001f) { x.vnavvs = 0.0f; x.ap_alt = a.alt; a.selalt = a.alt; }
        x.nextaltco = toalt; x.xtoalt = xtoalt;
        x.ap_alt = x.nextaltco;
        x.dist2vs = 99999.0f;
        const float t2go = fmaxf(0.1f, dist2wp + xtoalt) / fmaxf(0.01f, gs);
        x.actwp_vs = fmaxf(kSteepness * gs, (x.nextaltco - a.alt) / t2go);
    } else {
        x.dist2vs = -999.0f;
    }
}

// Route.direct(): waypoint k of the aircraft's route becomes the active one (route activation, and the waypoint
// recovery after a resolved conflict)
__device__ __forceinline__ void route_direct(Ac& a, TrafAc& x, const TrafParams& P, const long long i, const int k) {
    const int nwp = (int)((x.f >> BSG_TF_NWP_SHIFT) & 0xffu);
    const long long o = i * P.W + k;
    const double2 wp = P.rt_pos[o];
    const float4 con = P.rt_con[o];                    // wpalt, wpspd, wptoalt, wpxtoalt
    x.f = (x.f & ~((0xffu << BSG_TF_IWP_SHIFT) | BSG_TF_LASTWP)) | ((uint32_t)k << BSG_TF_IWP_SHIFT) |
          (k == nwp - 1 ? (uint32_t)BSG_TF_LASTWP : 0u) | BSG_TF_LNAV;
    x.wlat = wp.x; x.wlon = wp.y;
    float q, d;
    qdrdist_wgs(a.lat, a.lon, wp.x, wp.y, q, d);
    a.curlegdir = q;
    x.next_qdr = P.rt_dir[o];
    x.turndist = 0.0f;
    x.nextspd = con.y > 0.0f ? con.y : -999.0f;
    if (con.x >= -0.01f) { x.nextaltco = con.x; x.xtoalt = 0.0f; }
    else { x.nextaltco = con.z; x.xtoalt = con.w; }
    compute_vnav(a, x, con.z, x.xtoalt, d);
}

__device__ __forceinline__ void traf_load(Ac& a, TrafAc& x, const TrafParams& P, const long long i) {
    const double2 p = P.pos[i], w = P.actwp[i];
    const float4 k = P.kin[i], c = P.cmd[i], u = P.aux[i], v1 = P.vn1[i], v2 = P.vn2[i], s = P.asas[i];
    a.lat = p.x; a.lon = p.y;
    a.alt = k.x; a.tas = k.y; a.hdg = k.z; a.vs = k.w;
    a.selspd = c.x; a.selalt = c.y; a.selvs = c.z; a.aptrk = c.w;
    a.ax = u.x; a.curlegdir = u.y; x.next_qdr = u.z; x.turndist = u.w;
    a.cas = 0.0f; a.tgt = 0.0f; a.flags = kFlAlive; a.gsn = 0.0f; a.gse = 0.0f; a.coslat = 1.0f; a.tcpamax = 0.0f; a.inconf = false;
    x.wlat = w.x; x.wlon = w.y;
    x.nextaltco = v1.x; x.xtoalt = v1.y; x.actwp_vs = v1.z; x.dist2vs = v1.w;
    x.actwp_spd = v2.x; x.nextspd = v2.y; x.spdcon = v2.z; x.vnavvs = v2.w;
    x.asas_trk = s.x; x.asas_tas = s.y; x.asas_vs = s.z; x.asas_alt = s.w;
    x.ap_alt = a.selalt;
    x.f = P.flags[i];
}
__device__ __forceinline__ void traf_store(const Ac& a, const TrafAc& x, const TrafParams& P, const long long i) {
    P.pos[i] = make_double2(a.lat, a.lon);
    P.actwp[i] = make_double2(x.wlat, x.wlon);
    P.kin[i] = make_float4(a.alt, a.tas, a.hdg, a.vs);
    P.cmd[i] = make_float4(a.selspd, a.selalt, a.selvs, a.aptrk);
    P.aux[i] = make_float4(a.ax, a.curlegdir, x.next_qdr, x.turndist);
    P.vn1[i] = make_float4(x.nextaltco, x.xtoalt, x.actwp_vs, x.dist2vs);
    P.vn2[i] = make_float4(x.actwp_spd, x.nextspd, x.spdcon, x.vnavvs);
    P.asas[i] = make_float4(x.asas_trk, x.asas_tas, x.asas_vs, x.asas_alt);
    P.flags[i] = x.f;
}

// CD record of aircraft i (inert for padding and dead slots).  The one record computation of both packs: a reordered
// record is bit for bit the aircraft-order record.
__device__ __forceinline__ void traf_record(const TrafParams& P, const long long i, float (&f)[BSG_CD_REC_FIELDS]) {
    cd_rec_inert(f);
    if (i < P.n && (P.flags[i] & BSG_TF_ALIVE)) {
        const double2 p = P.pos[i];
        const float4 k = P.kin[i];
        cd_rec_position(f, p.x, p.y, P.lat0, P.lon0);
        float sh, ch;
        sincosf(k.z * kDeg2Rad, &sh, &ch);
        f[FU] = k.y * sh; f[FV] = k.y * ch; f[FALT] = k.x; f[FVS] = k.w;
    }
}

__global__ void traf_pack_kernel(const TrafParams P, float* __restrict__ rec, const long long n_pad) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_pad) return;
    float f[BSG_CD_REC_FIELDS];
    traf_record(P, i, f);
    cd_rec_store(rec, i, f);
}

// gather: record slot k <- aircraft perm[k] (slots past n: inert), and the same record into aircraft order when rec != NULL
__global__ void __launch_bounds__(256) traf_pack_ordered_kernel(const TrafParams P, const int32_t* __restrict__ perm,
                                                                float* __restrict__ rec_ordered, float* __restrict__ rec,
                                                                const long long n_pad) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n_pad) return;
    const long long i = k < P.n ? (long long)perm[k] : k;
    float f[BSG_CD_REC_FIELDS];
    traf_record(P, i, f);
    cd_rec_store(rec_ordered, k, f);
    if (rec) cd_rec_store(rec, i, f);
}

__global__ void traf_activate_kernel(const TrafParams P) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.n) return;
    const uint32_t f = P.flags[i];
    if (!(f & BSG_TF_ALIVE) || !(f & BSG_TF_ACTIVATE)) return;
    Ac a;
    TrafAc x;
    traf_load(a, x, P, i);
    x.f &= ~(uint32_t)BSG_TF_ACTIVATE;
    route_direct(a, x, P, i, 0);
    traf_store(a, x, P, i);
}

// MVP.MVP(): velocity change of the own aircraft that moves the closest point of approach with one intruder to the edge
// of the (enlarged) zone.  drel / vrel: intruder minus own.
__device__ __forceinline__ void mvp_pair(const TrafParams& P, const float qdr, const float dist, const float tcpa, const float tlos,
                                         const float dalt, const float du, const float dv, const float dvs,
                                         float& dv1, float& dv2, float& dv3, float& tsolv) {
    float sq, cq;
    sincosf(qdr * kDeg2Rad, &sq, &cq);
    const float drx = sq * dist, dry = cq * dist;
    float cx = fmaf(du, tcpa, drx), cy = fmaf(dv, tcpa, dry);
    float dabsh = sqrtf(fmaf(cx, cx, cy * cy));
    const float rh = P.rpz * P.resofach;
    const float ih = rh - dabsh;
    if (dabsh <= 10.0f) {                                  // head-on: push sideways
        dabsh = 10.0f;
        cx = dry / dist * dabsh;
        cy = -drx / dist * dabsh;
    }
    const float at = fabsf(tcpa);
    if (rh < dist && dabsh < dist) {                       // outside the zone: aim at the tangent
        const float erratum = cosf(asinf(rh / dist) - asinf(dabsh / dist));
        const float g = (rh / erratum - dabsh) / (at * dabsh);
        dv1 = g * cx; dv2 = g * cy;
    } else {
        const float g = ih / (at * dabsh);
        dv1 = g * cx; dv2 = g * cy;
    }
    const float hv = P.hpz * P.resofacv;
    const bool vmove = fabsf(dvs) > 0.0f;
    float iv = vmove ? hv : hv - fabsf(dalt);
    tsolv = vmove ? fabsf(dalt / dvs) : tlos;
    if (tsolv > P.dtlook) { tsolv = tlos; iv = hv; }
    dv3 = vmove ? (iv / tsolv) * (-dvs / fabsf(dvs)) : iv / tsolv;
}

// ---- index of K2's conflict list by own aircraft ---------------------------------------------------------------------
__global__ void traf_conf_count_kernel(const TrafParams P) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long ntot = P.npairs[0];
    const long long m = ntot < (unsigned long long)P.cap ? (long long)ntot : P.cap;
    if (k == 0) *P.total = 0;                          // (the allocation kernel runs after this one)
    if (k < m) atomicAdd(&P.count[P.pairs[k].x - P.row0], 1);
}
// every aircraft with conflicts reserves a contiguous run of the index: warp-aggregated (one atomicAdd per warp on the
// running total).  The runs come in no particular order -- nothing needs them ordered -- so no global scan is needed.
__global__ void traf_conf_alloc_kernel(const TrafParams P) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    const int c = i < P.n ? P.count[i] : 0;
    int incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl += v;
    }
    const int wsum = __shfl_sync(0xffffffffu, incl, 31);
    int base = 0;
    if (lane == 31 && wsum > 0) base = atomicAdd(P.total, wsum);
    base = __shfl_sync(0xffffffffu, base, 31);
    if (i < P.n) { P.offs[i] = base + incl - c; P.len[i] = c; }
}
// rows of the list into their aircraft's run; the counters count back down to zero, ready for the next substep
__global__ void traf_conf_scatter_kernel(const TrafParams P) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned long long ntot = P.npairs[0];
    const long long m = ntot < (unsigned long long)P.cap ? (long long)ntot : P.cap;
    if (k < m) {
        const long long i = P.pairs[k].x - P.row0;
        P.seg[P.offs[i] + atomicSub(&P.count[i], 1) - 1] = (int)k;
    }
}

// 6 CTAs per SM (<= 85 registers, no spills): 61 vs 68 us at 2^20 aircraft, 14.3 vs 16.4 us at 100k
__global__ void __launch_bounds__(128, 6) traf_substep_kernel(const TrafParams P) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P.n) return;
    if (!(P.flags[i] & BSG_TF_ALIVE)) return;
    Ac a;
    TrafAc x;
    traf_load(a, x, P, i);
    const bsg_perf& pf = P.perf;
    const float gs = a.tas, trk = a.hdg;                   // no wind
    int n_switch = 0;

    // ---- Autopilot.update: LNAV bearing / distance to the active waypoint, update_fms at its cadence ----------------
    float qdr, dist2wp;
    qdrdist_wgs(a.lat, a.lon, x.wlat, x.wlon, qdr, dist2wp);
    if (P.fms_ready) {
        const float nq = x.next_qdr < -900.0f ? qdr : x.next_qdr;
        const float turnrad = a.tas * a.tas / (fmaxf(0.01f, kTanBankDef) * kG0);
        x.turndist = fabsf(turnrad * tanf(kDeg2Rad * 0.5f * fabsf(degto180(mod360(qdr) - mod360(nq)))));
        const bool close2wp = dist2wp / fmaxf(0.0001f, fabsf(gs)) < 4.0f;
        const bool tooclose = close2wp && fabsf(degto180(mod360(trk) - mod360(qdr))) > 90.0f;
        const bool passed = fabsf(degto180(qdr - a.curlegdir)) > 90.0f;
        if ((x.f & BSG_TF_LNAV) && (tooclose || passed || dist2wp < x.turndist)) {
            x.actwp_spd = x.nextspd;                       // speeds are FROM-speeds: the passed waypoint's holds on the next leg
            x.spdcon = x.nextspd;
            const int nwp = (int)((x.f >> BSG_TF_NWP_SHIFT) & 0xffu);
            if (nwp == 0 || (x.f & BSG_TF_LASTWP)) {
                x.f &= ~(uint32_t)(BSG_TF_LNAV | BSG_TF_VNAV | BSG_TF_VNAVSPD);
            } else {                                       // Route.getnextwp
                const int k = (int)((x.f >> BSG_TF_IWP_SHIFT) & 0xffu) + 1;
                const long long o = i * P.W + k;
                const double2 wp = P.rt_pos[o];
                const float4 con = P.rt_con[o];
                x.f = (x.f & ~((0xffu << BSG_TF_IWP_SHIFT) | BSG_TF_LASTWP)) | ((uint32_t)k << BSG_TF_IWP_SHIFT) |
                      (k == nwp - 1 ? (uint32_t)BSG_TF_LASTWP : 0u);
                x.nextspd = con.y;
                x.xtoalt = con.w;
                x.next_qdr = P.rt_dir[o];
                x.wlat = wp.x; x.wlon = wp.y;
                qdrdist_wgs(a.lat, a.lon, wp.x, wp.y, qdr, dist2wp);
                a.curlegdir = qdr;
                if (con.x >= -0.01f) { x.nextaltco = con.x; x.xtoalt = 0.0f; }
                else x.nextaltco = con.z;
                if ((x.f & BSG_TF_VNAVSPD) && x.actwp_spd >= 0.0f) a.selspd = x.actwp_spd;
                const float lnq = x.next_qdr < -900.0f ? qdr : x.next_qdr;
                x.turndist = fabsf(turnrad * tanf(kDeg2Rad * 0.5f * fabsf(degto180(mod360(qdr) - mod360(lnq)))));
                compute_vnav(a, x, con.z, x.xtoalt, dist2wp);
                ++n_switch;
            }
        }
    }
    // ---- continuous VNAV / speed guidance ---------------------------------------------------------------------------
    const bool lnav = (x.f & BSG_TF_LNAV) != 0, vnav = (x.f & BSG_TF_VNAV) != 0, vnavspd = (x.f & BSG_TF_VNAVSPD) != 0;
    const bool startdescorclimb = (x.nextaltco >= -0.1f) &&
        ((a.alt > x.nextaltco && dist2wp < x.dist2vs + x.turndist) || a.alt < x.nextaltco);
    const bool swvnavvs = vnav && (lnav ? startdescorclimb : dist2wp <= fmaxf(0.1f * kNm, x.turndist));
    if (swvnavvs) x.vnavvs = x.actwp_vs;
    const float selvs_eff = fabsf(a.selvs) > 0.1f ? a.selvs : kVsDef;
    const float ap_vs = swvnavvs ? x.vnavvs : selvs_eff;
    x.ap_alt = swvnavvs ? x.nextaltco : a.selalt;
    if (swvnavvs) a.selalt = x.nextaltco;
    if (lnav) a.aptrk = mod360(qdr);
    const Atmos at = vatmos(a.alt);
    {
        const float nexttas = casormach2tas(x.nextspd, at);
        const float axm = (x.f & BSG_TF_PH_GD) ? pf.axmax_gd : pf.axmax_air;       // perf.axmax of the last perf.update
        const float dxspd = 0.5f * fabsf(nexttas * nexttas - a.tas * a.tas) / fmaxf(0.001f, fabsf(axm));
        const bool usenext = dist2wp < dxspd && x.nextspd > -990.0f && vnavspd && vnav && lnav;
        a.selspd = usenext ? x.nextspd : ((x.spdcon >= 0.0f && vnavspd) ? x.actwp_spd : a.selspd);
    }
    const float ap_tas = casormach2tas(a.selspd, at);

    // ---- ASAS: ConflictResolution.update = MVP.resolve (when the detection found any conflict) + resumenav -----------
    if (P.reso) {
        const long long ig = P.row0 + i;                   // this aircraft in the records of the whole airspace
        const float own_u = cd_rec_at(P.rec, ig, FU), own_v = cd_rec_at(P.rec, ig, FV);
        const float own_alt = cd_rec_at(P.rec, ig, FALT), own_vs = cd_rec_at(P.rec, ig, FVS);
        const unsigned long long ntot = P.nconf_all[0];
        const int k0 = P.offs[i], k1 = k0 + P.len[i];
        // the aircraft's conflicts in ascending intruder order (its run of the index is unordered; runs are short)
        auto next_conflict = [&](int last, int& row) {
            int best = 0x7fffffff;
            for (int k = k0; k < k1; ++k) {
                const int r = P.seg[k], j = P.pairs[r].y;
                if (j > last && j < best) { best = j; row = r; }
            }
            return best;
        };
        if (ntot > 0) {                                    // `if conf.confpairs:` -- resolve() rewrites every aircraft's commands
            float d1 = 0.0f, d2 = 0.0f, d3 = 0.0f, tsolv_min = 1e9f;
            int row = 0;
            for (int c = k0, j = -1; c < k1; ++c) {
                j = next_conflict(j, row);
                const float* q = P.attr + (long long)row * BSG_CD_ATTR_COUNT;
                float e1, e2, e3, ts;
                mvp_pair(P, q[BSG_CD_ATTR_QDR], q[BSG_CD_ATTR_DIST], q[BSG_CD_ATTR_TCPA], q[BSG_CD_ATTR_TINCONF],
                         cd_rec_at(P.rec, j, FALT) - own_alt, cd_rec_at(P.rec, j, FU) - own_u, cd_rec_at(P.rec, j, FV) - own_v,
                         cd_rec_at(P.rec, j, FVS) - own_vs, e1, e2, e3, ts);
                tsolv_min = fminf(tsolv_min, ts);
                d1 -= e1; d2 -= e2; d3 -= 0.5f * e3;      // cooperative: half the vertical part each
                if (x.f & BSG_TF_RESOOFF) { d1 = 0.0f; d2 = 0.0f; d3 = 0.0f; }
            }
            const float nu = own_u + d1, nv = own_v + d2, nw = own_vs + d3;
            const float newtrk = mod360(kRad2Deg * atan2f(nu, nv));
            const float newgs = sqrtf(fmaf(nu, nu, nv * nv));
            const float newvs = P.reso_mode == 1 ? own_vs : nw;
            float vmin = pf.vminer, vmax = pf.vmaxer;      // perf.vmin / vmax of the last perf.update
            if (x.f & BSG_TF_PH_AP) { vmin = pf.vminap; vmax = pf.vmaxap; }
            if (x.f & BSG_TF_PH_GD) { vmin = 0.0f; vmax = pf.vmaxic; }
            x.asas_tas = fmaxf(vmin, fminf(vmax, newgs));
            const float vsc = fmaxf(pf.vsmin, fminf(pf.vsmax, newvs));
            x.asas_trk = newtrk; x.asas_vs = vsc;
            const float alttemp = fmaf(vsc, tsolv_min, own_alt);
            const float sgn_alt = (float)((a.selalt > own_alt) - (a.selalt < own_alt));
            const float dvs_ = vsc - ap_vs * sgn_alt;
            const int signdvs = (dvs_ > 0.0f) - (dvs_ < 0.0f);
            const int signalt = (alttemp > a.selalt) - (alttemp < a.selalt);
            float altc = (signdvs == 0 || signdvs == signalt) ? alttemp : a.selalt;
            if (tsolv_min < P.dtlook && fabsf(d3) > 0.0f) altc = alttemp;
            x.asas_alt = P.reso_mode == 1 ? a.selalt : altc;
        }
        // resumenav: new conflicts join the aircraft's resopairs; each one stays until it is past CPA, out of horizontal
        // LoS and not bouncing; ASAS commands the aircraft while any is left
        int part[BSG_TRAF_PARTNERS];
        int4* pp = (int4*)(P.partners + i * BSG_TRAF_PARTNERS);
        {
            const int4 p0 = pp[0], p1 = pp[1];
            part[0] = p0.x; part[1] = p0.y; part[2] = p0.z; part[3] = p0.w;
            part[4] = p1.x; part[5] = p1.y; part[6] = p1.z; part[7] = p1.w;
        }
        int overflow = 0;
        for (int k = k0; k < k1; ++k) {
            const int j = P.pairs[P.seg[k]].y;
            bool have = false;
            int free_slot = -1;
#pragma unroll
            for (int s = BSG_TRAF_PARTNERS - 1; s >= 0; --s) {
                have |= part[s] == j;
                if (part[s] < 0) free_slot = s;
            }
            if (!have) {
                if (free_slot < 0) ++overflow;
                else {
#pragma unroll
                    for (int s = 0; s < BSG_TRAF_PARTNERS; ++s) if (s == free_slot) part[s] = j;
                }
            }
        }
        bool any_pair = false, active = false;
        const float own_x = cd_rec_at(P.rec, ig, FX), own_y = cd_rec_at(P.rec, ig, FY);
        const float own_ch = cd_rec_at(P.rec, ig, FCH), own_sh = cd_rec_at(P.rec, ig, FSH);
        const float own_trk = mod360(kRad2Deg * atan2f(own_u, own_v));
#pragma unroll
        for (int s = 0; s < BSG_TRAF_PARTNERS; ++s) {
            const int j = part[s];
            if (j < 0) continue;
            any_pair = true;
            const float cav = fmaf(-own_sh, cd_rec_at(P.rec, j, FSH), own_ch * cd_rec_at(P.rec, j, FCH));
            const float dx = (cd_rec_at(P.rec, j, FX) - own_x) * cav, dy = cd_rec_at(P.rec, j, FY) - own_y;
            const float ju = cd_rec_at(P.rec, j, FU), jv = cd_rec_at(P.rec, j, FV);
            const bool past_cpa = fmaf(dx, ju - own_u, dy * (jv - own_v)) > 0.0f;
            const float hdist = sqrtf(fmaf(dx, dx, dy * dy));
            const bool hor_los = hdist < P.rpz;
            const float jtrk = mod360(kRad2Deg * atan2f(ju, jv));
            const bool bouncing = fabsf(own_trk - jtrk) < 30.0f && hdist < P.rpz * P.resofach;
            if (!past_cpa || hor_los || bouncing) active = true;
            else part[s] = -1;
        }
        pp[0] = make_int4(part[0], part[1], part[2], part[3]);
        pp[1] = make_int4(part[4], part[5], part[6], part[7]);
        if (overflow) atomicAdd(&P.counters[BSG_TRAF_CTR_OVERFLOW], (uint32_t)overflow);
        if (any_pair) {
            x.f = active ? (x.f | BSG_TF_ASAS) : (x.f & ~(uint32_t)BSG_TF_ASAS);
            if (!active && ((x.f >> BSG_TF_NWP_SHIFT) & 0xffu) != 0u)             // waypoint recovery
                route_direct(a, x, P, i, (int)((x.f >> BSG_TF_IWP_SHIFT) & 0xffu));
        }
    }

    // ---- APorASAS.update: ASAS commands override the autopilot's while active ---------------------------------------
    const bool act = (x.f & BSG_TF_ASAS) != 0;
    const float p_trk = act ? x.asas_trk : a.aptrk;
    const float p_tas = act ? x.asas_tas : ap_tas;
    const float p_alt = act ? x.asas_alt : x.ap_alt;
    const float p_vs = fabsf(act ? x.asas_vs : ap_vs);
    // ---- perfoap.update (phase, axmax) + limits ---------------------------------------------------------------------
    Targets T;
    {
        const float alt_ft = a.alt * (1.0f / kFt), roc = a.vs * (1.0f / kFpm);
        int ph = PH_NA;
        if (alt_ft <= 75.0f) ph = PH_GD;
        if (alt_ft >= 75.0f && alt_ft <= 1000.0f && roc >= 150.0f) ph = PH_IC;
        if (alt_ft >= 75.0f && alt_ft <= 1000.0f && roc <= -150.0f) ph = PH_AP;
        if (alt_ft >= 1000.0f && roc >= 150.0f) ph = PH_CL;
        if (alt_ft >= 1000.0f && roc <= -150.0f) ph = PH_DE;
        if (alt_ft >= 10000.0f && roc <= 150.0f && roc >= -150.0f) ph = PH_CR;
        T.ph = ph;
        x.f = (x.f & ~(uint32_t)(BSG_TF_PH_GD | BSG_TF_PH_AP)) | (ph == PH_GD ? (uint32_t)BSG_TF_PH_GD : 0u) |
              (ph == PH_AP ? (uint32_t)BSG_TF_PH_AP : 0u);
        float vmin = pf.vminer, vmax = pf.vmaxer;
        if (ph == PH_AP) { vmin = pf.vminap; vmax = pf.vmaxap; }
        if (ph == PH_GD) { vmin = 0.0f; vmax = pf.vmaxic; }
        T.amax = ph == PH_GD ? pf.axmax_gd : pf.axmax_air;
        T.inv_amax = 1.0f / T.amax;
        T.allow_h = p_alt > pf.hmax ? pf.hmax : p_alt;
        const Atmos ah = vatmos(T.allow_h);
        const float intent_cas = tas2cas(p_tas, ah);
        float allow_tas = p_tas;                           // vcas2tas(vtas2cas(x)) == x when not clamped
        if (intent_cas < vmin) allow_tas = cas2tas(vmin, ah);
        if (intent_cas > vmax) allow_tas = cas2tas(vmax, ah);
        const float snd = vsound(ah);
        if (allow_tas > pf.mmo * snd) allow_tas = pf.mmo * snd;
        T.allow_tas = allow_tas;
        T.at = at; T.k_alt = a.alt; T.k_vs = a.vs;
    }
    // ---- Traffic.update_airspeed / update_groundspeed / update_pos (the env kernels' routine) -----------------------
    EnvParams E{};
    E.simdt = P.simdt; E.perf = pf;
    ac_finish_load(a, E);                                  // cos(lat) for update_pos
    ac_kinematics<false, true>(a, E, T, p_trk, p_vs);
    traf_store(a, x, P, i);
    if (n_switch) atomicAdd(&P.counters[BSG_TRAF_CTR_SWITCH], 1u);
    if (x.f & BSG_TF_ASAS) atomicAdd(&P.counters[BSG_TRAF_CTR_ACTIVE], 1u);
}

}  // namespace bsg

using namespace bsg;

static int traf_params(TrafParams& P, const bsg_traf_config* cfg, const bsg_traf_tensors* t, const char* who) {
    if (!cfg || !t) return bsg_fail(BSG_EINVAL, "bsg_traf_*: null argument");
    if (cfg->n < 0 || cfg->n > 0x7fffff00LL) return bsg_fail(BSG_EINVAL, "bsg_traf_*: n out of range");
    if (cfg->max_wpts < 0 || cfg->max_wpts > 255) return bsg_fail(BSG_EINVAL, "bsg_traf_*: max_wpts must be in [0, 255]");
    if (!(cfg->simdt > 0.0f)) return bsg_fail(BSG_EINVAL, "bsg_traf_*: simdt must be > 0");
    if (cfg->row0 < 0 || cfg->row0 % 256 || cfg->row0 + cfg->n > 0x7fffff00LL) return bsg_fail(BSG_EINVAL, "bsg_traf_*: row0 must be a non-negative multiple of 256");
    if (cfg->n > 0 && (!t->pos || !t->kin || !t->cmd || !t->aux || !t->actwp || !t->vnav1 || !t->vnav2 || !t->asas || !t->flags ||
                       !t->partners || !t->counters))
        return bsg_fail(BSG_EINVAL, "bsg_traf_*: a required tensor pointer is null");
    if (cfg->n > 0 && cfg->max_wpts > 0 && (!t->rt_pos || !t->rt_con || !t->rt_dir)) return bsg_fail(BSG_EINVAL, "bsg_traf_*: route tables missing");
    (void)who;
    memset(&P, 0, sizeof(P));
    P.n = cfg->n; P.W = cfg->max_wpts; P.reso = cfg->reso; P.reso_mode = cfg->reso_mode;
    P.simdt = cfg->simdt;
    P.rpz = cfg->rpz > 0.0f ? cfg->rpz : 5.0f * 1852.0f;
    P.hpz = cfg->hpz > 0.0f ? cfg->hpz : 1000.0f * 0.3048f;
    P.dtlook = cfg->dtlookahead > 0.0f ? cfg->dtlookahead : 300.0f;
    P.resofach = cfg->resofach > 0.0f ? cfg->resofach : 1.01f;
    P.resofacv = cfg->resofacv > 0.0f ? cfg->resofacv : 1.01f;
    P.perf = cfg->perf; P.lat0 = cfg->lat0; P.lon0 = cfg->lon0; P.row0 = cfg->row0;
    P.pos = (double2*)t->pos; P.kin = (float4*)t->kin; P.cmd = (float4*)t->cmd; P.aux = (float4*)t->aux;
    P.actwp = (double2*)t->actwp; P.vn1 = (float4*)t->vnav1; P.vn2 = (float4*)t->vnav2; P.asas = (float4*)t->asas;
    P.flags = t->flags; P.partners = t->partners;
    P.rt_pos = (const double2*)t->rt_pos; P.rt_con = (const float4*)t->rt_con; P.rt_dir = t->rt_dir; P.counters = t->counters;
    return BSG_OK;
}

extern "C" int bsg_traf_pack(const bsg_traf_config* cfg, const bsg_traf_tensors* t, float* d_rec, void* stream) {
    TrafParams P;
    int rc = traf_params(P, cfg, t, "bsg_traf_pack");
    if (rc != BSG_OK) return rc;
    if (!d_rec) return bsg_fail(BSG_EINVAL, "bsg_traf_pack: null d_rec");
    const long long n_pad = bsg_cd_padded(P.n);
    if (n_pad == 0) return BSG_OK;
    traf_pack_kernel<<<(unsigned)(n_pad / 256), 256, 0, (cudaStream_t)stream>>>(P, d_rec, n_pad);
    return bsg_cuda_check(cudaGetLastError(), "bsg_traf_pack launch");
}

// (cd_order.cu)
int bsg_traf_order_launch(const double2* pos, const uint32_t* flags, int64_t n, double lon0, int32_t* d_perm, void* d_work,
                          cudaStream_t st);

extern "C" int64_t bsg_traf_order_workspace(int64_t n) { return bsg_cd_order_workspace(n); }

extern "C" int bsg_traf_pack_ordered(const bsg_traf_config* cfg, const bsg_traf_tensors* t, int32_t reorder, int32_t* d_perm,
                                     float* d_rec_ordered, float* d_rec, void* d_work, int64_t work_bytes, void* stream) {
    TrafParams P;
    int rc = traf_params(P, cfg, t, "bsg_traf_pack_ordered");
    if (rc != BSG_OK) return rc;
    if (P.row0 != 0) return bsg_fail(BSG_EINVAL, "bsg_traf_pack_ordered: not for an airspace sharded over GPUs (row0 != 0)");
    if (!d_perm || !d_rec_ordered) return bsg_fail(BSG_EINVAL, "bsg_traf_pack_ordered: null d_perm or d_rec_ordered");
    if (reorder) {
        if (!d_work || work_bytes < bsg_traf_order_workspace(P.n))
            return bsg_fail(BSG_EINVAL, "bsg_traf_pack_ordered: workspace too small (bsg_traf_order_workspace)");
        if ((uintptr_t)d_work % 8) return bsg_fail(BSG_EINVAL, "bsg_traf_pack_ordered: workspace must be 8-byte aligned");
    }
    const long long n_pad = bsg_cd_padded(P.n);
    if (n_pad == 0) return BSG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (reorder) {
        rc = bsg_traf_order_launch(P.pos, P.flags, P.n, P.lon0, d_perm, d_work, st);
        if (rc != BSG_OK) return rc;
    }
    traf_pack_ordered_kernel<<<(unsigned)(n_pad / 256), 256, 0, st>>>(P, d_perm, d_rec_ordered, d_rec, n_pad);
    return bsg_cuda_check(cudaGetLastError(), "bsg_traf_pack_ordered launch");
}

extern "C" int bsg_traf_activate(const bsg_traf_config* cfg, const bsg_traf_tensors* t, void* stream) {
    TrafParams P;
    int rc = traf_params(P, cfg, t, "bsg_traf_activate");
    if (rc != BSG_OK) return rc;
    if (P.n == 0) return BSG_OK;
    if (P.W == 0) return bsg_fail(BSG_EINVAL, "bsg_traf_activate: max_wpts is 0");
    traf_activate_kernel<<<(unsigned)((P.n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(P);
    return bsg_cuda_check(cudaGetLastError(), "bsg_traf_activate launch");
}

extern "C" int64_t bsg_traf_workspace(int64_t n, int64_t conf_cap) {
    if (n < 0 || conf_cap < 0) return 0;
    return (int64_t)sizeof(int) * (3 * n + 1 + conf_cap) + 64;
}

extern "C" int bsg_traf_substep(const bsg_traf_config* cfg, const bsg_traf_tensors* t, const float* d_rec, int32_t fms_ready,
                                const int32_t* d_conf_pairs, const float* d_conf_attr, const unsigned long long* d_npairs,
                                const unsigned long long* d_nconf_all, int64_t conf_cap, void* d_work, int64_t work_bytes,
                                void* stream) {
    TrafParams P;
    int rc = traf_params(P, cfg, t, "bsg_traf_substep");
    if (rc != BSG_OK) return rc;
    if (P.n == 0) return BSG_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if (P.reso) {
        if (P.reso != 1) return bsg_fail(BSG_EINVAL, "bsg_traf_substep: reso must be 0 (off) or 1 (MVP)");
        if (!d_rec || !d_conf_pairs || !d_conf_attr || !d_npairs || conf_cap <= 0)
            return bsg_fail(BSG_EINVAL, "bsg_traf_substep: reso needs the CD records and the detection's conflict list");
        if (conf_cap > 0x7fffff00LL) return bsg_fail(BSG_EINVAL, "bsg_traf_substep: conf_cap exceeds int32");
        if (!d_work || work_bytes < bsg_traf_workspace(P.n, conf_cap)) return bsg_fail(BSG_EINVAL, "bsg_traf_substep: workspace too small");
        P.rec = d_rec; P.pairs = (const int2*)d_conf_pairs; P.attr = d_conf_attr; P.npairs = d_npairs; P.cap = conf_cap;
        P.nconf_all = d_nconf_all ? d_nconf_all : d_npairs;
        // workspace: count[n] (zero on entry: the caller zeroes it once, the scatter leaves it zero) | offs[n] | len[n] | total | seg[cap]
        P.count = (int*)d_work; P.offs = P.count + P.n; P.len = P.offs + P.n; P.total = P.len + P.n; P.seg = P.total + 1;
        const unsigned blocks = (unsigned)((conf_cap + 255) / 256);
        traf_conf_count_kernel<<<blocks, 256, 0, st>>>(P);
        traf_conf_alloc_kernel<<<(unsigned)((P.n + 255) / 256), 256, 0, st>>>(P);
        traf_conf_scatter_kernel<<<blocks, 256, 0, st>>>(P);
        BSG_CUDA(cudaGetLastError());
    }
    P.fms_ready = fms_ready ? 1 : 0;
    BSG_CUDA(cudaMemsetAsync(t->counters + BSG_TRAF_CTR_ACTIVE, 0, sizeof(uint32_t), st));   // (a per-substep figure)
    traf_substep_kernel<<<(unsigned)((P.n + 127) / 128), 128, 0, st>>>(P);
    return bsg_cuda_check(cudaGetLastError(), "bsg_traf_substep launch");
}
