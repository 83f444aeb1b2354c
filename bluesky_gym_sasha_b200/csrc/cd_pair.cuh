// cd_pair.cuh -- one ordered aircraft pair of state-based conflict detection, float32.
// Restates the per-element arithmetic of bluesky/traffic/asas/statebased.py::StateBased.detect
// (see oracle/statebased.py for the float64 restatement this is checked against; the reference never
// enables ASAS -- merge_env.py:157 only issues `reso off` -- BASELINE.json's north_star adds it).
//
// CD record (32 B, two float4; stored tile-blocked, cd_record.cuh):  A = (x, y, ch, sh)   B = (u, v, alt, vs)
//   x = Re*rad(lon - lon0), y = Re*rad(lat - lat0)   [m of arc from the airspace origin]
//   ch, sh = cos, sin of lat/2                       (cos of the pair's mean latitude = chi*chj - shi*shj)
//   u = gs sin(trk), v = gs cos(trk)                 [m/s east, north]
// Algebra used (identical to upstream's, fewer special-function ops):
//   dist sin(qdr) = x-difference * cos(mean lat), dist cos(qdr) = y-difference  (no atan2/sin/cos),
//   dcpa^2 = |d x w|^2 / |w|^2  (Lagrange identity for dist^2 - tcpa^2 |w|^2; no cancellation;
//            the literal form is kept when |w|^2 is clamped, i.e. for co-moving aircraft),
//   dxinhor / vrel = sqrt((R^2 - dcpa^2) / |w|^2)    (one MUFU.RCP shared with tcpa),
//   min/max(tcrosshi, tcrosslo) = t0 -+ |hpz / dvs|.
// 3 MUFU (rcp, sqrt, rcp) + ~45 FMA/ALU-pipe instructions per ordered pair.
#pragma once
#include <cuda_runtime.h>

namespace bsg {

constexpr float kTwoPiRe = 6.283185307179586f * 6371000.0f;
constexpr float kInvTwoPiRe = 1.0f / (6.283185307179586f * 6371000.0f);

__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

typedef unsigned long long u64;
// ---- packed f32x2 arithmetic (SASS FADD2 / FMUL2 / FFMA2) ------------------------------------------
__device__ __forceinline__ u64 pk2(float lo, float hi) {
    u64 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void up2(u64 v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ u64 add2(u64 a, u64 b) {
    u64 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ u64 mul2(u64 a, u64 b) {
    u64 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c) {
    u64 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}


struct CdPair {
    bool conf, los;
    float tcpa;
    // what upstream's detect() returns per conflict besides the pair (qdr, dist, dcpa, tcpa, tinconf): dx, dy give
    // qdr = atan2(dx, dy) and dist on the (rare) emitting path; unused fields are dropped by the compiler
    float tinconf, dcpa2, dist2, dx, dy;
};

// (i) = own row, (j) = intruder column.  `same` marks the diagonal (upstream adds 1e9*eye).
template <bool WRAP>
__device__ __forceinline__ CdPair cd_pair_eval(const float4 Ai, const float4 Bi, const float4 Aj,
                                               const float4 Bj, float R2, float hpz, float dtlook,
                                               bool same) {
    float dy = Aj.y - Ai.y;
    float dxl = Aj.x - Ai.x;
    if (WRAP) dxl -= kTwoPiRe * rintf(dxl * kInvTwoPiRe);
    float cav = fmaf(-Ai.w, Aj.w, Ai.z * Aj.z);
    float dx = dxl * cav;
    float du = Bj.x - Bi.x, dv = Bj.y - Bi.y;
    float dv2r = fmaf(du, du, dv * dv);
    bool clamped = dv2r < 1e-6f;                // upstream: dv2 = where(|dv2| < 1e-6, 1e-6, dv2)
    float dv2 = clamped ? 1e-6f : dv2r;
    float dot = fmaf(du, dx, dv * dy);
    float crs = fmaf(dx, dv, -dy * du);
    float inv = rcp_approx(dv2);
    float tcpa = -dot * inv;
    float dist2 = fmaf(dx, dx, dy * dy);
    // |dist^2 - tcpa^2 dv2| == |d x w|^2 / |w|^2 only while dv2 is the true |w|^2; keep upstream's
    // literal form for the (co-moving) clamped case
    float dcpa2 = clamped ? fabsf(fmaf(-tcpa * tcpa, dv2, dist2)) : crs * crs * inv;
    bool swhor = dcpa2 < R2;
    float dtin = sqrt_approx((R2 - dcpa2) * inv);
    float tinhor = swhor ? tcpa - dtin : 1e8f;
    float touthor = swhor ? tcpa + dtin : -1e8f;
    float dalt = Bj.z - Bi.z;
    float dvs = Bj.w - Bi.w;
    dvs = fabsf(dvs) < 1e-6f ? 1e-6f : dvs;
    float ninv = -rcp_approx(dvs);
    float t0 = dalt * ninv;
    float hw = fabsf(hpz * ninv);
    float tinconf = fmaxf(t0 - hw, tinhor);
    float toutconf = fminf(t0 + hw, touthor);
    CdPair o;
    o.conf = swhor && (tinconf <= toutconf) && (toutconf > 0.0f) && (tinconf < dtlook) && !same;
    o.los = (dist2 < R2) && (fabsf(dalt) < hpz) && !same;
    o.tcpa = tcpa; o.tinconf = tinconf; o.dcpa2 = dcpa2; o.dist2 = dist2; o.dx = dx; o.dy = dy;
    return o;
}

// Both orders of one unordered pair at once.  (j, i) mirrors (i, j) exactly -- every difference changes
// sign, tcpa / dcpa / dist are even in them -- except upstream's clamp of a near-zero relative vertical
// speed to +1e-6 in BOTH orders, which flips the sign of the (j, i) vertical crossing time.
struct CdSym {
    bool conf_ij, conf_ji, los;
    float tcpa;
    float tin_ij, tin_ji, dcpa2, dist2, dx, dy;      // attributes of the pair (dx, dy as seen from i; (j, i): negated)
};
__device__ __forceinline__ CdSym cd_pair_sym(const float4 Ai, const float4 Bi, const float4 Aj, const float4 Bj,
                                             float R2, float hpz, float dtlook) {
    float dy = Aj.y - Ai.y;
    float dxl = Aj.x - Ai.x;
    float cav = fmaf(-Ai.w, Aj.w, Ai.z * Aj.z);
    float dx = dxl * cav;
    float du = Bj.x - Bi.x, dv = Bj.y - Bi.y;
    float dv2r = fmaf(du, du, dv * dv);
    float dv2 = fmaxf(dv2r, 1e-6f);
    float dot = fmaf(du, dx, dv * dy);
    float crs = fmaf(dx, dv, -dy * du);
    float inv = rcp_approx(dv2);
    float tcpa = -dot * inv;
    float dcpa2 = crs * crs * inv;
    if (dv2r < 1e-6f) {            // co-moving pair (rare): upstream's literal |dist^2 - tcpa^2 dv2| with the clamp
        float dist2 = fmaf(dx, dx, dy * dy);
        dcpa2 = fabsf(fmaf(-tcpa * tcpa, dv2, dist2));
    }
    bool swhor = dcpa2 < R2;
    // sqrt of a negative number is NaN when dcpa >= R; fmaxf / fminf drop the NaN operand and the
    // predicates below require swhor anyway, so no select is needed for the 1e8 / -1e8 sentinels
    float dtin = sqrt_approx((R2 - dcpa2) * inv);
    float tinhor = tcpa - dtin, touthor = tcpa + dtin;
    float dalt = Bj.z - Bi.z;
    float dvs = Bj.w - Bi.w;
    bool vclamp = fabsf(dvs) < 1e-6f;
    dvs = vclamp ? 1e-6f : dvs;
    float ninv = -rcp_approx(dvs);
    float t0 = dalt * ninv;
    float hw = fabsf(hpz * ninv);
    float t0r = vclamp ? -t0 : t0;
    float tin = fmaxf(t0 - hw, tinhor), tout = fminf(t0 + hw, touthor);
    float tinr = fmaxf(t0r - hw, tinhor), toutr = fminf(t0r + hw, touthor);
    CdSym o;
    o.conf_ij = swhor && (tin <= tout) && (tout > 0.0f) && (tin < dtlook);
    o.conf_ji = swhor && (tinr <= toutr) && (toutr > 0.0f) && (tinr < dtlook);
    // LoS (dist < R and |dalt| < hpz) implies dcpa < R: only looked at under swhor
    const float d2 = fmaf(dx, dx, dy * dy);
    o.los = swhor && (d2 < R2) && (fabsf(dalt) < hpz);
    o.tcpa = tcpa; o.tin_ij = tin; o.tin_ji = tinr; o.dcpa2 = dcpa2; o.dist2 = d2; o.dx = dx; o.dy = dy;
    return o;
}

}  // namespace bsg
