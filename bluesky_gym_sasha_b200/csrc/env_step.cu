// env_step.cu -- K4/K5/K6: per-env scenario generators, action mapping, observation / reward /
// termination, and the env-step megakernel that strings them around the substep loop of
// env_kernels.cuh.  Every function cites the reference lines it restates; the float64 CPU
// restatement these are parity-tested against is oracle/envs.py.
#include "env_kernels.cuh"

namespace bsg {

struct StepOut { float reward; int terminated; int truncated; };

// rank (0..K-1) of this lane among the K nearest candidates of its group, else -1
template <int G>
__device__ __forceinline__ int nearest_rank(float dist, bool cand, int K) {
    const unsigned lane_g = threadIdx.x & (G - 1);
    unsigned long long key = cand ? (((unsigned long long)__float_as_uint(dist)) << 32) | lane_g : ~0ULL;
    int rank = -1;
    for (int r = 0; r < K; ++r) {
        unsigned long long m = group_min_u64<G>(key);
        if (m == key && key != ~0ULL) { rank = r; key = ~0ULL; }
    }
    return rank;
}

// vcas2tas(150 m/s, h) for the integer altitudes h = 2000 .. 4000 m that the DescentEnv / VerticalCREnv generators draw
// (alt_init = randint(2000, 4000)): float64, evaluated on the host when the handle is created (api.cu), so the generators
// keep the oracle's float64 values without a float64 pow chain at the tail of every launch with a finishing env
__device__ double g_tas150_tab[2001];

// =====================================================================================================
// DescentEnv (descent_env.py) -- 1 aircraft, G = 1
// =====================================================================================================
template <int G>
__device__ inline void descent_reset(Ac& a, EnvS& s, const EnvParams& P, long long e, int slot) {
    Philox rng = make_philox(P.seed, P.gid0 + e, (uint32_t)s.episode);      // descent_env.py:162-182
    int alt_init = rng.randint(0, 2000, 4000);
    s.target_alt = (double)(alt_init + rng.randint(1, -500, 500));
    double hdg = P.hdg_random ? (double)rng.randint(2, 1, 360) : 0.0;
    if (slot == 0) ac_create_tas(a, 52.0, 4.0, hdg, (double)alt_init, 150.0, g_tas150_tab[alt_init - 2000]);
    else ac_clear(a);
    s.total_reward = 0.0f; s.final_alt = 0.0f; s.num_ac = 1;
}
template <int G>
__device__ inline void descent_action(Ac& a, const EnvParams& P, const float* act, int slot) {
    float vs_cmd = act[0] * 12.5f;                                          // descent_env.py:146-160
    if (slot == 0) { a.selalt = vs_cmd >= 0.0f ? 1000000.0f : 0.0f; a.selvs = vs_cmd; }
}
template <int G>
__device__ inline StepOut descent_obs_reward(const Ac& a, EnvS& s, const EnvParams& P, float* obs, int slot,
                                             bool with_reward) {
    float q, dnm;                                                           // descent_env.py:89-117
    kwikqdrdist(52.0, 4.0, a.lat, a.lon, q, dnm);
    float rwy = 200.0f - dnm * 1.852f;
    float tgt = (float)s.target_alt;
    if (slot == 0) {
        obs[0] = (a.alt - 1500.0f) * (1.0f / 3000.0f);
        obs[1] = a.vs * 0.2f;
        obs[2] = (tgt - 1500.0f) * (1.0f / 3000.0f);
        obs[3] = (rwy - 100.0f) * (1.0f / 200.0f);
    }
    StepOut o = {0.0f, 0, 0};
    if (!with_reward) return o;
    if (rwy > 0.0f && a.alt > 0.0f) {                                       // descent_env.py:128-144
        o.reward = fabsf(tgt - a.alt) * (-5.0f / 3000.0f);
    } else if (a.alt <= 0.0f) {
        o.reward = -100.0f; o.terminated = 1; s.final_alt = -100.0f;
    } else {
        o.reward = a.alt * (-50.0f / 3000.0f); o.terminated = 1; s.final_alt = a.alt;
    }
    s.total_reward += o.reward;
    return o;
}
__device__ inline void descent_info(const EnvS& s, float* info) {           // descent_env.py:119-126
    info[0] = s.total_reward; info[1] = s.final_alt; info[2] = 0.0f; info[3] = 0.0f;
}

// =====================================================================================================
// HorizontalCREnv (horizontal_cr_env.py) -- slot 0 = ownship, slots 1..n = creconfs intruders
// =====================================================================================================
// The generator of an env that finishes runs at the END of a launch, on one warp, when the rest of the batch is done:
// its dependent chain of float64 special functions IS the tail of the launch (25 us of a 45 us launch before this form,
// measured with per-warp phase stamps).  So: the ISA / CAS conversions at the configured altitude come from the host (init_tas0),
// upstream's vtas2cas -> cre -> vcas2tas round trip of an intruder's speed is taken as the identity it is (the intruder
// flies the reference ground speed to 2e-16: |cas - 150| ~ 1e-14 << half an ulp of the float32 state), headings come from
// the track angle instead of atan2 of its own sine / cosine, sines and cosines are evaluated in pairs (sincos), and the
// waypoint straight north of the ownship (bearing 0 in functions.py:24-42) is lat0 + distance / R.
template <int G>
__device__ inline void horizontal_reset(Ac& a, EnvS& s, const EnvParams& P, long long e, int slot) {
    Philox rng = make_philox(P.seed, P.gid0 + e, (uint32_t)s.episode);      // horizontal_cr_env.py:82-101
    const int n = P.n_int;
    const double hdg0 = P.hdg_random ? (double)rng.randint(0, 1, 360) : 0.0;
    const double lat0 = 52.0, lon0 = 4.0, alt0 = (double)P.init_alt;     // reference: cre without acalt => 0
    const double tas0 = P.init_tas0;                                      // vcas2tas(150, init_alt), host-evaluated
    const double trkref = hdg0 * kDeg2RadD, gsref = tas0;
    double sr, cr;
    sincos(trkref, &sr, &cr);
    if (slot == 0) {
        ac_create_dir(a, lat0, lon0, hdg0, alt0, 150.0, tas0, cr, sr);
    } else if (slot <= n) {
        // Traffic.creconfs (oracle/traffic.py::creconfs), horizontal_cr_env.py:127-133
        const uint32_t d = 1u + 3u * (uint32_t)(slot - 1);
        const double dpsi = (double)rng.randint(d, 45, 315);
        const double cpa = (double)rng.randint(d + 1, 0, 5) * 1852.0;
        const double tlosh = (double)rng.randint(d + 2, 100, 1000);
        const double pzr = 5.0 * 1852.0;
        const double trk = trkref + dpsi * kDeg2RadD;
        double st, ct;
        sincos(trk, &st, &ct);
        const double gsn = gsref * ct, gse = gsref * st;
        const double vreln = gsref * cr - gsn, vrele = gsref * sr - gse;
        const double vrel = sqrt(vreln * vreln + vrele * vrele);
        const double drelcpa = tlosh * vrel + (cpa > pzr ? 0.0 : sqrt(pzr * pzr - cpa * cpa));
        const double dist = sqrt(drelcpa * drelcpa + cpa * cpa);
        const double rd = drelcpa / dist, rx = cpa / dist;
        const double brn = atan2(-rx * vreln + rd * vrele, rd * vreln + rx * vrele);      // [rad]
        double sb, cb;
        sincos(brn, &sb, &cb);
        // geo.kwikpos
        const double dnm = dist / 1852.0;
        const double lat = lat0 + dnm * cb / 60.0;
        double lon = lon0 + dnm * sb / fmax(0.01, 60.0 * 0.6156614753256583);           // cos(52 deg)
        lon = fmod(lon + 180.0, 360.0); if (lon < 0.0) lon += 360.0; lon -= 180.0;
        const double gs = sqrt(gsn * gsn + gse * gse);
        const double acspd = 150.0 * (gs / tas0);              // vtas2cas(gs) to first order in (gs / tas0 - 1) ~ 1e-16
        // achdg = degrees(atan2(gse, gsn)): the track angle folded into (-180, 180]
        double achdg = hdg0 + dpsi;
        achdg = achdg > 180.0 ? achdg - 360.0 : achdg;
        achdg = achdg > 180.0 ? achdg - 360.0 : achdg;
        ac_create_dir(a, lat, lon, achdg, alt0, acspd, gs, ct, st);
    } else {
        ac_clear(a);
    }
    const int wpt_dis = rng.randint(1u + 3u * (uint32_t)n, 100, 150);       // horizontal_cr_env.py:135-148
    s.wpt_lat = lat0 + ((double)wpt_dis / 6371.0) * kRad2DegD;              // get_point_at_distance(lat0, lon0, d, bearing 0)
    s.wpt_lon = lon0;
    s.wpt_reach = 0; s.total_reward = 0.0f; s.intrusions = 0; s.drift_sum = 0.0f; s.drift_n = 0;
    s.num_ac = n + 1;
}
template <int G>
__device__ inline void horizontal_action(Ac& a, const EnvParams& P, const float* act, int slot) {
    if (slot == 0) {                                                        // horizontal_cr_env.py:272-275
        a.aptrk = fmaf(act[0], 45.0f, a.hdg);      // un-wrapped, like the reference's "HDG KL001 x" (explicit fma: one
                                                   // rounding whatever the surrounding code looks like to the compiler)
        a.flags &= ~kFlLnav;
    }
}
template <int G>
__device__ inline StepOut horizontal_obs_reward(const Ac& a, EnvS& s, const EnvParams& P, float* obs, int slot,
                                                bool with_reward) {
    const int n = P.n_int;                                                  // horizontal_cr_env.py:150-213
    const double lat0 = group_bcast<G>(a.lat, 0), lon0 = group_bcast<G>(a.lon, 0);
    const float gs_own = ac_gs(a, P);
    const float hdg0 = group_bcast<G>(a.hdg, 0), gs0 = group_bcast<G>(gs_own, 0);
    const bool intr = slot >= 1 && slot <= n;
    float dis = 1e9f;
    if (intr) {
        // cos / sin of (own heading - bearing to the intruder) from the flat-earth offsets themselves: cos(qdr) = dn / ang,
        // sin(qdr) = de / ang (the reference goes through atan2 and back; same quantities, fewer roundings)
        float dn, de, ang, sd, cd, sh0, ch0;
        kwikoffsets(lat0, lon0, a.lat, a.lon, dn, de, ang, dis);
        __sincosf((hdg0 - 180.0f) * kDeg2Rad, &sh0, &ch0);          // hdg0 in [0, 360): shifted into the MUFU's accurate range
        sh0 = -sh0; ch0 = -ch0;
        const float inv = ang > 0.0f ? 1.0f / ang : 0.0f;
        const float cq = ang > 0.0f ? dn * inv : 1.0f, sq = de * inv;
        const float cb = fmaf(ch0, cq, sh0 * sq), sb = fmaf(sh0, cq, -ch0 * sq);
        sincos_deg((hdg0 - a.hdg), sd, cd);
        const int k = slot - 1;
        obs[k] = dis * (1.852f / 150.0f);
        obs[n + k] = cb;
        obs[2 * n + k] = sb;
        obs[3 * n + k] = -cd * gs_own * (1.0f / 150.0f);
        obs[4 * n + k] = (gs0 - sd * gs_own) * (1.0f / 150.0f);
    }
    float wq, wd;
    kwikqdrdist(lat0, lon0, s.wpt_lat, s.wpt_lon, wq, wd);
    const float wkm = wd * 1.852f;
    const float drift = wrap180_fold(hdg0 - wq);
    if (slot == 0) {
        float sd, cd;
        sincos_deg(drift, sd, cd);
        obs[5 * n] = wkm * (1.0f / 150.0f);
        obs[5 * n + 1] = cd;
        obs[5 * n + 2] = sd;
    }
    StepOut o = {0.0f, 0, 0};
    if (!with_reward) return o;
    const int nintr = group_sum<G>((intr && dis < 5.0f) ? 1 : 0);           // horizontal_cr_env.py:225-270
    float r = 0.0f;
    if (wkm < 5.0f && s.wpt_reach != 1) { s.wpt_reach = 1; r += 1.0f; }
    const float dr = fabsf(drift * kDeg2Rad);
    s.drift_sum += dr; s.drift_n += 1;
    r += dr * -0.1f;
    s.intrusions += nintr;
    r += -1.0f * (float)nintr;
    s.total_reward += r;
    o.reward = r; o.terminated = s.wpt_reach ? 1 : 0;
    return o;
}
__device__ inline void drift_info(const EnvS& s, float* info) {             // horizontal_cr_env.py:215-223
    info[0] = s.total_reward; info[1] = (float)s.intrusions;
    info[2] = s.drift_sum / (float)s.drift_n;       // 0/0 = NaN before the first step, like np.mean([])
    info[3] = 0.0f;
}

// =====================================================================================================
// SectorCREnv (sector_cr_env.py) -- G = 32, variable aircraft count, polygon airspace
// =====================================================================================================
__device__ inline bool d_inside_poly(double px, double py, const double* poly, int nv) {
    // areafilter.checkInside -> even-odd crossing in the (lat, lon) plane (oracle/geo.py::point_in_polygon)
    int c = 0;
    for (int k = 0; k < nv; ++k) {
        int k2 = (k + 1 == nv) ? 0 : k + 1;
        double x1 = poly[2 * k], y1 = poly[2 * k + 1], x2 = poly[2 * k2], y2 = poly[2 * k2 + 1];
        if ((y1 > py) != (y2 > py)) {
            double xint = x1 + (py - y1) * (x2 - x1) / (y2 - y1);
            c += px < xint ? 1 : 0;
        }
    }
    return (c & 1) == 1;
}

constexpr int kSectorMaxV = 32, kSectorMaxAc = 32, kSectorMaxTries = 4096;

// Scenario generator spread over the 32 lanes of the env's warp (a serial version on lane 0 took ~100 us of
// dependent float64 work and set the duration of the whole launch whenever any env of the batch reset).  Philox draws are
// addressed by index, so every lane computes the draws it needs; the DRAW ORDER of the reference is unchanged:
// draw k = polygon point k (k < nv), then the density draw(s), then num_ac perimeter positions, then two draws per
// rejection-sampling try.  scratch per warp (float64): [0,32) lat | [32,64) lon of the accepted aircraft; [96,128) sorted vx | [128,160) sorted vy | [160,192) edge length |
// [192,225) cumulative edge length | [225,257) sorted perimeter draws | [257,289) wx | [289,321) wy.
constexpr int kSectorScratch = 324;

template <int G>
__device__ inline void sector_reset(Ac& a, EnvS& s, const EnvParams& P, long long e, int slot, double* scratch) {
    // (instantiated for every G by do_reset's dispatch, but only ever run with G == 32: one full warp per env)
    double* poly = P.poly + e * (2 * kSectorMaxV);
    double* s_vx = scratch + 96, *s_vy = scratch + 128, *s_el = scratch + 160, *s_cum = scratch + 192;
    double* s_dl = scratch + 225, *s_wx = scratch + 257, *s_wy = scratch + 289;
    const Philox rng = make_philox(P.seed, P.gid0 + e, (uint32_t)s.episode);
    const double R = sqrt(3750.0 / 3.141592653589793);
    const double coslat0 = cos(kSectorLat0 * kDeg2RadD);
    // ---- A: candidate polygon point `slot` = random_point_on_circle with draw `slot` (functions.py:44-59) ----------
    const double al = 6.283185307179586 * rng.u01((uint32_t)slot);
    double sal, cal;
    sincos(al, &sal, &cal);
    const double cx = R * cal, cy = R * sal;
    // sort key: atan2(cy, cx) is al itself folded into (-pi, pi] (to rounding: only the ORDER of the keys is used)
    const double ca = al > 3.141592653589793 ? al - 6.283185307179586 : al;
    // ---- B: the polygon = the first nv candidates sorted by angle (sort_points_clockwise = ascending atan2(y, x),
    //      functions.py:61-75), nv the smallest count >= 3 whose area reaches 2400 (sector_cr_env.py:141-160: points are
    //      inserted in draw order until the area is large enough).  All 32 prefixes at once instead of a serial loop of
    //      insertions and shoelace sums on one lane (which took 7-30 us and set the duration of the launch): inserting
    //      point n between its neighbours by angle among the points drawn before it replaces the edge pred -> succ by
    //      pred -> p -> succ, so the signed shoelace sum of the first n + 1 points is a prefix sum of per-lane terms.
    int num_ac = 0, nv = 0, rflags = 0;
    uint32_t d = 0;
    double area = 0.0, perim = 0.0, minx = 0.0, maxx = 0.0, miny = 0.0, maxy = 0.0;
    {
        // (polygons rarely need more than a dozen points: the first 16 prefixes are tried first, all 32 only if none suffices)
        unsigned big = 0u;
        for (int pass = 0; pass < 2 && !big; ++pass) {
            const int jmax = pass ? 31 : 15;                                                  // (no lane has lane 31 before it)
            double pa = -1.0e300, px = 0.0, py = 0.0, sa = 1.0e300, sx = 0.0, sy = 0.0;        // nearest below / above by angle
            double ma = -1.0e300, mx = 0.0, my = 0.0, na = 1.0e300, nx = 0.0, ny = 0.0;        // largest / smallest of all
            for (int j = 0; j < jmax; ++j) {
                const double aj = __shfl_sync(0xffffffffu, ca, j), xj = __shfl_sync(0xffffffffu, cx, j), yj = __shfl_sync(0xffffffffu, cy, j);
                if (j < slot) {
                    if (aj <= ca) { if (aj >= pa) { pa = aj; px = xj; py = yj; } }             // (equal angles: the earlier draw sorts first)
                    else if (aj < sa) { sa = aj; sx = xj; sy = yj; }
                    if (aj >= ma) { ma = aj; mx = xj; my = yj; }
                    if (aj < na) { na = aj; nx = xj; ny = yj; }
                }
            }
            if (pa == -1.0e300) { px = mx; py = my; }                                          // the smallest angle follows the largest
            if (sa == 1.0e300) { sx = nx; sy = ny; }
            double S = slot > 0 ? (px * cy - py * cx) + (cx * sy - cy * sx) - (px * sy - py * sx) : 0.0;
            for (int o = 1; o < 32; o <<= 1) {                                                 // inclusive prefix sum over the lanes
                const double up = __shfl_up_sync(0xffffffffu, S, o);
                if (slot >= o) S += up;
            }
            big = __ballot_sync(0xffffffffu, slot >= 2 && slot <= jmax && fabs(S) * 0.5 >= 2400.0);
        }
        nv = big ? __ffs((int)big) : kSectorMaxV;                                              // lane n - 1 holds the polygon of n points
        if (!big) rflags |= 1;
        int rank = 0;                                                                      // my place among the first nv by angle (stable)
        for (int j = 0; j < nv; ++j) {
            const double aj = __shfl_sync(0xffffffffu, ca, j);
            rank += (aj < ca || (aj == ca && j < slot)) ? 1 : 0;
        }
        if (slot < nv) { s_vx[rank] = cx; s_vy[rank] = cy; }
        __syncwarp();
        // area of the chosen polygon with the reference's own shoelace sum (fn.polygon_area), edge lengths, bounding box
        const int jn = (slot + 1 == nv) ? 0 : slot + 1;
        const bool vert = slot < nv;
        const double vx = vert ? s_vx[slot] : 0.0, vy = vert ? s_vy[slot] : 0.0;
        const double wx = vert ? s_vx[jn] : 0.0, wy = vert ? s_vy[jn] : 0.0;
        const double term = vx * wy - vy * wx;
        const double ex = wx - vx, ey = wy - vy;
        const double el = sqrt(ex * ex + ey * ey);
        double acc = 0.0;
        for (int i = 0; i < nv; ++i) {                  // sums in the reference's order (i = 0 .. nv - 1), on every lane alike
            acc += __shfl_sync(0xffffffffu, term, i);
            const double eli = __shfl_sync(0xffffffffu, el, i);
            if (i == slot) s_cum[i] = perim;            // cum[i] = el[0] + ... + el[i-1]
            perim += eli;
        }
        area = fabs(acc) / 2.0;
        if (vert) {
            s_el[slot] = el;
            poly[2 * slot] = kSectorLat0 + vx / 60.0;                                     // nm_to_latlong: x north, y east
            poly[2 * slot + 1] = kSectorLon0 + vy / (60.0 * coslat0);
        }
        double lox = vert ? vx : 1.0e300, hix = vert ? vx : -1.0e300, loy = vert ? vy : 1.0e300, hiy = vert ? vy : -1.0e300;
        for (int o = 16; o > 0; o >>= 1) {
            lox = fmin(lox, __shfl_xor_sync(0xffffffffu, lox, o)); hix = fmax(hix, __shfl_xor_sync(0xffffffffu, hix, o));
            loy = fmin(loy, __shfl_xor_sync(0xffffffffu, loy, o)); hiy = fmax(hiy, __shfl_xor_sync(0xffffffffu, hiy, o));
        }
        minx = lox; maxx = hix; miny = loy; maxy = hiy;
        // density -> number of aircraft (sector_cr_env.py:98-103); every lane evaluates the same draws
        d = (uint32_t)nv;
        double rho;
        if (P.sector_uniform) { rho = rng.uniform(d, 0.003, 0.007); d += 1; }
        else { rho = rng.normal(d, 0.005, 0.001); d += 2; }
        double nraw = fmax(ceil(rho * area), 5.0);
        if (nraw > (double)kSectorMaxAc) { nraw = (double)kSectorMaxAc; rflags |= 2; }
        num_ac = (int)nraw;
    }
    __syncwarp();
    // ---- C: _generate_waypoints (:162-188): num_ac draws along the perimeter, sorted, mapped onto the edges ----------
    {
        const bool mine = slot < num_ac;
        const double v = mine ? rng.uniform(d + (uint32_t)slot, 0.0, perim) : 1.0e300;
        int rank = 0;                                  // position of my draw in ascending order (stable)
        for (int j = 0; j < G; ++j) {
            const double vj = group_bcast<G>(v, j);
            rank += (vj < v || (vj == v && j < slot)) ? 1 : 0;
        }
        if (mine) s_dl[rank] = v;
        __syncwarp();
        if (mine) {                                    // sorted draw number `slot` -> point on edge k
            const double dl = s_dl[slot];
            int k = 0;
            while (k < nv - 1 && dl > s_cum[k] + s_el[k]) ++k;
            const int j = (k + 1 == nv) ? 0 : k + 1;
            const double frac = (dl - s_cum[k]) / s_el[k];
            s_wx[slot] = s_vx[k] + frac * (s_vx[j] - s_vx[k]);
            s_wy[slot] = s_vy[k] + frac * (s_vy[j] - s_vy[k]);
        }
        d += (uint32_t)num_ac;
    }
    __syncwarp();
    // ---- D: _generate_ac (:190-217): rejection sampling in the bounding box, 32 tries at a time; try t uses draws
    //         d + 2t and d + 2t + 1 and accepted points keep their try order, exactly as in the serial loop ----------
    double* a_lat = scratch, *a_lon = scratch + 32;    // (the candidate arrays are no longer needed)
    int got = 0;
    for (int base = 0; base < kSectorMaxTries && got < num_ac; base += 32) {
        const uint32_t t = (uint32_t)(base + slot);
        const double x = rng.uniform(d + 2u * t, minx, maxx), y = rng.uniform(d + 2u * t + 1u, miny, maxy);
        const double la = kSectorLat0 + x / 60.0, lo = kSectorLon0 + y / (60.0 * coslat0);
        const bool in = d_inside_poly(la, lo, poly, nv);
        const unsigned m = __ballot_sync(0xffffffffu, in);
        const int idx = got + __popc(m & ((1u << slot) - 1u));
        if (in && idx < num_ac) { a_lat[idx] = la; a_lon[idx] = lo; }
        got += __popc(m);
    }
    __syncwarp();
    if (got < num_ac) { rflags |= 4; num_ac = got > 0 ? got : 1; }
    // ---- E: one aircraft per lane: heading towards its waypoint (fn.get_hdg, functions.py:150-178) and Traffic.cre
    double w0lat = 0.0, w0lon = 0.0;
    if (slot < num_ac && got > 0) {
        const double la = a_lat[slot], lo = a_lon[slot];
        const double wla = kSectorLat0 + s_wx[slot] / 60.0, wlo = kSectorLon0 + s_wy[slot] / (60.0 * coslat0);
        const double l1 = la * kDeg2RadD, l2 = wla * kDeg2RadD, dlo = (wlo - lo) * kDeg2RadD;
        const double hx = sin(dlo) * cos(l2), hy = cos(l1) * sin(l2) - sin(l1) * cos(l2) * cos(dlo);
        const double h = fmod(kRad2DegD * atan2(hx, hy) + 360.0, 360.0);
        ac_create_tas(a, la, lo, h, 350.0, 150.0, P.init_tas0);
        w0lat = wla; w0lon = wlo;
    } else if (slot < num_ac) {
        ac_create_tas(a, 0.0, 0.0, 0.0, 350.0, 150.0, P.init_tas0);      // (no point could be placed: flagged in rflags, as before)
    } else {
        ac_clear(a);
    }
    w0lat = group_bcast<G>(w0lat, 0); w0lon = group_bcast<G>(w0lon, 0);
    __syncwarp();
    s.num_ac = num_ac; s.nvert = nv; s.rflags = rflags; s.poly_area = area;
    s.wpt_lat = w0lat; s.wpt_lon = w0lon;
    s.total_reward = 0.0f; s.intrusions = 0; s.drift_sum = 0.0f; s.drift_n = 0; s.wpt_reach = 0;
}
template <int G>
__device__ inline void sector_action(Ac& a, const EnvParams& P, const float* act, int slot) {
    if (slot == 0) {                                                        // sector_cr_env.py:315-322
        a.aptrk = wrap180_fold(fmaf(act[0], 22.5f, a.hdg));
        a.flags &= ~kFlLnav;
        float kt = fmaf(act[1], 20.0f / 3.0f, a.cas) * 1.94384f;            // "SPD KL001 x": knots -> m/s
        a.selspd = (kt > 0.1f && kt < 1.0f) ? kt : kt * kKts;
    }
}
template <int G>
__device__ inline StepOut sector_obs_reward(const Ac& a, EnvS& s, const EnvParams& P, float* obs, int slot,
                                            long long e, bool with_reward) {
    const double lat0 = group_bcast<G>(a.lat, 0), lon0 = group_bcast<G>(a.lon, 0);     // sector_cr_env.py:237-313
    const float hdg0 = group_bcast<G>(a.hdg, 0), tas0 = group_bcast<G>(a.tas, 0);
    // cos / sin(hdg) * tas: the cached ground-speed components are exactly that without wind; with wind they carry
    // the wind vector, which the reference's observation does not include (it uses bs.traf.hdg and bs.traf.tas)
    float avx = a.gsn, avy = a.gse;
    if (P.wind_n > 0) { float sh_, ch_; sincosf(a.hdg * kDeg2Rad, &sh_, &ch_); avx = a.tas * ch_; avy = a.tas * sh_; }
    const float vx0 = group_bcast<G>(avx, 0), vy0 = group_bcast<G>(avy, 0);
    float wq, wd;
    kwikqdrdist(lat0, lon0, s.wpt_lat, s.wpt_lon, wq, wd);
    const float drift = wrap180_fold(hdg0 - wq);
    if (slot == 0) {
        float sd, cd;
        sincos_deg(drift, sd, cd);
        obs[0] = cd; obs[1] = sd; obs[2] = (tas0 - 150.0f) * (1.0f / 6.0f);
    }
    const bool other = slot >= 1 && slot < s.num_ac;
    const double coslat0 = cos(kSectorLat0 * kDeg2RadD);
    float dxm = (float)((a.lat - lat0) * (60.0 * 1852.0));                  // latlong_to_nm * NM2KM * 1000
    float dym = (float)((a.lon - lon0) * (60.0 * 1852.0) * coslat0);
    float dist = sqrtf(dxm * dxm + dym * dym);
    int rank = nearest_rank<G>(dist, other, 4);
    if (rank >= 0) {
        float dvx = avx - vx0, dvy = avy - vy0;
        float hyp = sqrtf(dvx * dvx + dvy * dvy);
        float ct = hyp > 0.0f ? dvx / hyp : 1.0f, st = hyp > 0.0f ? dvy / hyp : 0.0f;
        obs[3 + rank] = dxm * (1.0f / 13000.0f);
        obs[7 + rank] = dym * (1.0f / 13000.0f);
        obs[11 + rank] = dvx * (1.0f / 32.0f);
        obs[15 + rank] = dvy * (1.0f / 66.0f);
        obs[19 + rank] = ct;
        obs[23 + rank] = st;
        obs[27 + rank] = (dist - 50000.0f) * (1.0f / 15000.0f);
    }
    StepOut o = {0.0f, 0, 0};
    if (!with_reward) return o;
    float q, dnm = 1e9f;                                                    // sector_cr_env.py:227-235,324-339
    if (other) kwikqdrdist(lat0, lon0, a.lat, a.lon, q, dnm);
    const int nintr = group_sum<G>((other && dnm < 5.0f) ? 1 : 0);
    const float dr = fabsf(drift * kDeg2Rad);
    s.drift_sum += dr; s.drift_n += 1;
    s.intrusions += nintr;
    o.reward = dr * -0.1f - (float)nintr;
    s.total_reward += o.reward;
    // truncation: ownship left the polygon (sector_cr_env.py:134-139); one edge per lane
    const double* poly = P.poly + e * (2 * kSectorMaxV);
    int cross = 0;
    if (slot < s.nvert) {
        int k2 = (slot + 1 == s.nvert) ? 0 : slot + 1;
        double x1 = poly[2 * slot], y1 = poly[2 * slot + 1], x2 = poly[2 * k2], y2 = poly[2 * k2 + 1];
        if ((y1 > lon0) != (y2 > lon0)) cross = lat0 < x1 + (lon0 - y1) * (x2 - x1) / (y2 - y1) ? 1 : 0;
    }
    o.truncated = (group_sum<G>(cross) & 1) ? 0 : 1;
    return o;
}

// =====================================================================================================
// MergeEnv (merge_env.py) -- G = 32, slot 0 ownship + 19 FMS-guided intruders (FIX -> RWY)
// =====================================================================================================
template <int G>
__device__ inline void merge_reset(Ac& a, EnvS& s, const EnvParams& P, long long e, int slot) {
    Philox rng = make_philox(P.seed, P.gid0 + e, (uint32_t)s.episode);      // merge_env.py:103-130,148-158
    const int nac = 20;
    if (slot < nac) {
        double brg = rng.uniform(2u * slot, -15.0, 15.0);
        double dist = slot == 0 ? rng.uniform(1u, 50.0, 200.0) : rng.uniform(2u * slot + 1u, 20.0, 500.0);
        double lat, lon;
        d_point_at_distance(P.fix_lat, P.fix_lon, dist, brg, lat, lon);
        ac_create_tas(a, lat, lon, brg - 180.0, 10000.0, 100.0, P.init_tas0);
        if (slot > 0) {     // "INTi addwpt FIX" -> Route.direct + LNAV on; "INTi dest RWY" appends the last wp
            float q, dm;
            qdrdist_wgs(a.lat, a.lon, P.fix_lat, P.fix_lon, q, dm);
            a.curlegdir = q;
            a.flags |= kFlLnav;
        }
    } else {
        ac_clear(a);
    }
    s.wpt_reach = 0; s.faf = 0; s.total_reward = 0.0f; s.intrusions = 0; s.drift_sum = 0.0f; s.drift_n = 0;
    s.num_ac = nac;
}
template <int G>
__device__ inline void merge_action(Ac& a, const EnvParams& P, const float* act, int slot) {
    if (slot == 0) {                                                        // merge_env.py:286-293
        a.aptrk = wrap180_fold(fmaf(act[0], 15.0f, a.hdg));
        a.flags &= ~kFlLnav;
        float kt = fmaf(act[1], 20.0f, a.cas) * 1.94384f;
        a.selspd = (kt > 0.1f && kt < 1.0f) ? kt : kt * kKts;
    }
}
template <int G>
__device__ inline StepOut merge_obs_reward(const Ac& a, EnvS& s, const EnvParams& P, float* obs, int slot,
                                           bool with_reward) {
    const double lat0 = group_bcast<G>(a.lat, 0), lon0 = group_bcast<G>(a.lon, 0);     // merge_env.py:160-236
    const float hdg0 = group_bcast<G>(a.hdg, 0), tas0 = group_bcast<G>(a.tas, 0);
    // cos / sin(hdg) * tas: the cached ground-speed components are exactly that without wind; with wind they carry
    // the wind vector, which the reference's observation does not include (it uses bs.traf.hdg and bs.traf.tas)
    float avx = a.gsn, avy = a.gse;
    if (P.wind_n > 0) { float sh_, ch_; sincosf(a.hdg * kDeg2Rad, &sh_, &ch_); avx = a.tas * ch_; avy = a.tas * sh_; }
    const float vx0 = group_bcast<G>(avx, 0), vy0 = group_bcast<G>(avy, 0);
    float wq, wd;
    if (s.wpt_reach == 0) kwikqdrdist(lat0, lon0, P.fix_lat, P.fix_lon, wq, wd);
    else kwikqdrdist(lat0, lon0, kRwyLat, kRwyLon, wq, wd);
    const float drift = wrap180_fold(hdg0 - wq);
    if (slot == 0) {
        float sd, cd;
        sincos_deg(drift, sd, cd);
        obs[0] = cd; obs[1] = sd; obs[2] = tas0; obs[3] = wd * (1.0f / 250.0f); obs[4] = (float)s.wpt_reach;
    }
    const bool other = slot >= 1 && slot < s.num_ac;
    float brg = 0.0f, dnm = 1e9f;
    if (other) kwikqdrdist(lat0, lon0, a.lat, a.lon, brg, dnm);
    int rank = nearest_rank<G>(dnm, other, 5);
    if (rank >= 0) {
        float sb, cb;
        sincos_deg(brg, sb, cb);
        float dm = dnm * 1852.0f;
        float dvx = avx - vx0, dvy = avy - vy0;
        float hyp = sqrtf(dvx * dvx + dvy * dvy);
        float ct = hyp > 0.0f ? dvx / hyp : 1.0f, st = hyp > 0.0f ? dvy / hyp : 0.0f;
        obs[5 + rank] = dm * cb * 1e-6f;
        obs[10 + rank] = dm * sb * 1e-6f;
        obs[15 + rank] = dvx * (1.0f / 150.0f);
        obs[20 + rank] = dvy * (1.0f / 150.0f);
        obs[25 + rank] = ct;
        obs[30 + rank] = st;
        obs[35 + rank] = dnm * (1.0f / 250.0f);
    }
    StepOut o = {0.0f, 0, 0};
    if (!with_reward) return o;
    float r = 0.0f;                                                         // merge_env.py:246-284
    if (wd < 10.0f && s.wpt_reach != 1) { s.wpt_reach = 1; s.faf = 1; r += 1.0f; }
    else if (wd < 20.0f && s.wpt_reach == 1) { s.faf = 2; o.terminated = 1; }
    const float dr = fabsf(drift * kDeg2Rad);
    s.drift_sum += dr; s.drift_n += 1;
    r += dr * -0.1f;
    const int nintr = group_sum<G>((other && dnm < 4.0f) ? 1 : 0);
    s.intrusions += nintr;
    r -= (float)nintr;
    s.total_reward += r;
    o.reward = r;
    return o;
}
__device__ inline void merge_info(const EnvS& s, float* info) {             // merge_env.py:238-244
    info[0] = s.total_reward; info[1] = (float)s.faf; info[2] = s.drift_sum / (float)s.drift_n; info[3] = (float)s.intrusions;
}

// =====================================================================================================
// PlanWaypointEnv (plan_waypoint_env.py) -- 1 aircraft, 5 waypoints, G = 1
// =====================================================================================================
template <int G>
__device__ inline void planwp_reset(Ac& a, EnvS& s, const EnvParams& P, long long e, int slot) {
    Philox rng = make_philox(P.seed, P.gid0 + e, (uint32_t)s.episode);      // plan_waypoint_env.py:157-172,200-213
    double hdg = P.hdg_random ? (double)rng.randint(0, 1, 360) : 0.0;
    if (slot == 0) ac_create_tas(a, 52.0, 4.0, hdg, 0.0, 150.0, P.init_tas0); else ac_clear(a);
    double* w = P.ef64 + e * BSG_F64_COUNT + BSG_F64_WPTS;
    for (int k = 0; k < 5; ++k) {
        int dis = rng.randint(1u + 2u * k, 0, 75), brg = rng.randint(2u + 2u * k, 0, 359);
        d_point_at_distance(52.0, 4.0, (double)dis, (double)brg, w[2 * k], w[2 * k + 1]);
    }
    s.wpt_reach = 0; s.total_reward = 0.0f; s.num_ac = 1;
}
template <int G>
__device__ inline StepOut planwp_obs_reward(const Ac& a, EnvS& s, const EnvParams& P, float* obs, int slot,
                                            long long e, bool with_reward) {
    const double* w = P.ef64 + e * BSG_F64_COUNT + BSG_F64_WPTS;            // plan_waypoint_env.py:82-124
    StepOut o = {0.0f, 0, 0};
    int reach = s.wpt_reach;
    for (int k = 0; k < 5; ++k) {
        float q, dnm;
        kwikqdrdist(a.lat, a.lon, w[2 * k], w[2 * k + 1], q, dnm);
        float dkm = dnm * 1.852f, sd, cd;
        sincos_deg(wrap180_fold(a.hdg - q), sd, cd);
        const float live = (s.wpt_reach >> k) & 1 ? 0.0f : 1.0f;           // flags from BEFORE this step's check
        obs[k] = live * dkm * (1.0f / 75.0f);
        obs[5 + k] = live * cd;
        obs[10 + k] = live * sd;
        obs[15 + k] = 1.0f - live;
        if (with_reward && dkm < 5.0f && !((reach >> k) & 1)) { reach |= 1 << k; o.reward += 1.0f; }   // :215-228
    }
    if (with_reward) {
        s.wpt_reach = reach;
        s.total_reward += o.reward;
        o.terminated = (reach == 31) ? 1 : 0;
    }
    return o;
}

// =====================================================================================================
// VerticalCREnv (vertical_cr_env.py) -- DescentEnv + 5 creconfs intruders with an altitude offset, G = 8
// =====================================================================================================
template <int G>
__device__ inline void vertical_reset(Ac& a, EnvS& s, const EnvParams& P, long long e, int slot) {
    Philox rng = make_philox(P.seed, P.gid0 + e, (uint32_t)s.episode);      // vertical_cr_env.py:258-281
    const int alt_init = rng.randint(0, 2000, 4000);
    const double target = (double)(alt_init + rng.randint(1, -500, 500));
    const double hdg0 = P.hdg_random ? (double)rng.randint(2, 1, 360) : 0.0;
    const double lat0 = 52.0, lon0 = 4.0, alt0 = (double)alt_init;
    // (the ownship's TAS from the host-evaluated float64 table: the float64 pow chains were 8 us of dependent latency at the
    // tail of every launch with a finishing env; the intruders' commanded CAS below in float32, the precision of that state)
    const double tas0 = g_tas150_tab[alt_init - 2000];
    s.target_alt = target;
    if (slot == 0) {
        ac_create_tas(a, lat0, lon0, hdg0, alt0, 150.0, tas0);
    } else if (slot <= 5) {                                                  // _generate_conflicts :185-200
        const uint32_t d = 3u + 4u * (uint32_t)(slot - 1);
        double dpsi = (double)rng.randint(d, 45, 315);
        double cpa = (double)rng.randint(d + 1, 0, 5) * 1852.0;
        double tlosh = (double)rng.randint(d + 2, 100, (int)((200.0 * 0.9) * 1000.0 / tas0));
        double average_tod = (200.0 * 1000.0 / tas0) - 2.0 * target / 12.5;
        int dH;
        if (tlosh > average_tod) dH = rng.randint(d + 3, (int)(-alt0 + 500.0), (int)((target - alt0) + 100.0));
        else dH = rng.randint(d + 3, (int)((target - alt0) - 500.0), (int)((target - alt0) + 500.0));
        // Traffic.creconfs with dH, tlosv = 1e11 (oracle/traffic.py::creconfs)
        const double pzr = 5.0 * 1852.0, pzh = 1000.0 * 0.3048;
        double trkref = hdg0 * kDeg2RadD, gsref = tas0;
        double trk = trkref + dpsi * kDeg2RadD;
        double acalt = alt0 + (double)dH;
        double sgn = dH > 0 ? 1.0 : (dH < 0 ? -1.0 : 0.0);
        double acvs = 0.0 - sgn * (fabs((double)dH) - pzh) / 1e11;
        double gsn = gsref * cos(trk), gse = gsref * sin(trk);
        double vreln = gsref * cos(trkref) - gsn, vrele = gsref * sin(trkref) - gse;
        double vrel = sqrt(vreln * vreln + vrele * vrele);
        double drelcpa = tlosh * vrel + (cpa > pzr ? 0.0 : sqrt(pzr * pzr - cpa * cpa));
        double dist = sqrt(drelcpa * drelcpa + cpa * cpa);
        double rd = drelcpa / dist, rx = cpa / dist;
        double brn = kRad2DegD * atan2(-rx * vreln + rd * vrele, rd * vreln + rx * vrele);
        double dnm = dist / 1852.0;
        double lat = lat0 + dnm * cos(brn * kDeg2RadD) / 60.0;
        double lon = lon0 + dnm * sin(brn * kDeg2RadD) / fmax(0.01, 60.0 * cos(lat0 * kDeg2RadD));
        lon = fmod(lon + 180.0, 360.0); if (lon < 0.0) lon += 360.0; lon -= 180.0;
        // upstream: acspd = vtas2cas(gs, acalt), then cre: tas = vcas2tas(acspd, acalt) -- the round trip is the identity
        const double gs = sqrt(gsn * gsn + gse * gse);
        const double acspd = (double)tas2cas((float)gs, vatmos((float)acalt));
        ac_create_tas(a, lat, lon, kRad2DegD * atan2(gse, gsn), acalt, acspd, gs);
        a.vs = (float)acvs;                 // creconfs: vs[-1] = acvs; the env then selaltcmd(alt + dH, 0)
        a.selalt = (float)acalt; a.selvs = 0.0f;
    } else {
        ac_clear(a);
    }
    s.total_reward = 0.0f; s.intrusions = 0; s.final_alt = 0.0f; s.num_ac = 6;
}
template <int G>
__device__ inline StepOut vertical_obs_reward(const Ac& a, EnvS& s, const EnvParams& P, float* obs, int slot,
                                              bool with_reward) {
    const double lat0 = group_bcast<G>(a.lat, 0), lon0 = group_bcast<G>(a.lon, 0);     // vertical_cr_env.py:114-183
    const float gs_own = ac_gs(a, P);
    const float hdg0 = group_bcast<G>(a.hdg, 0), gs0 = group_bcast<G>(gs_own, 0);
    const float alt0 = group_bcast<G>(a.alt, 0), vs0 = group_bcast<G>(a.vs, 0);
    float q, dnm;
    kwikqdrdist(52.0, 4.0, lat0, lon0, q, dnm);
    const float rwy = 200.0f - dnm * 1.852f;
    const float tgt = (float)s.target_alt;
    if (slot == 0) {
        obs[0] = (alt0 - 1500.0f) * (1.0f / 3000.0f);
        obs[1] = vs0 * 0.2f;
        obs[2] = (tgt - 1500.0f) * (1.0f / 3000.0f);
        obs[3] = (rwy - 100.0f) * (1.0f / 200.0f);
    }
    const bool intr = slot >= 1 && slot <= 5;
    float dis = 1e9f;
    if (intr) {
        float dn, de, ang, sd, cd, sh0, ch0;                         // (as in horizontal_obs_reward: no atan2 / sincos round trip)
        kwikoffsets(lat0, lon0, a.lat, a.lon, dn, de, ang, dis);
        __sincosf((hdg0 - 180.0f) * kDeg2Rad, &sh0, &ch0);
        sh0 = -sh0; ch0 = -ch0;
        const float inv = ang > 0.0f ? 1.0f / ang : 0.0f;
        const float cq = ang > 0.0f ? dn * inv : 1.0f, sq = de * inv;
        const float cb = fmaf(ch0, cq, sh0 * sq), sb = fmaf(sh0, cq, -ch0 * sq);
        sincos_deg((hdg0 - a.hdg), sd, cd);
        const int k = slot - 1;
        obs[4 + k] = dis * (1.852f / 200.0f);
        obs[9 + k] = cb;
        obs[14 + k] = sb;
        obs[19 + k] = (a.alt - alt0) * (1.0f / 3000.0f);
        obs[24 + k] = -cd * gs_own * (1.0f / 150.0f);
        obs[29 + k] = (gs0 - sd * gs_own) * (1.0f / 150.0f);
        obs[34 + k] = a.vs - vs0;
    }
    StepOut o = {0.0f, 0, 0};
    if (!with_reward) return o;
    const int nintr = group_sum<G>((intr && dis < 5.0f && fabsf(alt0 - a.alt) < 1000.0f * 0.3048f) ? 1 : 0);   // :213-240
    s.intrusions += nintr;
    float pen;
    if (rwy > 0.0f && alt0 > 0.0f) {
        pen = fabsf(tgt - alt0) * (-5.0f / 3000.0f);
    } else if (alt0 <= 0.0f) {
        pen = -100.0f; o.terminated = 1; s.final_alt = -100.0f;
    } else {
        pen = alt0 * (-50.0f / 3000.0f); o.terminated = 1; s.final_alt = alt0;
    }
    o.reward = pen - 50.0f * (float)nintr;
    s.total_reward += o.reward;
    return o;
}

// =====================================================================================================
// StaticObstacleEnv (static_obstacle_env.py) -- G = 16: lane 0 flies the aircraft, lanes 0..9 each own one
// polygon no-fly area.  poly record per env (doubles): [0,320) vertices [10][16][lat,lon]; [320,340) centres;
// [340,350) radius NM; [350,360) vertex counts.
// =====================================================================================================
constexpr int kObsN = 10, kObsMaxV = 16, kObsCentre = 320, kObsRadius = 340, kObsNv = 350, kObsPoly = 360;

__device__ inline void d_kwikqdrdist(double lata, double lona, double latb, double lonb, double& qdr, double& dnm) {
    double dlat = (latb - lata) * kDeg2RadD;
    double dlon = (dmod360((lonb - lona) + 180.0) - 180.0) * kDeg2RadD;
    double cav = cos((lata + latb) * (0.5 * kDeg2RadD));
    dnm = 6371000.0 * sqrt(dlat * dlat + dlon * dlon * cav * cav) / 1852.0;
    qdr = dmod360(kRad2DegD * atan2(dlon * cav, dlat));
}
template <int G>
__device__ inline int obstacles_hit(double lat, double lon, const double* pe, int slot) {
    int inside = 0;                                   // areafilter.checkInside, one obstacle per lane
    if (slot < kObsN) inside = d_inside_poly(lat, lon, pe + slot * (2 * kObsMaxV), (int)pe[kObsNv + slot]) ? 1 : 0;
    return group_sum<G>(inside);
}
// Scenario generator spread over the group's 16 lanes (serial, it was ~150 us of dependent float64 trigonometry on one
// lane and, with ~2 % of the envs resetting in any step, set the duration of every launch).  Draw order of the reference
// kept: [cre heading] | 10 x (distance, bearing) of the obstacle centres | per obstacle: area draw, then one draw per
// polygon point until the polygon is large enough | (distance, bearing) tries for the waypoint.  Per obstacle the 16
// candidate points are evaluated by the 16 lanes at once; lane 0 only does the cheap insertion / shoelace loop that
// decides how many of them are used.  scratch per group (float64): [0,16) cand x | [16,32) cand y | [32,48) cand angle.
constexpr int kStaticScratch = 48;

template <int G>
__device__ inline void static_reset(Ac& a, EnvS& s, const EnvParams& P, long long e, int slot, double* scratch) {
    double* pe = P.poly + e * kObsPoly;
    double* c_x = scratch, *c_y = scratch + 16, *c_a = scratch + 32;
    const double lat0 = 52.0, lon0 = 4.0;
    const Philox rng = make_philox(P.seed, P.gid0 + e, (uint32_t)s.episode);      // static_obstacle_env.py:96-131
    uint32_t d = P.hdg_random ? 1u : 0u;                                    // cre's heading draw (overwritten below)
    int rflags = 0;
    if (slot < kObsN) {                                                     // centres :221-232, one per lane
        const int dis = rng.randint(d + 2u * slot, 20, 150), brg = rng.randint(d + 2u * slot + 1u, 0, 360);
        d_point_at_distance(lat0, lon0, (double)dis, (double)brg, pe[kObsCentre + 2 * slot], pe[kObsCentre + 2 * slot + 1]);
    }
    d += 2u * kObsN;
    __syncwarp(group_mask<G>());
    for (int i = 0; i < kObsN; ++i) {                                       // _generate_polygon :156-169
        const double R = sqrt((double)rng.randint(d++, 100, 1000) / 3.141592653589793);
        if (slot < kObsMaxV) {                                              // candidate point `slot` of this obstacle
            const double al = 6.283185307179586 * rng.u01(d + (uint32_t)slot);
            const double x = R * cos(al), y = R * sin(al);
            c_x[slot] = x; c_y[slot] = y; c_a[slot] = atan2(y, x);
        }
        __syncwarp(group_mask<G>());
        int nv = 0;
        if (slot == 0) {
            double vx[kObsMaxV], vy[kObsMaxV], va[kObsMaxV];
            auto insert_point = [&]() {
                const double x = c_x[nv], y = c_y[nv], ang = c_a[nv];
                int k = nv;
                while (k > 0 && va[k - 1] > ang) { vx[k] = vx[k - 1]; vy[k] = vy[k - 1]; va[k] = va[k - 1]; --k; }
                vx[k] = x; vy[k] = y; va[k] = ang; ++nv;
            };
            auto shoelace = [&]() {
                double acc = 0.0;
                for (int q = 0; q < nv; ++q) { int r = (q + 1 == nv) ? 0 : q + 1; acc += vx[q] * vy[r] - vy[q] * vx[r]; }
                return fabs(acc) / 2.0;
            };
            insert_point(); insert_point(); insert_point();
            double area = shoelace();
            while (area < 50.0 && nv < kObsMaxV) { insert_point(); area = shoelace(); }
            if (area < 50.0) rflags |= 1;
            const double clat = pe[kObsCentre + 2 * i], clon = pe[kObsCentre + 2 * i + 1];
            const double cc = cos(clat * kDeg2RadD);
            for (int q = 0; q < nv; ++q) {                                  // nm_to_latlong(centre, point)
                pe[i * (2 * kObsMaxV) + 2 * q] = clat + vx[q] / 60.0;
                pe[i * (2 * kObsMaxV) + 2 * q + 1] = clon + vy[q] / (60.0 * cc);
            }
            pe[kObsRadius + i] = R;
            pe[kObsNv + i] = (double)nv;
        }
        nv = group_bcast<G>(nv, 0);
        d += (uint32_t)nv;
        __syncwarp(group_mask<G>());                                        // candidates are rewritten for the next obstacle
    }
    rflags = group_bcast<G>(rflags, 0);
    double wlat = 0.0, wlon = 0.0;                                          // _generate_waypoint :198-219
    for (int loops = 1;; ++loops) {
        const int dis = rng.randint(d, 100, 170), brg = rng.randint(d + 1u, 0, 360);
        d += 2u;
        d_point_at_distance(lat0, lon0, (double)dis, (double)brg, wlat, wlon);      // (every lane: same inputs, same result)
        if (obstacles_hit<G>(wlat, wlon, pe, slot) == 0) break;             // one obstacle per lane
        if (loops > 1000) { rflags |= 4; break; }
    }
    double hdg = 0.0, dnm;
    d_kwikqdrdist(lat0, lon0, wlat, wlon, hdg, dnm);                        // hdg = ap.trk = initial_wpt_qdr
    if (slot == 0) ac_create_tas(a, lat0, lon0, hdg, 350.0, 150.0, P.init_tas0); else ac_clear(a);
    s.wpt_lat = wlat; s.wpt_lon = wlon; s.rflags = rflags;
    s.wpt_reach = 0; s.intrusions = 0; s.total_reward = 0.0f; s.drift_sum = 0.0f; s.drift_n = 0; s.num_ac = 1;
}
// static_obstacle_env.py:294-341 after every bs.sim.step(); returns true when the episode ends
template <int G>
__device__ inline bool static_substep_check(const Ac& a, EnvS& s, const EnvParams& P, long long e, int slot) {
    const double lat0 = group_bcast<G>(a.lat, 0), lon0 = group_bcast<G>(a.lon, 0);
    const int nin = obstacles_hit<G>(lat0, lon0, P.poly + e * kObsPoly, slot);
    float r = 0.0f;
    if (s.last_wdist < 5.0f && s.wpt_reach != 1) { s.wpt_reach = 1; r += 1.0f; }      // distance / drift of the last _get_obs
    const float dr = fabsf(s.last_drift * kDeg2Rad);
    s.drift_sum += dr; s.drift_n += 1;
    r += dr * -0.01f;
    if (nin) { r += -5.0f * (float)nin; s.intrusions = 1; }
    s.step_reward = r;
    s.step_done = (s.wpt_reach == 1 || nin) ? 1 : 0;
    return s.step_done != 0;
}
template <int G>
__device__ inline void static_action(Ac& a, const EnvParams& P, const float* act, int slot) {
    if (slot == 0) {                                                        // static_obstacle_env.py:343-350
        a.aptrk = wrap180_fold(fmaf(act[0], 45.0f, a.hdg));
        a.flags &= ~kFlLnav;
        float kt = fmaf(act[1], 20.0f / 3.0f, a.cas) * 1.94384f;
        a.selspd = (kt > 0.1f && kt < 1.0f) ? kt : kt * kKts;
    }
}
template <int G>
__device__ inline StepOut static_obs_reward(const Ac& a, EnvS& s, const EnvParams& P, float* obs, int slot,
                                            long long e, bool with_reward) {
    const double* pe = P.poly + e * kObsPoly;                               // static_obstacle_env.py:234-283
    const double lat0 = group_bcast<G>(a.lat, 0), lon0 = group_bcast<G>(a.lon, 0);
    const float hdg0 = group_bcast<G>(a.hdg, 0);
    float wq, wd;
    kwikqdrdist(lat0, lon0, s.wpt_lat, s.wpt_lon, wq, wd);
    s.last_wdist = wd * 1.852f;
    s.last_drift = wrap180_fold(hdg0 - wq);
    if (slot == 0) {
        float sd, cd;
        sincos_deg(s.last_drift, sd, cd);
        obs[0] = s.last_wdist * (1.0f / 170.0f); obs[1] = cd; obs[2] = sd;
    }
    if (slot < kObsN) {
        float q, dnm, sb, cb;
        kwikqdrdist(lat0, lon0, pe[kObsCentre + 2 * slot], pe[kObsCentre + 2 * slot + 1], q, dnm);
        sincos_deg(wrap180_fold(hdg0 - q), sb, cb);
        obs[3 + slot] = (float)pe[kObsRadius + slot] * (1.0f / 50.0f);
        obs[13 + slot] = dnm * (1.852f / 170.0f);
        obs[23 + slot] = cb;
        obs[33 + slot] = sb;
    }
    StepOut o = {0.0f, 0, 0};
    if (!with_reward) return o;
    o.reward = s.step_reward;                          // the LAST substep's reward (static_obstacle_env.py:139-152)
    o.terminated = s.step_done;
    s.total_reward += o.reward;
    return o;
}

// =====================================================================================================
// dispatch helpers
// =====================================================================================================
template <int ENV, int G>
__device__ __forceinline__ void do_reset(Ac& a, EnvS& s, const EnvParams& P, long long e, int slot, double* scratch) {
    if (ENV == BSG_ENV_DESCENT) descent_reset<G>(a, s, P, e, slot);
    if (ENV == BSG_ENV_HORIZONTAL_CR) horizontal_reset<G>(a, s, P, e, slot);
    if (ENV == BSG_ENV_SECTOR_CR) sector_reset<G>(a, s, P, e, slot, scratch);
    if (ENV == BSG_ENV_MERGE) merge_reset<G>(a, s, P, e, slot);
    if (ENV == BSG_ENV_PLAN_WAYPOINT) planwp_reset<G>(a, s, P, e, slot);
    if (ENV == BSG_ENV_VERTICAL_CR) vertical_reset<G>(a, s, P, e, slot);
    if (ENV == BSG_ENV_STATIC_OBSTACLE) static_reset<G>(a, s, P, e, slot, scratch);
    s.step = 0; s.needs_reset = 0; s.episode += 1; s.nconf = 0; s.nlos = 0;
    if (P.cd_pairs && slot == 0) P.ei32[e * BSG_I32_COUNT + BSG_I32_NPAIRS] = 0;      // no detection yet in the new episode
}
template <int ENV, int G>
__device__ __forceinline__ StepOut do_obs(const Ac& a, EnvS& s, const EnvParams& P, float* obs, int slot, long long e,
                                          bool with_reward) {
    if (ENV == BSG_ENV_DESCENT) return descent_obs_reward<G>(a, s, P, obs, slot, with_reward);
    if (ENV == BSG_ENV_HORIZONTAL_CR) return horizontal_obs_reward<G>(a, s, P, obs, slot, with_reward);
    if (ENV == BSG_ENV_SECTOR_CR) return sector_obs_reward<G>(a, s, P, obs, slot, e, with_reward);
    if (ENV == BSG_ENV_PLAN_WAYPOINT) return planwp_obs_reward<G>(a, s, P, obs, slot, e, with_reward);
    if (ENV == BSG_ENV_VERTICAL_CR) return vertical_obs_reward<G>(a, s, P, obs, slot, with_reward);
    if (ENV == BSG_ENV_STATIC_OBSTACLE) return static_obs_reward<G>(a, s, P, obs, slot, e, with_reward);
    return merge_obs_reward<G>(a, s, P, obs, slot, with_reward);
}
// Env._get_info values of env e, stored key-major -- info[k * E + e] -- so that the host sees one contiguous row per key
template <int ENV>
__device__ __forceinline__ void do_info(const EnvS& s, const EnvParams& P, const int e) {
    float info[6];
    if (ENV == BSG_ENV_DESCENT) descent_info(s, info);
    else if (ENV == BSG_ENV_MERGE) merge_info(s, info);
    else if (ENV == BSG_ENV_PLAN_WAYPOINT) {            // plan_waypoint_env.py:126-133
        info[0] = s.total_reward; info[1] = (float)__popc((unsigned)s.wpt_reach); info[2] = 0.0f; info[3] = 0.0f;
    } else if (ENV == BSG_ENV_VERTICAL_CR) {            // vertical_cr_env.py:202-211
        info[0] = s.total_reward; info[1] = (float)s.intrusions; info[2] = s.final_alt; info[3] = 0.0f;
    } else if (ENV == BSG_ENV_STATIC_OBSTACLE) {        // static_obstacle_env.py:285-292
        info[0] = s.total_reward; info[1] = (float)s.wpt_reach; info[2] = (float)s.intrusions;
        info[3] = s.drift_sum / (float)s.drift_n;
    } else drift_info(s, info);
    info[4] = (float)s.nconf; info[5] = (float)s.nlos;
#pragma unroll
    for (int k = 0; k < 6; ++k) P.info[(long long)k * P.E + e] = info[k];
}

// =====================================================================================================
// K6: the env-step megakernel (also serves reset and the kinematics-only parity entry point)
// =====================================================================================================
template <int ENV, int G, bool WIND>
__global__ void __launch_bounds__(kEnvThreads, kEnvBlocksPerSm) env_kernel(const EnvParams P) {
    __shared__ GroupSmem<(G > 1) ? G : 2> s_grp[(G > 1) ? kEnvThreads / G : 1];
    __shared__ uint16_t s_pairs[(G > 1 && G <= 8) ? kSmallPairs : 1];
    if (G > 1 && G <= 8 && P.cd_enabled && P.mode != kModeReset) {
        build_pair_table(s_pairs);
        __syncthreads();
    }
    __shared__ double s_scratch[(ENV == BSG_ENV_SECTOR_CR) ? (kEnvThreads / 32) * kSectorScratch
                                : (ENV == BSG_ENV_STATIC_OBSTACLE) ? (kEnvThreads / G) * kStaticScratch : 1];
    const int tid = threadIdx.x;
    const int gt = blockIdx.x * kEnvThreads + tid;          // (E * G < 2^31: bsg_create checks)
    if (gt == 0 && P.mode == kModeStep && P.final_count) {
        // two counters take turns (no memset node between launches): this launch counts in [fc_slot], clears the other one
        // for the next launch and publishes which is live in [2]
        P.final_count[P.fc_slot ^ 1] = 0;
        P.final_count[2] = P.fc_slot;
    }
    const int e = gt / G;
    const int slot = gt % G;
    if (e >= P.E) return;                       // group-uniform (G divides the block size)
    double* scratch = (ENV == BSG_ENV_SECTOR_CR) ? &s_scratch[(threadIdx.x / 32) * kSectorScratch]
                    : (ENV == BSG_ENV_STATIC_OBSTACLE) ? &s_scratch[(threadIdx.x / G) * kStaticScratch] : s_scratch;
    // (group index made opaque: otherwise the compiler, short of registers, rebuilds the group's shared-memory address from
    // the thread index -- S2R, shift, multiply-add -- at most of the dozen places per substep that use it)
    int grp = (G > 1) ? tid / G : 0;
    asm volatile("" : "+r"(grp));
    auto& S = s_grp[grp];

    // Every load of the step is issued here, before anything waits on one of them: with the state cold in DRAM (the usual
    // case: 14 MB per batch touched once per env step) the aircraft record, the env counters and the actions arrive in ONE
    // memory round trip instead of three dependent ones, and the records read after the substep loop are on their way to L2.
    Ac a;
    ac_load(a, P, gt);
    float act[2] = {0.0f, 0.0f};
    if (P.mode == kModeStep) {
        act[0] = P.actions[(long long)e * P.act_dim];
        if (ENV == BSG_ENV_SECTOR_CR || ENV == BSG_ENV_MERGE || ENV == BSG_ENV_STATIC_OBSTACLE) act[1] = P.actions[(long long)e * P.act_dim + 1];
    }
    EnvS s;
    env_load_pre(s, P, e);
    if (slot == 0) {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(P.ef64 + (long long)e * BSG_F64_COUNT));
        asm volatile("prefetch.global.L2 [%0];" ::"l"(P.ef32 + (long long)e * BSG_F32_COUNT));
    }
    if (ENV == BSG_ENV_SECTOR_CR && slot < 4) asm volatile("prefetch.global.L2 [%0];" ::"l"(P.poly + (long long)e * (2 * kSectorMaxV) + 16 * slot));
    float* obs = P.obs + (long long)e * P.obs_dim;

    // One control flow for reset / step / autoreset so that the scenario generator and the observation
    // code exist ONCE in the kernel (they are big; duplicating them blew the instruction cache).
    bool resetting;
    if (P.mode == kModeReset) {
        resetting = P.reset_mask ? (P.reset_mask[e] != 0) : true;
        if (!resetting) return;
    } else {
        resetting = (P.mode == kModeStep) && (P.autoreset == BSG_AUTORESET_NEXT_STEP) && (s.needs_reset != 0);
    }

    if (!resetting) {
        ac_finish_load(a, P);
        const bool alive = (a.flags & kFlAlive) != 0;
        // The targets of the last launch (ISA / CAS conversions: ~400 instructions of pow-type arithmetic) stay valid while
        // what they are a function of -- alt, vs, selspd, selalt -- stays put: the record carries allow_tas with a valid bit
        // that the end of a launch sets when its last targets belong to the stored (alt, vs), and that an action which
        // moves selspd / selalt clears.  Same inputs, same function: the cached value is the recomputed one bit for bit.
        bool tgt_cached = (P.mode == kModeStep && (a.flags & kFlTgt) != 0) || !alive;   // (empty slots: nothing to compute)
        if (P.mode == kModeStep) {
            const float o_selspd = a.selspd, o_selalt = a.selalt;
            if (ENV == BSG_ENV_DESCENT || ENV == BSG_ENV_VERTICAL_CR) descent_action<G>(a, P, act, slot);
            if (ENV == BSG_ENV_PLAN_WAYPOINT) horizontal_action<G>(a, P, act, slot);
            if (ENV == BSG_ENV_STATIC_OBSTACLE) static_action<G>(a, P, act, slot);
            if (ENV == BSG_ENV_HORIZONTAL_CR) horizontal_action<G>(a, P, act, slot);
            if (ENV == BSG_ENV_SECTOR_CR) sector_action<G>(a, P, act, slot);
            if (ENV == BSG_ENV_MERGE) merge_action<G>(a, P, act, slot);
            tgt_cached = tgt_cached && a.selspd == o_selspd && a.selalt == o_selalt;
            if (WIND && ENV != BSG_ENV_DESCENT && ENV != BSG_ENV_VERTICAL_CR && slot == 0 && a.alt > 50.0f * kFt) {
                // Autopilot.selhdgcmd with wind: the commanded HEADING becomes the track it produces right now
                float wn, we, sh, ch;
                wind_at(P, a.lat, a.lon, a.alt, wn, we);
                sincosf(a.aptrk * kDeg2Rad, &sh, &ch);
                a.aptrk = mod360(kRad2Deg * atan2f(fmaf(a.tas, sh, we), fmaf(a.tas, ch, wn)));
            }
        }
        int nconf = s.nconf, nlos = s.nlos;
        if (G > 8 && P.cd_enabled) {
            if (slot == 0) S.nb = -1;
            __syncwarp(group_mask<G>());
        }
        // (the envs whose action reads traf.cas convert tas -> cas after the loop and need the atmosphere for it)
        constexpr bool kNeedAtmos = ENV == BSG_ENV_SECTOR_CR || ENV == BSG_ENV_MERGE || ENV == BSG_ENV_STATIC_OBSTACLE;
        Targets T;
        compute_targets<kNeedAtmos>(a, P, T, tgt_cached);
        // `fixed`: the last full kinematics update left (tas, hdg, vs, alt, ax, ground-speed components) exactly as they
        // were.  They are a pure function of themselves, the targets T (recomputed only when alt / vs move) and the
        // commands (which change only between env steps, or through LNAV in MergeEnv, or with the wind): the next update
        // would reproduce them bit for bit, so while EVERY aircraft of the env is fixed -- intruders always, the ownship
        // once it has finished its turn -- a substep only advances the positions, with the very expressions of
        // ac_kinematics.
        bool fixed = false;
        bool moved = false;                                 // the ground-speed vector changed in the last update (K3's (B) list)
#pragma unroll 1
        for (int k = 0; k < P.n_sub; ++k) {                 // n_sub x bs.sim.step()
            s.simk += 1;
            const bool fms_ready = ENV == BSG_ENV_MERGE && (s.simk % P.fms_rel_freq) == 0;
            if (alive) {
                if (a.alt != T.k_alt || a.vs != T.k_vs) compute_targets<true>(a, P, T, false);
                ac_autopilot<ENV>(a, P, fms_ready);
            }
            if constexpr (G > 1) if (P.cd_enabled) {
                const bool emit = P.cd_pairs != nullptr && (k == P.n_sub - 1 || ENV == BSG_ENV_STATIC_OBSTACLE);
                // metric origin of the CD records: a fixed point of the env's airspace (aircraft stay within a few hundred km
                // of it: float32 metres resolve 3 cm there), so no per-substep broadcast of the ownship position is needed
                const double lat_ref = ENV == BSG_ENV_MERGE ? P.fix_lat : (ENV == BSG_ENV_SECTOR_CR ? kSectorLat0 : 52.0);
                const double lon_ref = ENV == BSG_ENV_MERGE ? P.fix_lon : (ENV == BSG_ENV_SECTOR_CR ? kSectorLon0 : 4.0);
                group_cd<G, ENV == BSG_ENV_MERGE || WIND>(S, slot, a, alive, s.num_ac, P, (float)(P.n_sub - 1 - k) * P.simdt, s_pairs, nconf,
                                                          nlos, emit, e, moved, lat_ref, lon_ref);
                if (emit && slot == 0) P.ei32[(long long)e * BSG_I32_COUNT + BSG_I32_NPAIRS] = S.np;
            }
            if (!WIND && ENV != BSG_ENV_MERGE && group_all<G>(fixed || !alive)) {
                moved = false;
                if (alive) {                                // update_pos alone (same expressions as ac_kinematics)
                    a.lat += (double)(kRad2Deg * (P.simdt * a.gsn * (1.0f / kRearth)));
                    a.coslat = __cosf((float)a.lat * kDeg2Rad);
                    a.lon += (double)(kRad2Deg * (P.simdt * a.gse * rcp_approx(a.coslat) * (1.0f / kRearth)));
                }
            } else if (alive) {
                const float o_tas = a.tas, o_hdg = a.hdg, o_vs = a.vs, o_alt = a.alt, o_ax = a.ax, o_gsn = a.gsn, o_gse = a.gse;
                ac_kinematics<WIND>(a, P, T);
                moved = a.gsn != o_gsn || a.gse != o_gse;
                fixed = !moved && a.tas == o_tas && a.hdg == o_hdg && a.vs == o_vs && a.alt == o_alt && a.ax == o_ax;
            }
            if (ENV == BSG_ENV_STATIC_OBSTACLE && P.mode == kModeStep) {   // per-substep reward / termination
                if (k == 0) env_load_post(s, P, e);
                if (static_substep_check<G>(a, s, P, e, slot)) break;
            }
        }
        // update_airspeed's cas = vtas2cas(tas, alt) uses the altitude from before update_pos: T.at of the last substep
        // (only the envs whose action reads traf.cas need it: Sector, Merge, StaticObstacle)
        if ((kNeedAtmos || P.mode == kModeTraf) && alive && P.n_sub > 0) {
            a.cas = tas2cas(a.tas, T.at);
        }
        // targets cache for the next launch: valid when the last targets belong to the state that is stored
        a.tgt = T.allow_tas;
        a.flags = (alive && T.k_alt == a.alt && T.k_vs == a.vs) ? (a.flags | kFlTgt) : (a.flags & ~kFlTgt);
        s.nconf = nconf; s.nlos = nlos;
        if (P.mode == kModeTraf) {
            ac_store(a, P, gt);
            if (slot == 0) env_store_pre(s, P, e);
            return;
        }
        if (ENV != BSG_ENV_STATIC_OBSTACLE) env_load_post(s, P, e);
    }

#pragma unroll 1
    for (int pass = 0; pass < 2; ++pass) {
        const bool fresh = resetting;                    // this pass starts from a newly generated scenario
        if (resetting) do_reset<ENV, G>(a, s, P, e, slot, scratch);
        StepOut o = do_obs<ENV, G>(a, s, P, obs, slot, e, !fresh);
        if (P.wind_obs && slot == 0) {                   // wrappers/wind.py:55-64 (_get_wind_observation)
            float wn = 0.0f, we = 0.0f, sh, ch;
            if (WIND) wind_at(P, a.lat, a.lon, a.alt, wn, we);
            sincosf(a.hdg * kDeg2Rad, &sh, &ch);
            obs[P.obs_dim - 2] = (wn * ch + we * sh) * (1.0f / 50.0f);
            obs[P.obs_dim - 1] = (-wn * sh + we * ch) * (1.0f / 50.0f);
        }
        if (pass == 1) break;                            // SAME_STEP: the step's reward / flags / info stay
        if (fresh) {
            if (slot == 0) { P.reward[e] = 0.0f; P.term[e] = 0; P.trunc[e] = 0; do_info<ENV>(s, P, e); }
            break;
        }
        s.step += 1;
        if (P.max_steps > 0 && s.step >= P.max_steps) o.truncated = 1;      // gymnasium TimeLimit
        if (slot == 0) {
            P.reward[e] = o.reward; P.term[e] = (uint8_t)o.terminated; P.trunc[e] = (uint8_t)o.truncated;
            do_info<ENV>(s, P, e);
        }
        if (!(o.terminated || o.truncated)) break;
        if (P.autoreset == BSG_AUTORESET_NEXT_STEP) { s.needs_reset = 1; break; }
        if (P.autoreset != BSG_AUTORESET_SAME_STEP) break;
        if (P.final_obs) {                               // the terminal observation survives, compacted
            int k = 0;
            if (slot == 0) { k = atomicAdd(P.final_count + P.fc_slot, 1); P.final_ids[k] = (int32_t)e; }
            k = group_bcast<G>(k, 0);
            __syncwarp(group_mask<G>());
            float* fo = P.final_obs + (long long)k * P.obs_dim;
            for (int i = slot; i < P.obs_dim; i += G) fo[i] = obs[i];
            __syncwarp(group_mask<G>());
        }
        resetting = true;
    }
    ac_store(a, P, gt);
    if (slot == 0) env_store(s, P, e);
}

}  // namespace bsg

using namespace bsg;

int bsg_upload_tas150_table(const double* h_tab) {
    return bsg_cuda_check(cudaMemcpyToSymbol(g_tas150_tab, h_tab, sizeof(double) * 2001), "tas table upload");
}

template <int ENV, int G>
static int launch_env_t(const EnvParams& P, cudaStream_t st) {
    long long threads = (long long)P.E * G;
    int blocks = (int)((threads + kEnvThreads - 1) / kEnvThreads);
    if (blocks == 0) return BSG_OK;
    if (P.wind_n > 0) env_kernel<ENV, G, true><<<blocks, kEnvThreads, 0, st>>>(P);
    else env_kernel<ENV, G, false><<<blocks, kEnvThreads, 0, st>>>(P);
    return bsg_cuda_check(cudaGetLastError(), "env_kernel launch");
}

int bsg_launch_env(const EnvParams& P, int slots, cudaStream_t st) {
    switch (P.env_type) {
        case BSG_ENV_DESCENT:
            return launch_env_t<BSG_ENV_DESCENT, 1>(P, st);
        case BSG_ENV_HORIZONTAL_CR:
            if (slots == 8) return launch_env_t<BSG_ENV_HORIZONTAL_CR, 8>(P, st);
            if (slots == 16) return launch_env_t<BSG_ENV_HORIZONTAL_CR, 16>(P, st);
            return launch_env_t<BSG_ENV_HORIZONTAL_CR, 32>(P, st);
        case BSG_ENV_SECTOR_CR:
            return launch_env_t<BSG_ENV_SECTOR_CR, 32>(P, st);
        case BSG_ENV_MERGE:
            return launch_env_t<BSG_ENV_MERGE, 32>(P, st);
        case BSG_ENV_PLAN_WAYPOINT:
            return launch_env_t<BSG_ENV_PLAN_WAYPOINT, 1>(P, st);
        case BSG_ENV_VERTICAL_CR:
            return launch_env_t<BSG_ENV_VERTICAL_CR, 8>(P, st);
        case BSG_ENV_STATIC_OBSTACLE:
            return launch_env_t<BSG_ENV_STATIC_OBSTACLE, 16>(P, st);
    }
    return bsg_fail(BSG_EINVAL, "unknown env_type");
}
