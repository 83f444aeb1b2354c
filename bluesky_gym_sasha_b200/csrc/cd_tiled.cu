// cd_tiled.cu -- K2: single-airspace state-based conflict detection, tiled all-pairs (n-body style).
// Replaces the dense N x N float64 matrices of bluesky/traffic/asas/statebased.py::StateBased.detect
// (upstream's optional single-threaded C++ twin is `cstatebased`); O(N) memory instead of ~15 N^2.
//
// Bound: FP32 issue rate.  Measured on B200 (scripts/pipe_probe.cu): FFMA and ALU-pipe ops (FMNMX, FSETP,
// FSEL, LOP3) share one issue port per SM sub-partition at 1 warp-instruction/clk; the packed FFMA2 /
// FADD2 / FMUL2 (f32x2, new on sm_100) occupy the FMA pipe for 2 clk but only ONE issue slot, so the
// comparison / select / MUFU work of a pair can issue underneath the packed arithmetic of the next.
// The hot loop is therefore written in f32x2: one thread owns R = 2 rows and evaluates them against
// column *pairs* (j, j+1): 26 packed FMA-pipe ops per two pairs + 13 scalar ALU/MUFU ops per pair
// (~28 issue slots and 26 FMA-pipe clk per ordered pair, vs 56 issue slots for the scalar formulation).
//
// Layout: records are tile-blocked SoA (cd_record.cuh), so a column tile is one contiguous 8 KB block that the TMA
// engine copies into shared memory (cp.async.bulk + mbarrier complete_tx, two stages; SASS UBLKCP) and a broadcast
// LDS.128 yields two ready-made packed operands (j..j+1, j+2..j+3) of one field.
// Decomposition: work item = (256 own rows) x (8 column tiles); a persistent grid of (SMs x resident
// CTAs) strides over the items, so the tail is < 1 item.  The hot loop only decides "conflict candidate";
// candidates (conflicts, LoS pairs, the diagonal, co-moving pairs: ~1e-5 of all pairs) are re-evaluated
// exactly by the scalar reference routine cd_pair_eval() out of line, which also feeds the per-row
// counters, tcpamax and the pair list.
#include <cuda_runtime.h>
#include <stdint.h>

#include "bsg_internal.h"
#include "bsg_math.cuh"
#include "cd_pair.cuh"
#include "cd_record.cuh"

namespace bsg {

constexpr int kNT = 128;                 // threads per CTA
constexpr int kR = 2;                    // rows per thread
constexpr int kRowsPerCta = kNT * kR;    // 256 = one tile of rows
constexpr int kTilesPerItem = 8;          // upper bound; the launch picks fewer when there are few items per CTA (tiles_per_item)
// culled form: work item = one row block x up to kTilesPerChunk listed column tiles.  Measured at N = 100k (2.8 % of
// the tile pairs kept): 1 -> 0.506 ms, 2 -> 0.539, 4 -> 0.574, 8 -> 0.626: balance beats the per-item set-up cost.
constexpr int kTilesPerChunk = 1;
constexpr uint32_t kTileBytes = kTileFloats * 4;

typedef unsigned long long u64;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

struct CdArgs {
    const float* rec;      // [n_tiles][8][256]
    int n_all, row0, n_rows;
    float R2, hpz, dtlook;
    uint32_t* nconf_row;
    uint32_t* nlos_row;
    float* tcpamax;
    int32_t* pairs;        // conflict pairs [cap][2], attributes [cap][BSG_CD_ATTR_COUNT], LoS pairs [los_cap][2]
    float* attr;
    long long cap;
    int32_t* lospairs;
    long long los_cap;
    unsigned long long* npairs;
    int n_rowblocks, n_colgroups, n_tiles, tiles_per_item;
    // culled form (bsg_cd_detect_culled): per row block the column tiles that can hold a conflict partner
    const int32_t* tile_list;     // [n_rowblocks][list_stride]
    const int32_t* list_cnt;      // [n_rowblocks]
    const int32_t* chunk_off;     // [n_rowblocks + 1] exclusive scan of ceil(list_cnt / kTilesPerChunk)
    int list_stride;
    unsigned int* work_counter;   // dynamic item fetch (items differ in size: a static stride leaves a long tail)
    // peer form (bsg_cd_detect_peers): the records stay where each GPU packed them; column tile t is read from
    // peer_rec[t / tiles_per_peer] over NVLink by the same TMA bulk copies (n_peers == 0: one local buffer, rec)
    const float* peer_rec[8];
    int n_peers, tiles_per_peer;
    const float* rec_rows;        // the buffer holding this call's own rows; its first record has global index rows_base
    int rows_base;
    int deal_n, deal_k;           // BSG_CD_DEAL: only the row blocks with (row tile % deal_n) == deal_k (0, 0: all)
};

// record idx as cd_pair.cuh's two halves A = (x, y, ch, sh), B = (u, v, alt, vs)
__device__ __forceinline__ void load_record(const float* __restrict__ rec, int idx, float4& A, float4& B) {
    const float* t = cd_rec(rec, idx);
    A = make_float4(t[FX * kTJ], t[FY * kTJ], t[FCH * kTJ], t[FSH * kTJ]);
    B = make_float4(t[FU * kTJ], t[FV * kTJ], t[FALT * kTJ], t[FVS * kTJ]);
}

__device__ __forceinline__ const float* tile_base(const CdArgs& a, int t) {
    if (a.n_peers == 0) return a.rec + (size_t)t * kTileFloats;
    const int p = t / a.tiles_per_peer;
    return a.peer_rec[p] + (size_t)(t - p * a.tiles_per_peer) * kTileFloats;
}

// Exact (reference-order) evaluation of one candidate pair, out of line, on records already at hand (own row from its
// packed registers, column from the shared-memory tile: no global loads on the rare path, which matters once culling
// has concentrated the candidates).  bit0 = conflict, bit1 = LoS.
template <bool WRAP>
__device__ __noinline__ uint32_t cd_candidate_rec(const float4 Ai, const float4 Bi, const float4 Aj, const float4 Bj,
                                                  float R2, float hpz, float dtlook, bool same, float& tcpa) {
    CdPair p = cd_pair_eval<WRAP>(Ai, Bi, Aj, Bj, R2, hpz, dtlook, same);
    tcpa = p.tcpa;
    return (p.conf ? 1u : 0u) | (p.los ? 2u : 0u);
}
// qdr, dist, dcpa, tcpa, tinconf of one conflict (what upstream's detect() returns per conflict besides the pair), written
// to row q of the attribute list.  Re-evaluates the pair: this runs once per conflict that made it into the list.
template <bool WRAP>
__device__ __noinline__ void cd_write_attr(float* q, const float4 Ai, const float4 Bi, const float4 Aj, const float4 Bj,
                                           float R2, float hpz, float dtlook) {
    const CdPair p = cd_pair_eval<WRAP>(Ai, Bi, Aj, Bj, R2, hpz, dtlook, false);
    q[BSG_CD_ATTR_QDR] = mod360(kRad2Deg * atan2f(p.dx, p.dy));
    q[BSG_CD_ATTR_DIST] = sqrtf(p.dist2);
    q[BSG_CD_ATTR_DCPA] = sqrtf(p.dcpa2);
    q[BSG_CD_ATTR_TCPA] = p.tcpa;
    q[BSG_CD_ATTR_TINCONF] = p.tinconf;
}

struct RowPack {            // loop-invariant operands of one own-row, duplicated into both f32x2 halves
    u64 nX, nY, CH, nSH, nU, nV, nALT, nVS;
};

// true when either column of the packed pair is a conflict candidate for this row.  SYM: ... or for the column as own
// aircraft against this row.  The two orders of a pair only differ through upstream's clamp of a near-zero relative
// vertical speed to +1e-6 in BOTH orders (the crossing time changes sign with the order): for clamped pairs the test
// is made with dalt := -|dalt|, which is the union of the two orders' windows.
template <bool WRAP, bool SYM>
__device__ __forceinline__ bool cd_hot2(const RowPack& r, u64 Xc, u64 Yc, u64 CHc, u64 SHc, u64 Uc, u64 Vc,
                                            u64 ALTc, u64 VSc, u64 R2P, u64 HPZP, u64 NEG1, float dtl) {
    u64 dy = add2(Yc, r.nY);
    u64 dxl = add2(Xc, r.nX);
    if (WRAP) {
        float a, b;
        up2(dxl, a, b);
        a -= kTwoPiRe * rintf(a * kInvTwoPiRe);
        b -= kTwoPiRe * rintf(b * kInvTwoPiRe);
        dxl = pk2(a, b);
    }
    u64 cav = fma2(SHc, r.nSH, mul2(CHc, r.CH));
    u64 dx = mul2(dxl, cav);
    u64 du = add2(Uc, r.nU), dv = add2(Vc, r.nV);
    u64 dv2 = fma2(du, du, mul2(dv, dv));
    u64 dot = fma2(du, dx, mul2(dv, dy));
    u64 crs = fma2(dy, du, mul2(mul2(dx, NEG1), dv));          // dy du - dx dv (only its square is used)
    float v0, v1;
    up2(dv2, v0, v1);
    v0 = fmaxf(v0, 1e-6f);
    v1 = fmaxf(v1, 1e-6f);
    u64 NINV = pk2(rcp_approx(-v0), rcp_approx(-v1));          // -1/|w|^2
    u64 tcpa = mul2(dot, NINV);                                // -dot/|w|^2
    u64 rem = fma2(mul2(crs, crs), NINV, R2P);                 // R^2 - dcpa^2
    u64 q = mul2(rem, NINV);                                   // -(R^2 - dcpa^2)/|w|^2
    float rem0, rem1, q0, q1;
    up2(rem, rem0, rem1);
    up2(q, q0, q1);
    u64 DTIN = pk2(sqrt_approx(-q0), sqrt_approx(-q1));        // NaN when dcpa >= R: max/min drop it, the
    u64 touthor = add2(tcpa, DTIN);                            // predicate below requires rem > 0 anyway
    u64 tinhor = fma2(DTIN, NEG1, tcpa);
    u64 dalt = add2(ALTc, r.nALT), dvs = add2(VSc, r.nVS);
    float s0, s1, a0, a1;
    up2(dvs, s0, s1);
    up2(dalt, a0, a1);
    const bool c0 = fabsf(s0) < 1e-6f, c1 = fabsf(s1) < 1e-6f;
    s0 = c0 ? 1e-6f : s0;
    s1 = c1 ? 1e-6f : s1;
    float r0 = rcp_approx(fabsf(s0)), r1 = rcp_approx(fabsf(s1));
    // t0 = dalt / -dvs = (-sign(dvs) dalt) / |dvs|
    a0 = __uint_as_float(__float_as_uint(a0) ^ (~__float_as_uint(s0) & 0x80000000u));
    a1 = __uint_as_float(__float_as_uint(a1) ^ (~__float_as_uint(s1) & 0x80000000u));
    if (SYM) { a0 = c0 ? fabsf(a0) : a0; a1 = c1 ? fabsf(a1) : a1; }
    u64 RV = pk2(r0, r1);
    u64 t0 = mul2(pk2(a0, a1), RV);
    u64 hw = mul2(HPZP, RV);
    u64 toutver = add2(t0, hw);
    u64 tinver = fma2(hw, NEG1, t0);
    float ih0, ih1, oh0, oh1, iv0, iv1, ov0, ov1;
    up2(tinhor, ih0, ih1);
    up2(touthor, oh0, oh1);
    up2(tinver, iv0, iv1);
    up2(toutver, ov0, ov1);
    float tin0 = fmaxf(iv0, ih0), tout0 = fminf(ov0, oh0);
    float tin1 = fmaxf(iv1, ih1), tout1 = fminf(ov1, oh1);
    bool h0 = (rem0 > 0.0f) && (tin0 <= tout0) && (tout0 > -0.01f) && (tin0 < dtl);
    bool h1 = (rem1 > 0.0f) && (tin1 <= tout1) && (tout1 > -0.01f) && (tin1 < dtl);
    return h0 || h1;
}

// One work item: 256 own rows (2 per thread, in packed registers) against n_t column tiles, which are either
// consecutive (t_begin ..) or taken from a list (culled form).  Column tiles arrive through the 2-stage TMA ring.
template <bool WRAP, bool LIST, bool SYM>
__device__ __forceinline__ void cd_process_item(const CdArgs& a, float (*s_tile)[kTileFloats], uint64_t* s_full, uint32_t* parity,
                                                const int rb, const int t_begin, const int n_t, const int32_t* __restrict__ list,
                                                const u64 R2P, const u64 HPZP, const u64 NEG1, const float dtlh, const int row_end) {
    const int tid = threadIdx.x;
    auto tile_of = [&](int tt) { return LIST ? (int)list[tt] : t_begin + tt; };
    const int own_tile = a.row0 / kRowsPerCta + rb;          // (SYM: rows are tile-aligned)
    // own rows -> packed registers.  Rows past the shard end are made inert (alt -kInertAlt: can never be a
    // candidate), so the hot loop needs no validity test.
    RowPack rp[kR];
    int ri[kR];
    uint32_t nconf[kR], nlos[kR];
    float tmax[kR];
    const int rbase = a.row0 + rb * kRowsPerCta;
#pragma unroll
    for (int k = 0; k < kR; ++k) {
        int r = rbase + tid + k * kNT;
        ri[k] = r;
        float4 A, B;
        load_record(a.rec_rows, (r < row_end ? r : row_end - 1) - a.rows_base, A, B);
        if (r >= row_end) B.z = -kInertAlt;             // inert row (padding columns sit at +kInertAlt)
        rp[k].nX = pk2(-A.x, -A.x); rp[k].nY = pk2(-A.y, -A.y);
        rp[k].CH = pk2(A.z, A.z);   rp[k].nSH = pk2(-A.w, -A.w);
        rp[k].nU = pk2(-B.x, -B.x); rp[k].nV = pk2(-B.y, -B.y);
        rp[k].nALT = pk2(-B.z, -B.z); rp[k].nVS = pk2(-B.w, -B.w);
        nconf[k] = 0; nlos[k] = 0; tmax[k] = 0.0f;
    }

    if (tid == 0) {        // prologue: first tile of the item
        mbar_expect_tx(&s_full[0], kTileBytes);
        tma_load_1d(&s_tile[0][0], tile_base(a, tile_of(0)), kTileBytes, &s_full[0]);
    }
#pragma unroll 1
    for (int tt = 0; tt < n_t; ++tt) {
        const int s = tt & 1;
        const int t = tile_of(tt);
        if (tid == 0 && tt + 1 < n_t) {     // prefetch the next tile into the other stage
            mbar_expect_tx(&s_full[s ^ 1], kTileBytes);
            tma_load_1d(&s_tile[s ^ 1][0], tile_base(a, tile_of(tt + 1)), kTileBytes, &s_full[s ^ 1]);
        }
        mbar_wait(&s_full[s], parity[s]);
        parity[s] ^= 1u;
        const float* tile = s_tile[s];
        const int c0 = t * kTJ;
#pragma unroll 1
        for (int j = 0; j < kTJ; j += 4) {
            // 8 broadcast LDS.128: four consecutive columns of each field = two packed operands
            const ulonglong2 X = *reinterpret_cast<const ulonglong2*>(tile + FX * kTJ + j);
            const ulonglong2 Y = *reinterpret_cast<const ulonglong2*>(tile + FY * kTJ + j);
            const ulonglong2 CH = *reinterpret_cast<const ulonglong2*>(tile + FCH * kTJ + j);
            const ulonglong2 SH = *reinterpret_cast<const ulonglong2*>(tile + FSH * kTJ + j);
            const ulonglong2 U = *reinterpret_cast<const ulonglong2*>(tile + FU * kTJ + j);
            const ulonglong2 V = *reinterpret_cast<const ulonglong2*>(tile + FV * kTJ + j);
            const ulonglong2 AL = *reinterpret_cast<const ulonglong2*>(tile + FALT * kTJ + j);
            const ulonglong2 VS = *reinterpret_cast<const ulonglong2*>(tile + FVS * kTJ + j);
            bool hit[kR];               // per own row: any of the four columns j .. j+3 flagged
#pragma unroll
            for (int k = 0; k < kR; ++k) {
                hit[k] = cd_hot2<WRAP, SYM>(rp[k], X.x, Y.x, CH.x, SH.x, U.x, V.x, AL.x, VS.x, R2P, HPZP, NEG1, dtlh);
                hit[k] |= cd_hot2<WRAP, SYM>(rp[k], X.y, Y.y, CH.y, SH.y, U.y, V.y, AL.y, VS.y, R2P, HPZP, NEG1, dtlh);
            }
            bool any = false;
#pragma unroll
            for (int k = 0; k < kR; ++k) any |= hit[k];
            if (any) {                   // rare: exact re-evaluation of the flagged rows' four pairs
#pragma unroll
                for (int k = 0; k < kR; ++k) {       // (static k: a runtime row index would push the row registers to local memory)
                    if (!hit[k] || ri[k] >= row_end) continue;
                    float nx, ny, chh, nsh, nu, nv, nal, nvs, dummy;
                    up2(rp[k].nX, nx, dummy); up2(rp[k].nY, ny, dummy); up2(rp[k].CH, chh, dummy); up2(rp[k].nSH, nsh, dummy);
                    up2(rp[k].nU, nu, dummy); up2(rp[k].nV, nv, dummy); up2(rp[k].nALT, nal, dummy); up2(rp[k].nVS, nvs, dummy);
                    const float4 Ai = make_float4(-nx, -ny, chh, -nsh), Bi = make_float4(-nu, -nv, -nal, -nvs);
                    const int rk = ri[k];
                    uint32_t nc = 0, nl = 0;
                    float tm = 0.0f;
#pragma unroll 1
                    for (int q = 0; q < 4; ++q) {
                        const int jc = j + q, cj = c0 + jc;
                        if (cj >= a.n_all) continue;
                        float tc;
                        const float4 Aj = make_float4(tile[FX * kTJ + jc], tile[FY * kTJ + jc], tile[FCH * kTJ + jc], tile[FSH * kTJ + jc]);
                        const float4 Bj = make_float4(tile[FU * kTJ + jc], tile[FV * kTJ + jc], tile[FALT * kTJ + jc], tile[FVS * kTJ + jc]);
                        const uint32_t f = cd_candidate_rec<WRAP>(Ai, Bi, Aj, Bj, a.R2, a.hpz, a.dtlook, rk == cj, tc);
                        if (SYM && t > own_tile) {       // the mirrored ordered pair (cj, ri): its row lives in another tile
                            float tcr;
                            const uint32_t fr = cd_candidate_rec<WRAP>(Aj, Bj, Ai, Bi, a.R2, a.hpz, a.dtlook, false, tcr);
                            const int o = cj - a.row0;
                            if ((fr & 2u) && a.nlos_row) atomicAdd(&a.nlos_row[o], 1u);
                            if ((fr & 2u) && a.npairs) {
                                const unsigned long long slot = atomicAdd(a.npairs + 1, 1ULL);
                                if (a.lospairs && (long long)slot < a.los_cap) { a.lospairs[2 * slot] = cj; a.lospairs[2 * slot + 1] = rk; }
                            }
                            if (fr & 1u) {
                                atomicAdd(&a.nconf_row[o], 1u);
                                if (a.tcpamax && tcr > 0.0f) atomicMax((int*)&a.tcpamax[o], __float_as_int(tcr));
                                if (a.npairs) {
                                    const unsigned long long slot = atomicAdd(a.npairs, 1ULL);
                                    if ((long long)slot < a.cap) {
                                        if (a.pairs) { a.pairs[2 * slot] = cj; a.pairs[2 * slot + 1] = rk; }
                                        if (a.attr) cd_write_attr<WRAP>(a.attr + BSG_CD_ATTR_COUNT * slot, Aj, Bj, Ai, Bi, a.R2, a.hpz, a.dtlook);
                                    }
                                }
                            }
                        }
                        if (f & 2u) {
                            nl++;
                            if (a.npairs) {
                                const unsigned long long slot = atomicAdd(a.npairs + 1, 1ULL);
                                if (a.lospairs && (long long)slot < a.los_cap) { a.lospairs[2 * slot] = rk; a.lospairs[2 * slot + 1] = cj; }
                            }
                        }
                        if (f & 1u) {
                            nc++;
                            tm = fmaxf(tm, tc);
                            if (a.npairs) {
                                const unsigned long long slot = atomicAdd(a.npairs, 1ULL);
                                if ((long long)slot < a.cap) {
                                    if (a.pairs) { a.pairs[2 * slot] = rk; a.pairs[2 * slot + 1] = cj; }
                                    if (a.attr) cd_write_attr<WRAP>(a.attr + BSG_CD_ATTR_COUNT * slot, Ai, Bi, Aj, Bj, a.R2, a.hpz, a.dtlook);
                                }
                            }
                        }
                    }
                    nconf[k] += nc; nlos[k] += nl; tmax[k] = fmaxf(tmax[k], tm);
                }
            }
            // The lanes that went through the rare path must rejoin the others HERE.  Left to the compiler, some shapes of
            // the rare path (an out-of-line call with side effects inside it) end in a barrier that is not marked
            // reconvergent, the warp then runs the rest of the tile's hot loop in two halves, and the whole detection takes
            // 27 % longer (15.4 vs 12.2 ms at N = 100k) for a path that 1e-5 of the pairs take.
            __syncwarp();
        }
        __syncthreads();     // stage s may be overwritten by the prefetch of iteration t+1
    }
#pragma unroll
    for (int k = 0; k < kR; ++k) {
        if (ri[k] < row_end) {
            const int o = ri[k] - a.row0;
            if (nconf[k]) {
                atomicAdd(&a.nconf_row[o], nconf[k]);
                if (a.tcpamax) atomicMax((int*)&a.tcpamax[o], __float_as_int(tmax[k]));
            }
            if (nlos[k] && a.nlos_row) atomicAdd(&a.nlos_row[o], nlos[k]);
        }
    }
}

// 4 CTAs per SM (124 registers); 5 (96 registers, no spills) measured slower (DESIGN §4)
template <bool WRAP, bool LIST, bool SYM>
__global__ void __launch_bounds__(kNT, 4) cd_tiled_kernel(const CdArgs a) {
    __shared__ __align__(128) float s_tile[2][kTileFloats];
    __shared__ __align__(8) uint64_t s_full[2];
    __shared__ int s_item[3];

    const int tid = threadIdx.x;
    if (tid == 0) {
        mbar_init(&s_full[0], 1);
        mbar_init(&s_full[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    uint32_t parity[2] = {0u, 0u};
    // The hot loop must flag a SUPERSET of what the exact routine accepts (it differs from it only by
    // float rounding), so its zone and look-ahead are inflated slightly; the exact routine decides.
    const float R2h = a.R2 * 1.0002f, hpzh = a.hpz * 1.0001f + 0.01f, dtlh = a.dtlook + 0.01f;
    const u64 R2P = pk2(R2h, R2h), HPZP = pk2(hpzh, hpzh), NEG1 = pk2(-1.0f, -1.0f);
    const int row_end = a.row0 + a.n_rows;

    if (!LIST) {
        // all column tiles, 8 per item; a persistent grid strides over the items
        const long long n_items = (long long)a.n_rowblocks * a.n_colgroups;
        for (long long item = blockIdx.x; item < n_items; item += gridDim.x) {
            const int rb = (int)(item / a.n_colgroups);
            const int t_begin = (int)(item % a.n_colgroups) * a.tiles_per_item;
            const int n_t = min(a.tiles_per_item, a.n_tiles - t_begin);
            cd_process_item<WRAP, false, false>(a, s_tile, s_full, parity, rb, t_begin, n_t, nullptr, R2P, HPZP, NEG1, dtlh, row_end);
        }
    } else {
        // culled form: items (row block, chunk of its tile list) differ in size and are handed out through a global
        // counter, so no CTA is left with a long tail
        const int n_items = a.chunk_off[a.n_rowblocks];
        for (;;) {
            if (tid == 0) {
                const int item = (int)atomicAdd(a.work_counter, 1u);
                int lo = 0, hi = a.n_rowblocks;
                if (item < n_items) {              // item -> row block: binary search in the scan of chunk counts
                    while (hi - lo > 1) {
                        int mid = (lo + hi) >> 1;
                        if (a.chunk_off[mid] <= item) lo = mid; else hi = mid;
                    }
                }
                s_item[0] = lo;
                s_item[1] = item < n_items ? item - a.chunk_off[lo] : 0;
                s_item[2] = item;
            }
            __syncthreads();
            const int rb = s_item[0], k0 = s_item[1] * kTilesPerChunk, item = s_item[2];
            __syncthreads();                       // s_item is rewritten for the next item
            if (item >= n_items) break;
            cd_process_item<WRAP, true, SYM>(a, s_tile, s_full, parity, rb, 0, min(kTilesPerChunk, a.list_cnt[rb] - k0),
                                        a.tile_list + (size_t)rb * a.list_stride + k0, R2P, HPZP, NEG1, dtlh, row_end);
        }
    }
}

// ---- culled form: which column tiles can hold a conflict / LoS partner of a row block -----------------
// Per tile of 256 records: bounding box in the kernel's own metric (x, y metres of arc), the smallest cos(lat)
// (dx = x-difference * cos(mean lat) >= x-difference * min cos), the largest ground speed, the altitude band
// and the largest |vs|.  Padding records (index >= n_all) are ignored.
enum { TB_XMIN = 0, TB_XMAX, TB_YMIN, TB_YMAX, TB_COSMIN, TB_VMAX, TB_AMIN, TB_AMAX, TB_VSMAX, TB_COUNT = 12 };

__global__ void __launch_bounds__(kTJ) cd_tile_bounds_kernel(const CdArgs a, int n_all, float* __restrict__ bounds) {
    __shared__ float s_red[9][kTJ / 32];
    const int tile = blockIdx.x, j = threadIdx.x, idx = tile * kTJ + j;
    const float* t = tile_base(a, tile) + j;
    const bool live = idx < n_all;
    const float x = t[FX * kTJ], y = t[FY * kTJ], ch = t[FCH * kTJ], sh = t[FSH * kTJ];
    const float u = t[FU * kTJ], v = t[FV * kTJ], alt = t[FALT * kTJ], vs = t[FVS * kTJ];
    float m[9];
    m[TB_XMIN] = live ? x : 3.0e38f;  m[TB_XMAX] = live ? x : -3.0e38f;
    m[TB_YMIN] = live ? y : 3.0e38f;  m[TB_YMAX] = live ? y : -3.0e38f;
    m[TB_COSMIN] = live ? fmaf(ch, ch, -sh * sh) : 1.0f;                 // cos(lat) from the half-angle pair
    m[TB_VMAX] = live ? sqrtf(fmaf(u, u, v * v)) : 0.0f;
    m[TB_AMIN] = live ? alt : 3.0e38f; m[TB_AMAX] = live ? alt : -3.0e38f;
    m[TB_VSMAX] = live ? fabsf(vs) : 0.0f;
    const bool is_min[9] = {true, false, true, false, true, false, true, false, false};
#pragma unroll
    for (int q = 0; q < 9; ++q) {
        float r = m[q];
        for (int o = 16; o > 0; o >>= 1) {
            float w = __shfl_xor_sync(0xffffffffu, r, o);
            r = is_min[q] ? fminf(r, w) : fmaxf(r, w);
        }
        if ((j & 31) == 0) s_red[q][j >> 5] = r;
    }
    __syncthreads();
    if (j < 9) {
        float r = s_red[j][0];
        for (int w = 1; w < kTJ / 32; ++w) r = is_min[j] ? fminf(r, s_red[j][w]) : fmaxf(r, s_red[j][w]);
        bounds[tile * TB_COUNT + j] = r;
    }
}

// One thread per (row block, column tile): keep the column tile unless NO aircraft pair of the two tiles can be
// in conflict or LoS -- horizontally closer than R + (v_a + v_b) T at time 0 is necessary for the protected zones
// to touch within the look-ahead T, and so is a vertical gap below hpz + (|vs_a| + |vs_b|) T.  Margins cover
// float rounding.  Kept tiles are appended to the row block's list in arbitrary order.
__global__ void cd_cull_kernel(const float* __restrict__ bounds, int n_tiles, int row_tile0, int n_rowblocks, float R,
                               float hpz, float T, int32_t* __restrict__ list, int32_t* __restrict__ cnt, int stride,
                               int sym, int alltiles, int deal_n, int deal_k) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= (long long)n_rowblocks * n_tiles) return;
    const int rb = (int)(p / n_tiles), ct = (int)(p % n_tiles);
    if (deal_n > 1 && (row_tile0 + rb) % deal_n != deal_k) return;   // BSG_CD_DEAL: another GPU's row block (its list stays empty)
    if (sym && ct < row_tile0 + rb) return;                     // symmetric form: the mirror tile pair covers it
    if (alltiles) { list[(size_t)rb * stride + atomicAdd(&cnt[rb], 1)] = ct; return; }
    const float* A = bounds + (size_t)(row_tile0 + rb) * TB_COUNT;
    const float* B = bounds + (size_t)ct * TB_COUNT;
    if (A[TB_XMIN] > A[TB_XMAX] || B[TB_XMIN] > B[TB_XMAX]) return;         // a tile of padding only
    const float gx = fmaxf(0.0f, fmaxf(B[TB_XMIN] - A[TB_XMAX], A[TB_XMIN] - B[TB_XMAX]));
    const float gy = fmaxf(0.0f, fmaxf(B[TB_YMIN] - A[TB_YMAX], A[TB_YMIN] - B[TB_YMAX]));
    const float cmin = fmaxf(0.0f, fminf(A[TB_COSMIN], B[TB_COSMIN]) - 1e-6f);
    const float dmin = sqrtf(fmaf(gx * cmin, gx * cmin, gy * gy));
    const float reach = (R * 1.001f + 1.0f) + (A[TB_VMAX] + B[TB_VMAX]) * (T + 0.05f) * 1.0001f;
    const float ga = fmaxf(0.0f, fmaxf(B[TB_AMIN] - A[TB_AMAX], A[TB_AMIN] - B[TB_AMAX]));
    const float vreach = (hpz * 1.001f + 0.1f) + (A[TB_VSMAX] + B[TB_VSMAX]) * (T + 0.05f) * 1.0001f;
    if (dmin <= reach && ga <= vreach) list[(size_t)rb * stride + atomicAdd(&cnt[rb], 1)] = ct;
}

// chunk_off = exclusive scan of ceil(cnt / kTilesPerChunk) over the row blocks (one block, any n)
__global__ void __launch_bounds__(1024) cd_chunk_scan_kernel(const int32_t* __restrict__ cnt, int n, int32_t* __restrict__ chunk_off) {
    __shared__ int s_part[1024];
    const int tid = threadIdx.x, per = (n + 1023) / 1024;
    const int lo = min(tid * per, n), hi = min(lo + per, n);
    int sum = 0;
    for (int i = lo; i < hi; ++i) sum += (cnt[i] + kTilesPerChunk - 1) / kTilesPerChunk;
    s_part[tid] = sum;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {                 // inclusive Hillis-Steele scan of the per-thread sums
        int v = tid >= o ? s_part[tid - o] : 0;
        __syncthreads();
        s_part[tid] += v;
        __syncthreads();
    }
    int run = s_part[tid] - sum;
    for (int i = lo; i < hi; ++i) { chunk_off[i] = run; run += (cnt[i] + kTilesPerChunk - 1) / kTilesPerChunk; }
    if (tid == 1023) chunk_off[n] = s_part[1023];
}

__global__ void cd_finalize_kernel(const uint32_t* __restrict__ nconf_row, uint8_t* __restrict__ inconf, long long n) {
    long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) inconf[i] = nconf_row[i] > 0;
}

// float64 SoA -> CD records (cd_record.cuh); padding entries are inert aircraft.
__global__ void cd_pack_kernel(const double* __restrict__ lat, const double* __restrict__ lon,
                               const double* __restrict__ trk, const double* __restrict__ gs,
                               const double* __restrict__ alt, const double* __restrict__ vs,
                               const int32_t* __restrict__ perm, long long n,
                               long long n_pad, double lat0, double lon0, float* __restrict__ rec) {
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // record index
    if (k >= n_pad) return;
    float f[BSG_CD_REC_FIELDS];
    if (k < n) {
        const long long i = perm ? (long long)perm[k] : k;                     // the aircraft it holds (bsg_cd_pack_ordered)
        cd_rec_position(f, lat[i], lon[i], lat0, lon0);
        double st, ct;
        sincos(trk[i] * kDeg2RadD, &st, &ct);
        f[FU] = (float)(gs[i] * st); f[FV] = (float)(gs[i] * ct); f[FALT] = (float)alt[i]; f[FVS] = (float)vs[i];
    } else {
        cd_rec_inert(f);
    }
    cd_rec_store(rec, k, f);
}

}  // namespace bsg

using namespace bsg;

extern "C" int64_t bsg_cd_padded(int64_t n) { return ((n + kTJ - 1) / kTJ) * kTJ; }

// (also the last stage of bsg_cd_pack_ordered, cd_order.cu: d_perm[k] = the aircraft record k holds)
int bsg_cd_pack_launch(const double* d_lat, const double* d_lon, const double* d_trk, const double* d_gs, const double* d_alt,
                       const double* d_vs, const int32_t* d_perm, int64_t n, double lat0, double lon0, float* d_rec, cudaStream_t st) {
    int64_t n_pad = bsg_cd_padded(n);
    if (n_pad == 0) return BSG_OK;
    int blocks = (int)((n_pad + 255) / 256);
    cd_pack_kernel<<<blocks, 256, 0, st>>>(d_lat, d_lon, d_trk, d_gs, d_alt, d_vs, d_perm, n, n_pad, lat0, lon0, d_rec);
    return bsg_cuda_check(cudaGetLastError(), "bsg_cd_pack launch");
}

extern "C" int bsg_cd_pack(const double* d_lat, const double* d_lon, const double* d_trk, const double* d_gs,
                           const double* d_alt, const double* d_vs, int64_t n, double lat0, double lon0,
                           float* d_rec, void* stream) {
    if (n < 0 || (n > 0 && (!d_lat || !d_lon || !d_trk || !d_gs || !d_alt || !d_vs)) || !d_rec)
        return bsg_fail(BSG_EINVAL, "bsg_cd_pack: null pointer or negative n");
    return bsg_cd_pack_launch(d_lat, d_lon, d_trk, d_gs, d_alt, d_vs, nullptr, n, lat0, lon0, d_rec, (cudaStream_t)stream);
}

// ---- launch plumbing shared by the three entry points ------------------------------------------------
static int cd_fill_args(CdArgs& a, int64_t n_all, int64_t row0, int64_t n_rows, float rpz, float hpz, float dtlookahead,
                        uint32_t* d_nconf_row, uint32_t* d_nlos_row, float* d_tcpamax, const bsg_cd_lists* lists) {
    static const bsg_cd_lists none = {nullptr, nullptr, 0, nullptr, 0, nullptr};
    const bsg_cd_lists& L = lists ? *lists : none;
    if (n_all < 0 || row0 < 0 || n_rows < 0 || row0 + n_rows > n_all) return bsg_fail(BSG_EINVAL, "CD: row range outside [0, n_all)");
    if (n_all > 0x7fffff00LL) return bsg_fail(BSG_EINVAL, "CD: n_all exceeds int32 pair indices");
    if (n_rows > 0 && !d_nconf_row) return bsg_fail(BSG_EINVAL, "CD: null d_nconf_row");
    if ((L.d_conf_pairs || L.d_conf_attr || L.d_los_pairs) && !L.d_npairs) return bsg_fail(BSG_EINVAL, "CD: pair lists need d_npairs");
    if (L.conf_cap < 0 || L.los_cap < 0) return bsg_fail(BSG_EINVAL, "CD: negative list capacity");
    memset(&a, 0, sizeof(a));
    a.n_all = (int)n_all; a.row0 = (int)row0; a.n_rows = (int)n_rows;
    if (rpz <= 0.0f) rpz = 5.0f * 1852.0f;
    if (hpz <= 0.0f) hpz = 1000.0f * 0.3048f;
    if (dtlookahead <= 0.0f) dtlookahead = 300.0f;
    a.R2 = rpz * rpz; a.hpz = hpz; a.dtlook = dtlookahead;
    a.nconf_row = d_nconf_row; a.nlos_row = d_nlos_row; a.tcpamax = d_tcpamax;
    a.pairs = L.d_conf_pairs; a.attr = L.d_conf_attr; a.cap = L.conf_cap;
    a.lospairs = L.d_los_pairs; a.los_cap = L.los_cap; a.npairs = L.d_npairs;
    a.n_tiles = (int)(bsg_cd_padded(n_all) / kTJ);
    a.n_rowblocks = (int)((n_rows + kRowsPerCta - 1) / kRowsPerCta);
    a.tiles_per_item = kTilesPerItem;
    a.n_colgroups = (a.n_tiles + kTilesPerItem - 1) / kTilesPerItem;
    return BSG_OK;
}

static int cd_launch(CdArgs& a, bool wrap, bool cull, bool sym, bool alltiles, void* d_work, int64_t work_bytes, uint8_t* d_inconf,
                     cudaStream_t st) {
    if (a.npairs) BSG_CUDA(cudaMemsetAsync(a.npairs, 0, 2 * sizeof(unsigned long long), st));
    if (a.n_rows == 0) return BSG_OK;
    BSG_CUDA(cudaMemsetAsync(a.nconf_row, 0, sizeof(uint32_t) * a.n_rows, st));
    if (a.nlos_row) BSG_CUDA(cudaMemsetAsync(a.nlos_row, 0, sizeof(uint32_t) * a.n_rows, st));
    if (a.tcpamax) BSG_CUDA(cudaMemsetAsync(a.tcpamax, 0, sizeof(float) * a.n_rows, st));
    int dev = 0, sms = 0, occ = 0;
    BSG_CUDA(cudaGetDevice(&dev));
    BSG_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    if (cull) {
        if (a.row0 % kRowsPerCta) return bsg_fail(BSG_EINVAL, "culled CD: row0 must be a multiple of 256");
        if (sym && (a.row0 != 0 || a.n_rows != a.n_all)) return bsg_fail(BSG_EINVAL, "BSG_CD_SYMMETRIC needs n_rows == n_all (one GPU holds every row)");
        if (wrap) return bsg_fail(BSG_EINVAL, "culled CD: airspaces across the antimeridian use the plain form");
        if (!d_work || work_bytes < bsg_cd_cull_workspace(a.n_all, a.n_rows))
            return bsg_fail(BSG_EINVAL, "culled CD: workspace missing or too small (bsg_cd_cull_workspace)");
        char* w = (char*)d_work;
        float* bounds = (float*)w;                       w += 16 * (((size_t)a.n_tiles * TB_COUNT * 4 + 15) / 16);
        int32_t* cnt = (int32_t*)w;                      w += 16 * (((size_t)a.n_rowblocks * 4 + 15) / 16);
        int32_t* chunk_off = (int32_t*)w;                w += 16 * (((size_t)(a.n_rowblocks + 1) * 4 + 15) / 16);
        a.work_counter = (unsigned int*)w;               w += 16;
        int32_t* list = (int32_t*)w;
        a.tile_list = list; a.list_cnt = cnt; a.chunk_off = chunk_off; a.list_stride = a.n_tiles;
        BSG_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int32_t) * a.n_rowblocks, st));
        BSG_CUDA(cudaMemsetAsync(a.work_counter, 0, sizeof(unsigned int), st));
        cd_tile_bounds_kernel<<<a.n_tiles, kTJ, 0, st>>>(a, a.n_all, bounds);
        const long long n_pairs = (long long)a.n_rowblocks * a.n_tiles;
        cd_cull_kernel<<<(int)((n_pairs + 255) / 256), 256, 0, st>>>(bounds, a.n_tiles, a.row0 / kRowsPerCta, a.n_rowblocks,
                                                                     sqrtf(a.R2), a.hpz, a.dtlook, list, cnt, a.list_stride,
                                                                     sym ? 1 : 0, alltiles ? 1 : 0, a.deal_n, a.deal_k);
        cd_chunk_scan_kernel<<<1, 1024, 0, st>>>(cnt, a.n_rowblocks, chunk_off);
        BSG_CUDA(cudaGetLastError());
        if (sym) BSG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, cd_tiled_kernel<false, true, true>, kNT, 0));
        else BSG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, cd_tiled_kernel<false, true, false>, kNT, 0));
        if (occ < 1) occ = 1;
        if (sym) cd_tiled_kernel<false, true, true><<<sms * occ, kNT, 0, st>>>(a);
        else cd_tiled_kernel<false, true, false><<<sms * occ, kNT, 0, st>>>(a);
    } else {
        if (wrap) BSG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, cd_tiled_kernel<true, false, false>, kNT, 0));
        else BSG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, cd_tiled_kernel<false, false, false>, kNT, 0));
        if (occ < 1) occ = 1;
        // Items are dealt to the persistent CTAs by a static stride, so the launch ends with a partial round: a row shard of
        // 1/8 of 100k aircraft is 2401 eight-tile items on 592 CTAs = 4.06 rounds, i.e. a fifth round that is 6 % full
        // (0.687 of the FP32 peak per GPU against 0.758 on one GPU).  The tiles per item are therefore chosen per launch:
        // the count (1..8) that minimises rounds x (tiles + the pipeline bubble at the start of an item, ~6 % of a tile).
        {
            const long long slots = (long long)sms * occ;
            double best = 1e30;
            int best_t = kTilesPerItem;
            for (int t = kTilesPerItem; t >= 1; --t) {
                const long long items = (long long)a.n_rowblocks * ((a.n_tiles + t - 1) / t);
                const double cost = (double)((items + slots - 1) / slots) * ((double)t + 0.06);
                if (cost < best * 0.999) { best = cost; best_t = t; }
            }
            a.tiles_per_item = best_t;
            a.n_colgroups = (a.n_tiles + best_t - 1) / best_t;
        }
        const long long n_items = (long long)a.n_rowblocks * a.n_colgroups;
        const int grid = (int)((n_items < (long long)sms * occ) ? n_items : (long long)sms * occ);
        if (wrap) cd_tiled_kernel<true, false, false><<<grid, kNT, 0, st>>>(a);
        else cd_tiled_kernel<false, false, false><<<grid, kNT, 0, st>>>(a);
    }
    BSG_CUDA(cudaGetLastError());
    if (d_inconf) {
        cd_finalize_kernel<<<(int)((a.n_rows + 255) / 256), 256, 0, st>>>(a.nconf_row, d_inconf, a.n_rows);
        BSG_CUDA(cudaGetLastError());
    }
    return BSG_OK;
}

extern "C" int bsg_cd_detect(const float* d_rec, int64_t n_all, int64_t row0, int64_t n_rows, float rpz, float hpz,
                             float dtlookahead, uint32_t flags, uint32_t* d_nconf_row, uint32_t* d_nlos_row,
                             float* d_tcpamax, uint8_t* d_inconf, const bsg_cd_lists* lists, void* stream) {
    if (flags & BSG_CD_SYMMETRIC) return bsg_fail(BSG_EINVAL, "bsg_cd_detect: BSG_CD_SYMMETRIC is served by bsg_cd_detect_culled (it needs the work-list scratch)");
    CdArgs a;
    int rc = cd_fill_args(a, n_all, row0, n_rows, rpz, hpz, dtlookahead, d_nconf_row, d_nlos_row, d_tcpamax, lists);
    if (rc != BSG_OK) return rc;
    if (n_rows > 0 && !d_rec) return bsg_fail(BSG_EINVAL, "bsg_cd_detect: null d_rec");
    a.rec = d_rec; a.rec_rows = d_rec; a.rows_base = 0;
    return cd_launch(a, (flags & BSG_CD_LON_WRAP) != 0, false, false, false, nullptr, 0, d_inconf, (cudaStream_t)stream);
}

extern "C" int64_t bsg_cd_cull_workspace(int64_t n_all, int64_t n_rows) {
    const int64_t n_tiles = bsg_cd_padded(n_all) / kTJ, n_rb = (n_rows + kRowsPerCta - 1) / kRowsPerCta;
    // bounds | list_cnt | chunk_off | work counter | tile_list
    return 16 * ((n_tiles * TB_COUNT * 4 + 15) / 16) + 16 * ((n_rb * 4 + 15) / 16) + 16 * (((n_rb + 1) * 4 + 15) / 16) + 16 +
           n_rb * n_tiles * 4 + 64;
}

extern "C" int bsg_cd_detect_culled(const float* d_rec, int64_t n_all, int64_t row0, int64_t n_rows, float rpz, float hpz,
                                    float dtlookahead, uint32_t flags, uint32_t* d_nconf_row, uint32_t* d_nlos_row,
                                    float* d_tcpamax, uint8_t* d_inconf, const bsg_cd_lists* lists,
                                    void* d_work, int64_t work_bytes, void* stream) {
    CdArgs a;
    int rc = cd_fill_args(a, n_all, row0, n_rows, rpz, hpz, dtlookahead, d_nconf_row, d_nlos_row, d_tcpamax, lists);
    if (rc != BSG_OK) return rc;
    if (n_rows > 0 && !d_rec) return bsg_fail(BSG_EINVAL, "bsg_cd_detect_culled: null d_rec");
    a.rec = d_rec; a.rec_rows = d_rec; a.rows_base = 0;
    a.deal_n = (int)((flags >> 8) & 0xffu); a.deal_k = (int)((flags >> 16) & 0xffu);
    if (a.deal_n > 1 && a.deal_k >= a.deal_n) return bsg_fail(BSG_EINVAL, "bsg_cd_detect_culled: BSG_CD_DEAL(n, k) needs k < n");
    return cd_launch(a, (flags & BSG_CD_LON_WRAP) != 0, true, (flags & BSG_CD_SYMMETRIC) != 0, (flags & BSG_CD_ALLTILES) != 0, d_work, work_bytes,
                     d_inconf, (cudaStream_t)stream);
}

extern "C" int bsg_cd_detect_peers(const float* const* h_peer_rec, int32_t n_peers, int32_t my_rank, int64_t n_per_peer,
                                   float rpz, float hpz, float dtlookahead, uint32_t flags, uint32_t* d_nconf_row,
                                   uint32_t* d_nlos_row, float* d_tcpamax, uint8_t* d_inconf, const bsg_cd_lists* lists,
                                   void* d_work, int64_t work_bytes, void* stream) {
    if (!h_peer_rec || n_peers < 1 || n_peers > 8 || my_rank < 0 || my_rank >= n_peers)
        return bsg_fail(BSG_EINVAL, "bsg_cd_detect_peers: need 1..8 peer buffers and a rank among them");
    if (n_per_peer <= 0 || n_per_peer % kTJ) return bsg_fail(BSG_EINVAL, "bsg_cd_detect_peers: n_per_peer must be a positive multiple of 256");
    for (int p = 0; p < n_peers; ++p)
        if (!h_peer_rec[p]) return bsg_fail(BSG_EINVAL, "bsg_cd_detect_peers: null peer buffer");
    CdArgs a;
    int rc = cd_fill_args(a, n_per_peer * n_peers, n_per_peer * my_rank, n_per_peer, rpz, hpz, dtlookahead, d_nconf_row, d_nlos_row,
                          d_tcpamax, lists);
    if (rc != BSG_OK) return rc;
    a.rec = nullptr;
    for (int p = 0; p < n_peers; ++p) a.peer_rec[p] = h_peer_rec[p];
    a.n_peers = n_peers; a.tiles_per_peer = (int)(n_per_peer / kTJ);
    a.rec_rows = h_peer_rec[my_rank]; a.rows_base = (int)(n_per_peer * my_rank);
    return cd_launch(a, (flags & BSG_CD_LON_WRAP) != 0, (flags & BSG_CD_CULL) != 0, false, false, d_work, work_bytes, d_inconf,
                     (cudaStream_t)stream);
}
