// cd_exhaustive.cu -- test harness, not part of libbsg_b200.so: state-based conflict detection of EVERY ordered pair
// (i in a row range, j over all records), with no hot filter and no tile culling.  It is the reference that the forms of
// cd_tiled.cu (plain, culled, symmetric, dealt, peers) are compared with, row for row and bit for bit.
//
// The decision and the attributes come from the same cd_pair_eval<WRAP> (cd_pair.cuh) that K2's exact routine runs, inside
// __noinline__ functions shaped like cd_candidate_rec / cd_write_attr, so both compile to the same arithmetic: a pair
// that the hot filter or the cull drops shows up here and nowhere else.  One thread per (row, block of 256 columns).
#include <cuda_runtime.h>
#include <stdint.h>

#include "cd_pair.cuh"
#include "cd_record.cuh"

namespace bsg {

constexpr int kExRows = 128;          // rows per CTA

// bit0 = conflict, bit1 = LoS (cd_tiled.cu: cd_candidate_rec)
template <bool WRAP>
__device__ __noinline__ uint32_t ex_pair_rec(const float4 Ai, const float4 Bi, const float4 Aj, const float4 Bj, float R2,
                                             float hpz, float dtlook, bool same, float& tcpa) {
    CdPair p = cd_pair_eval<WRAP>(Ai, Bi, Aj, Bj, R2, hpz, dtlook, same);
    tcpa = p.tcpa;
    return (p.conf ? 1u : 0u) | (p.los ? 2u : 0u);
}
// qdr, dist, dcpa, tcpa, tinconf of one conflict (cd_tiled.cu: cd_write_attr)
template <bool WRAP>
__device__ __noinline__ void ex_write_attr(float* q, const float4 Ai, const float4 Bi, const float4 Aj, const float4 Bj,
                                           float R2, float hpz, float dtlook) {
    const CdPair p = cd_pair_eval<WRAP>(Ai, Bi, Aj, Bj, R2, hpz, dtlook, false);
    q[BSG_CD_ATTR_QDR] = mod360(kRad2Deg * atan2f(p.dx, p.dy));
    q[BSG_CD_ATTR_DIST] = sqrtf(p.dist2);
    q[BSG_CD_ATTR_DCPA] = sqrtf(p.dcpa2);
    q[BSG_CD_ATTR_TCPA] = p.tcpa;
    q[BSG_CD_ATTR_TINCONF] = p.tinconf;
}

__device__ __forceinline__ void ex_load(const float* __restrict__ rec, long long idx, float4& A, float4& B) {
    const float* t = cd_rec(rec, idx);
    A = make_float4(t[FX * kTJ], t[FY * kTJ], t[FCH * kTJ], t[FSH * kTJ]);
    B = make_float4(t[FU * kTJ], t[FV * kTJ], t[FALT * kTJ], t[FVS * kTJ]);
}

struct ExArgs {
    const float* rec;
    long long n_all, row0, n_rows;
    float R2, hpz, dtlook;
    uint32_t *nconf_row, *nlos_row;
    float* tcpamax;
    int32_t* pairs;
    float* attr;
    long long cap;
    int32_t* lospairs;
    long long los_cap;
    unsigned long long* npairs;
};

template <bool WRAP>
__global__ void __launch_bounds__(kExRows) cd_exhaustive_kernel(const ExArgs a) {
    const long long r = (long long)blockIdx.x * kExRows + threadIdx.x;
    if (r >= a.n_rows) return;
    const long long i = a.row0 + r;
    const long long j0 = (long long)blockIdx.y * kTJ, j1 = min(j0 + kTJ, a.n_all);
    float4 Ai, Bi;
    ex_load(a.rec, i, Ai, Bi);
    uint32_t nc = 0, nl = 0;
    float tm = 0.0f;
    for (long long j = j0; j < j1; ++j) {
        float4 Aj, Bj;
        ex_load(a.rec, j, Aj, Bj);
        float tc;
        const uint32_t f = ex_pair_rec<WRAP>(Ai, Bi, Aj, Bj, a.R2, a.hpz, a.dtlook, i == j, tc);
        if (f & 2u) {
            nl++;
            const unsigned long long slot = atomicAdd(a.npairs + 1, 1ULL);
            if ((long long)slot < a.los_cap) { a.lospairs[2 * slot] = (int32_t)i; a.lospairs[2 * slot + 1] = (int32_t)j; }
        }
        if (f & 1u) {
            nc++;
            tm = fmaxf(tm, tc);
            const unsigned long long slot = atomicAdd(a.npairs, 1ULL);
            if ((long long)slot < a.cap) {
                a.pairs[2 * slot] = (int32_t)i; a.pairs[2 * slot + 1] = (int32_t)j;
                ex_write_attr<WRAP>(a.attr + BSG_CD_ATTR_COUNT * slot, Ai, Bi, Aj, Bj, a.R2, a.hpz, a.dtlook);
            }
        }
    }
    if (nc) {
        atomicAdd(&a.nconf_row[r], nc);
        atomicMax((int*)&a.tcpamax[r], __float_as_int(tm));      // tm >= +0: the int order is the float order
    }
    if (nl) atomicAdd(&a.nlos_row[r], nl);
}

}  // namespace bsg

using namespace bsg;

// Every ordered pair (i, j), i in [row0, row0 + n_rows), j in [0, n_all), of the CD records d_rec (bsg_cd_pack layout),
// with the zone (rpz, hpz, dtlook) used as given.  Per row: conflicts, LoS pairs, the largest positive tcpa of its
// conflicts (0 when none).  Lists: up to cap conflicts (pairs + qdr, dist, dcpa, tcpa, tinconf) and los_cap LoS pairs, in
// arbitrary order; d_npairs = (conflicts, LoS pairs) found.  Zeroes its outputs first.  Returns a cudaError_t.
extern "C" int cd_exhaustive(const float* d_rec, int64_t n_all, int64_t row0, int64_t n_rows, float rpz, float hpz,
                             float dtlook, int wrap, uint32_t* d_nconf_row, uint32_t* d_nlos_row, float* d_tcpamax,
                             int32_t* d_pairs, float* d_attr, int64_t cap, int32_t* d_lospairs, int64_t los_cap,
                             unsigned long long* d_npairs, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemsetAsync(d_npairs, 0, 2 * sizeof(unsigned long long), st);
    if (e != cudaSuccess || n_rows <= 0) return (int)e;
    if ((e = cudaMemsetAsync(d_nconf_row, 0, sizeof(uint32_t) * n_rows, st)) != cudaSuccess) return (int)e;
    if ((e = cudaMemsetAsync(d_nlos_row, 0, sizeof(uint32_t) * n_rows, st)) != cudaSuccess) return (int)e;
    if ((e = cudaMemsetAsync(d_tcpamax, 0, sizeof(float) * n_rows, st)) != cudaSuccess) return (int)e;
    ExArgs a;
    a.rec = d_rec; a.n_all = n_all; a.row0 = row0; a.n_rows = n_rows;
    a.R2 = rpz * rpz; a.hpz = hpz; a.dtlook = dtlook;          // (as cd_tiled.cu's cd_fill_args forms them)
    a.nconf_row = d_nconf_row; a.nlos_row = d_nlos_row; a.tcpamax = d_tcpamax;
    a.pairs = d_pairs; a.attr = d_attr; a.cap = cap; a.lospairs = d_lospairs; a.los_cap = los_cap; a.npairs = d_npairs;
    const dim3 grid((unsigned)((n_rows + kExRows - 1) / kExRows), (unsigned)((n_all + kTJ - 1) / kTJ));
    if (wrap) cd_exhaustive_kernel<true><<<grid, kExRows, 0, st>>>(a);
    else cd_exhaustive_kernel<false><<<grid, kExRows, 0, st>>>(a);
    return (int)cudaGetLastError();
}
