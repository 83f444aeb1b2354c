// cd_record.cuh -- storage of the 32-byte CD record (include/bsg.h: BSG_CD_TILE, BSG_CD_REC_*), shared by the detection
// (cd_tiled.cu), the airspace substep (traf_airspace.cu) and the event tracker (traf_events.cu).  Records are tile-blocked
// SoA, rec[tile][field][BSG_CD_TILE] floats, so one tile is a contiguous 8 KB block.  What the fields mean and the
// algebra on them: cd_pair.cuh.
#pragma once
#include "bsg_internal.h"
#include "bsg_math.cuh"

namespace bsg {

constexpr int kTJ = BSG_CD_TILE;                          // records per tile
constexpr int kTileFloats = BSG_CD_REC_FIELDS * kTJ;
enum { FX = BSG_CD_REC_X, FY = BSG_CD_REC_Y, FCH = BSG_CD_REC_CH, FSH = BSG_CD_REC_SH,
       FU = BSG_CD_REC_U, FV = BSG_CD_REC_V, FALT = BSG_CD_REC_ALT, FVS = BSG_CD_REC_VS };
// |dalt| ~ 3e9 to any aircraft: never a conflict or LoS candidate.  Padding records sit at +kInertAlt; the detection
// makes its own rows past the shard end inert at -kInertAlt.
constexpr float kInertAlt = 3.0e9f;

// record j; its field f is at [f * kTJ].  For kernels that read or write a whole record.
template <typename T, typename I>
__device__ __forceinline__ T* cd_rec(T* rec, const I j) {
    return rec + (size_t)(j / kTJ) * kTileFloats + (j % kTJ);
}
// field `field` of record j: cd_rec(rec, j)[field * kTJ], formed as one index.  For kernels that read single fields.
__device__ __forceinline__ float cd_rec_at(const float* rec, const long long j, const int field) {
    return rec[(j / kTJ) * kTileFloats + field * kTJ + j % kTJ];
}

// x, y [m of arc from (lat0, lon0)] and the cos, sin of half the latitude of an aircraft at (lat, lon) [deg]
__device__ __forceinline__ void cd_rec_position(float (&f)[BSG_CD_REC_FIELDS], const double lat, const double lon,
                                                const double lat0, const double lon0) {
    double dl = fmod((lon - lon0) + 180.0, 360.0);
    if (dl < 0.0) dl += 360.0;
    dl -= 180.0;
    double s, c;
    sincos(lat * (0.5 * kDeg2RadD), &s, &c);
    f[FX] = (float)(kRearthD * kDeg2RadD * dl); f[FY] = (float)(kRearthD * kDeg2RadD * (lat - lat0));
    f[FCH] = (float)c; f[FSH] = (float)s;
}

// the record of padding and of dead aircraft slots
__device__ __forceinline__ void cd_rec_inert(float (&f)[BSG_CD_REC_FIELDS]) {
    f[FX] = 0.0f; f[FY] = 0.0f; f[FCH] = 1.0f; f[FSH] = 0.0f;
    f[FU] = 0.0f; f[FV] = 0.0f; f[FALT] = kInertAlt; f[FVS] = 0.0f;
}

template <typename I>
__device__ __forceinline__ void cd_rec_store(float* __restrict__ rec, const I j, const float (&f)[BSG_CD_REC_FIELDS]) {
    float* t = cd_rec(rec, j);
#pragma unroll
    for (int q = 0; q < BSG_CD_REC_FIELDS; ++q) t[q * kTJ] = f[q];
}

}  // namespace bsg
