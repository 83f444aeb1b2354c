// cd_order.cu -- spatial order for the culled conflict detection, on the device (no library sort).
//
// bsg_cd_detect_culled skips (row block, column tile) pairs whose bounding boxes are out of each other's reach, which
// only pays off when consecutive records -- the kernel's 256-record tiles -- are spatially compact.  Exact sorting is not
// needed for that, only coherence: the aircraft are binned into a uniform grid over their bounding box (latitude strips x
// fine longitude bins, about 16 bins per tile so a tile's footprint is roughly square) and laid out strip by strip,
// alternate strips running east and west (a tile that straddles two strips then still covers one compact corner instead of
// both ends of the airspace).  A counting sort: bounding box (atomic min / max), cell histogram, one-block scan, scatter,
// then the pack kernel gathers through the permutation.  Five small launches, O(N), ~20 us at N = 100k against 0.66 ms
// for two library radix sorts and six gathers.  The order inside a cell is whatever the atomics give: every output of
// the detection is a set, a count or a maximum, so results do not depend on it.
#include <cuda_runtime.h>
#include <stdint.h>

#include "bsg_internal.h"

namespace bsg {

constexpr int kOrderMaxCells = 16384;
constexpr int kBinsPerTile = 16;

struct OrderWork {              // layout of the workspace
    long long box[4];           // lat min, lat max, dlon min, dlon max as order-preserving integers
    int grid[4];                // ny, nx, cells, pad (written by the cell kernel's first thread)
    int hist[kOrderMaxCells];
    int offs[kOrderMaxCells + 1];
    // int cell[n] follows
};

__device__ __forceinline__ long long dkey(double v) {       // order-preserving map double -> signed 64-bit integer
    long long b = __double_as_longlong(v);
    return b >= 0 ? b : (b ^ 0x7fffffffffffffffLL);
}
__device__ __forceinline__ double dunkey(long long k) { return __longlong_as_double(k >= 0 ? k : (k ^ 0x7fffffffffffffffLL)); }
__device__ __forceinline__ double dlon_of(double lon, double lon0) {
    double dl = fmod((lon - lon0) + 180.0, 360.0);
    if (dl < 0.0) dl += 360.0;
    return dl - 180.0;
}

__global__ void order_init_kernel(OrderWork* w) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < kOrderMaxCells) w->hist[i] = 0;
    if (i == 0) { w->box[0] = w->box[2] = 0x7fffffffffffffffLL; w->box[1] = w->box[3] = -0x7fffffffffffffffLL - 1; }
}

// where the order kernels read an aircraft's position: the float64 SoA arrays of bsg_cd_pack_ordered, or the traffic
// state of bsg_traf_pack_ordered, whose dead slots (inert records) stay out of the bounding box
struct SoaPos {
    const double *lat, *lon;
    __device__ __forceinline__ bool in_box(long long) const { return true; }
    __device__ __forceinline__ double2 operator()(long long i) const { return make_double2(lat[i], lon[i]); }
};
struct TrafPos {
    const double2* pos;
    const uint32_t* flags;
    __device__ __forceinline__ bool in_box(long long i) const { return (flags[i] & BSG_TF_ALIVE) != 0; }
    __device__ __forceinline__ double2 operator()(long long i) const { return pos[i]; }
};

template <typename Pos>
__global__ void __launch_bounds__(256) order_bbox_kernel(const Pos pos, long long n, double lon0, OrderWork* w) {
    double a0 = 1e300, a1 = -1e300, o0 = 1e300, o1 = -1e300;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        if (!pos.in_box(i)) continue;
        const double2 p = pos(i);
        const double la = p.x, dl = dlon_of(p.y, lon0);
        a0 = fmin(a0, la); a1 = fmax(a1, la); o0 = fmin(o0, dl); o1 = fmax(o1, dl);
    }
    for (int o = 16; o > 0; o >>= 1) {
        a0 = fmin(a0, __shfl_xor_sync(0xffffffffu, a0, o)); a1 = fmax(a1, __shfl_xor_sync(0xffffffffu, a1, o));
        o0 = fmin(o0, __shfl_xor_sync(0xffffffffu, o0, o)); o1 = fmax(o1, __shfl_xor_sync(0xffffffffu, o1, o));
    }
    if ((threadIdx.x & 31) == 0 && a0 <= a1) {
        atomicMin(&w->box[0], dkey(a0)); atomicMax(&w->box[1], dkey(a1));
        atomicMin(&w->box[2], dkey(o0)); atomicMax(&w->box[3], dkey(o1));
    }
}

// grid shape from the bounding box: strips as tall as a tile is wide, kBinsPerTile longitude bins per tile
__device__ __forceinline__ void order_grid(const OrderWork* w, long long n, double& la0, double& o0, double& sy, double& sx, int& ny, int& nx) {
    la0 = dunkey(w->box[0]); o0 = dunkey(w->box[2]);
    const double la1 = dunkey(w->box[1]), o1 = dunkey(w->box[3]);
    const double h = fmax(la1 - la0, 1e-9);
    const double wd = fmax((o1 - o0) * cos(0.5 * (la0 + la1) * 0.017453292519943295), 1e-9);
    const double tiles = fmax(1.0, ceil((double)n / (double)BSG_CD_TILE));
    double strips = fmax(1.0, rint(sqrt(tiles * h / wd)));
    strips = fmin(strips, 512.0);
    double bins = fmax(1.0, ceil(tiles / strips * (double)kBinsPerTile));
    bins = fmin(bins, floor((double)kOrderMaxCells / strips));
    ny = (int)strips; nx = (int)fmax(bins, 1.0);
    sy = (double)ny / h * (1.0 - 1e-12); sx = (double)nx / fmax(o1 - o0, 1e-9) * (1.0 - 1e-12);
}

template <typename Pos>
__global__ void __launch_bounds__(256) order_cell_kernel(const Pos pos, long long n, double lon0, OrderWork* w, int* __restrict__ cell) {
    double la0, o0, sy, sx;
    int ny, nx;
    order_grid(w, n, la0, o0, sy, sx, ny, nx);
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i == 0) { w->grid[0] = ny; w->grid[1] = nx; w->grid[2] = ny * nx; }
    if (i >= n) return;
    const double2 p = pos(i);
    int iy = (int)((p.x - la0) * sy), ix = (int)((dlon_of(p.y, lon0) - o0) * sx);
    iy = min(max(iy, 0), ny - 1); ix = min(max(ix, 0), nx - 1);
    if (iy & 1) ix = nx - 1 - ix;                      // alternate strips run the other way
    const int c = iy * nx + ix;
    cell[i] = c;
    atomicAdd(&w->hist[c], 1);
}

// exclusive scan of the cell histogram (one block); the histogram becomes the scatter cursors (zeroed)
__global__ void __launch_bounds__(1024) order_scan_kernel(OrderWork* w) {
    __shared__ int s_part[1024];
    const int tid = threadIdx.x, per = kOrderMaxCells / 1024;
    int sum = 0;
    for (int k = 0; k < per; ++k) sum += w->hist[tid * per + k];
    s_part[tid] = sum;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        const int v = tid >= o ? s_part[tid - o] : 0;
        __syncthreads();
        s_part[tid] += v;
        __syncthreads();
    }
    int run = s_part[tid] - sum;
    for (int k = 0; k < per; ++k) {
        const int h = w->hist[tid * per + k];
        w->offs[tid * per + k] = run;
        w->hist[tid * per + k] = 0;
        run += h;
    }
    if (tid == 1023) w->offs[kOrderMaxCells] = run;
}

__global__ void __launch_bounds__(256) order_scatter_kernel(long long n, OrderWork* w, const int* __restrict__ cell, int32_t* __restrict__ perm) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int c = cell[i];
    perm[w->offs[c] + atomicAdd(&w->hist[c], 1)] = (int32_t)i;
}

// a detection on ordered records -> aircraft order: pair list rows (the first min(npairs, cap), count read here) are
// rewritten in place through perm, per-row outputs scattered, out[perm[k]] = in[k].  One grid-stride range over the conflict
// rows, then the LoS rows, then the aircraft, so that each thread has one short chain of dependent loads: O(pairs + n).
struct UnpermArgs {
    const int32_t* perm;
    long long n;
    int2 *conf, *los;
    long long conf_cap, los_cap;
    const unsigned long long* npairs;
    const uint32_t *nconf_in, *nlos_in;
    const float* tcpamax_in;
    const uint8_t* inconf_in;
    uint32_t *nconf_out, *nlos_out;
    float* tcpamax_out;
    uint8_t* inconf_out;
};

__global__ void __launch_bounds__(256) cd_unpermute_kernel(const UnpermArgs a) {
    const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
    const int32_t* __restrict__ perm = a.perm;
    const long long mc = a.conf ? (long long)min(a.npairs[0], (unsigned long long)a.conf_cap) : 0;
    const long long ml = a.los ? (long long)min(a.npairs[1], (unsigned long long)a.los_cap) : 0;
    for (long long t = t0; t < mc + ml + a.n; t += stride) {
        if (t < mc + ml) {
            int2* __restrict__ row = t < mc ? a.conf + t : a.los + (t - mc);
            const int2 p = *row;
            *row = make_int2(perm[p.x], perm[p.y]);
        } else {
            const long long k = t - mc - ml;
            const int32_t j = perm[k];
            if (a.nconf_out) a.nconf_out[j] = a.nconf_in[k];
            if (a.nlos_out) a.nlos_out[j] = a.nlos_in[k];
            if (a.tcpamax_out) a.tcpamax_out[j] = a.tcpamax_in[k];
            if (a.inconf_out) a.inconf_out[j] = a.inconf_in[k];
        }
    }
}

// the order of n aircraft into perm: bounding box, cells, scan, scatter (five launches)
template <typename Pos>
static int order_launch(const Pos pos, long long n, double lon0, int32_t* perm, void* d_work, cudaStream_t st) {
    OrderWork* w = (OrderWork*)d_work;
    int* cell = (int*)((char*)d_work + sizeof(OrderWork));
    const int blocks = (int)((n + 255) / 256);
    order_init_kernel<<<kOrderMaxCells / 256, 256, 0, st>>>(w);
    order_bbox_kernel<<<blocks < 592 ? blocks : 592, 256, 0, st>>>(pos, n, lon0, w);
    order_cell_kernel<<<blocks, 256, 0, st>>>(pos, n, lon0, w, cell);
    order_scan_kernel<<<1, 1024, 0, st>>>(w);
    order_scatter_kernel<<<blocks, 256, 0, st>>>(n, w, cell, perm);
    return bsg_cuda_check(cudaGetLastError(), "spatial order launch");
}

}  // namespace bsg

using namespace bsg;

// (cd_tiled.cu)
int bsg_cd_pack_launch(const double* d_lat, const double* d_lon, const double* d_trk, const double* d_gs, const double* d_alt,
                       const double* d_vs, const int32_t* d_perm, int64_t n, double lat0, double lon0, float* d_rec, cudaStream_t st);

extern "C" int64_t bsg_cd_order_workspace(int64_t n) { return (int64_t)sizeof(OrderWork) + 4 * (n > 0 ? n : 0) + 16; }

extern "C" int bsg_cd_pack_ordered(const double* d_lat, const double* d_lon, const double* d_trk, const double* d_gs,
                                   const double* d_alt, const double* d_vs, int64_t n, double lat0, double lon0,
                                   float* d_rec, int32_t* d_perm, void* d_work, int64_t work_bytes, void* stream) {
    if (n < 0 || (n > 0 && (!d_lat || !d_lon || !d_trk || !d_gs || !d_alt || !d_vs || !d_perm)) || !d_rec)
        return bsg_fail(BSG_EINVAL, "bsg_cd_pack_ordered: null pointer or negative n");
    if (n > 0x7fffff00LL) return bsg_fail(BSG_EINVAL, "bsg_cd_pack_ordered: n exceeds int32 indices");
    if (n == 0) return BSG_OK;
    if (!d_work || work_bytes < bsg_cd_order_workspace(n)) return bsg_fail(BSG_EINVAL, "bsg_cd_pack_ordered: workspace too small");
    if ((uintptr_t)d_work % 8) return bsg_fail(BSG_EINVAL, "bsg_cd_pack_ordered: workspace must be 8-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    int rc = order_launch(SoaPos{d_lat, d_lon}, n, lon0, d_perm, d_work, st);
    if (rc != BSG_OK) return rc;
    return bsg_cd_pack_launch(d_lat, d_lon, d_trk, d_gs, d_alt, d_vs, d_perm, n, lat0, lon0, d_rec, st);
}

// (traf_airspace.cu: bsg_traf_pack_ordered; the caller has validated the arguments and the workspace)
int bsg_traf_order_launch(const double2* pos, const uint32_t* flags, int64_t n, double lon0, int32_t* d_perm, void* d_work,
                          cudaStream_t st) {
    return order_launch(TrafPos{pos, flags}, n, lon0, d_perm, d_work, st);
}

extern "C" int bsg_cd_unpermute(const int32_t* d_perm, int64_t n, const bsg_cd_lists* lists, const uint32_t* d_nconf_in,
                                const uint32_t* d_nlos_in, const float* d_tcpamax_in, const uint8_t* d_inconf_in,
                                uint32_t* d_nconf_out, uint32_t* d_nlos_out, float* d_tcpamax_out, uint8_t* d_inconf_out,
                                void* stream) {
    if (n < 0 || n > 0x7fffff00LL) return bsg_fail(BSG_EINVAL, "bsg_cd_unpermute: n must be in [0, 2^31 - 256]");
    if (n > 0 && !d_perm) return bsg_fail(BSG_EINVAL, "bsg_cd_unpermute: null d_perm");
    if ((!d_nconf_in != !d_nconf_out) || (!d_nlos_in != !d_nlos_out) || (!d_tcpamax_in != !d_tcpamax_out) ||
        (!d_inconf_in != !d_inconf_out))
        return bsg_fail(BSG_EINVAL, "bsg_cd_unpermute: a per-row output needs both its input and its output pointer");
    if ((d_nconf_in && (const void*)d_nconf_in == (const void*)d_nconf_out) ||
        (d_nlos_in && (const void*)d_nlos_in == (const void*)d_nlos_out) ||
        (d_tcpamax_in && (const void*)d_tcpamax_in == (const void*)d_tcpamax_out) ||
        (d_inconf_in && (const void*)d_inconf_in == (const void*)d_inconf_out))
        return bsg_fail(BSG_EINVAL, "bsg_cd_unpermute: per-row input and output must be distinct (a scatter cannot run in place)");
    UnpermArgs a{};
    a.perm = d_perm; a.n = n;
    if (lists) {
        if (lists->conf_cap < 0 || lists->los_cap < 0) return bsg_fail(BSG_EINVAL, "bsg_cd_unpermute: negative list capacities");
        if ((lists->d_conf_pairs || lists->d_los_pairs) && !lists->d_npairs)
            return bsg_fail(BSG_EINVAL, "bsg_cd_unpermute: pair lists need d_npairs");
        a.conf = lists->conf_cap > 0 ? (int2*)lists->d_conf_pairs : nullptr;
        a.los = lists->los_cap > 0 ? (int2*)lists->d_los_pairs : nullptr;
        a.conf_cap = lists->conf_cap; a.los_cap = lists->los_cap; a.npairs = lists->d_npairs;
    }
    if (n == 0) a.conf = a.los = nullptr;               // no records, no pairs
    a.nconf_in = d_nconf_in; a.nlos_in = d_nlos_in; a.tcpamax_in = d_tcpamax_in; a.inconf_in = d_inconf_in;
    a.nconf_out = d_nconf_out; a.nlos_out = d_nlos_out; a.tcpamax_out = d_tcpamax_out; a.inconf_out = d_inconf_out;
    // threads: one per aircraft and list row (at most), up to 8 blocks per SM
    const long long work = n + (a.conf ? a.conf_cap : 0) + (a.los ? a.los_cap : 0);
    if (work == 0) return BSG_OK;
    const long long blocks = (work + 255) / 256;
    cd_unpermute_kernel<<<(unsigned)(blocks < 1184 ? blocks : 1184), 256, 0, (cudaStream_t)stream>>>(a);
    return bsg_cuda_check(cudaGetLastError(), "bsg_cd_unpermute launch");
}
