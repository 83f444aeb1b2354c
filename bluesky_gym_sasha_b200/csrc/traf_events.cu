// traf_events.cu -- conflict and loss-of-separation events of an airspace, tracked on the device (bsg_traf_events_update).
//
// Upstream's ConflictDetection.update keeps confpairs_all / lospairs_all: every unordered pair that enters the conflict
// (LoS) set of a detection after being out of it is one more event.  Per detection, two kernels:
//   traf_ev_insert_kernel -- every row of the detection's conflict and LoS lists (bsg_cd_lists, any order, length
//                            min(npairs, cap) read on the device) inserts its normalised key (kind bit | a < b) into the
//                            CURRENT open-addressing set with atomicCAS, which merges the two orientations of a pair.  The
//                            thread that claims the slot looks the key up in the PREVIOUS set: found, the event goes on (its
//                            log row is carried over); not found, a new event starts (totals, log row claimed by atomicAdd).
//                            LoS keys fold this detection's horizontal distance and |dalt| into the event's minima.
//   traf_ev_retire_kernel -- walks the previous set's dense slot list (not its table): a key that is absent from the current
//                            set ends its event (log end = nstep); every visited slot is cleared, so the previous set is
//                            empty again and serves as the current set of the next detection (the caller swaps them).
// Work per detection is proportional to the pairs of this detection and of the previous one, not to the table size.
//
// Bound: latency of random 16-byte slot accesses in L2 / HBM, not bandwidth.  Algorithmic bytes per listed pair: the 8-byte
// list row, one 16-byte CAS into the current table and one 16-byte probe of the previous one, 4 bytes of dense list; per
// event of the previous detection one more probe, a 16-byte read and a 16-byte clear; per new event a 16-byte log row
// (+ 8 bytes of LoS minima; every LoS row also reads 2 x 5 floats of CD records).
#include <cuda_runtime.h>
#include <stdint.h>

#include "bsg_internal.h"

namespace bsg {

constexpr int kEvTile = 256;                    // aircraft per CD record tile (cd_tiled.cu: kTJ)
constexpr int kEvThreads = 256;
constexpr int64_t kEvMaxPairs = 1LL << 28;      // conf_cap + los_cap: slot indices of the tables stay below 2^30
constexpr int64_t kEvHeader = 16;               // set header: uint32 number of occupied slots, padded to 16 bytes

// one slot of a set: key 0 = empty (a < b, so no pair has key 0); log = row of the event in its log, -1 = not logged
struct __align__(16) EvSlot {
    unsigned long long key;
    int log, pad;
};

struct EvParams {
    EvSlot *cur, *prev;
    unsigned *cur_count;
    const unsigned* prev_count;
    int *cur_slots;
    const int* prev_slots;
    unsigned long long mask;                    // table capacity - 1
    int4* log[2];                               // [kind]: a, b, start, end
    float2* sev;                                // LoS log: dmin, dalt_min
    long long log_cap[2];
    unsigned long long* ctr;
    const float* rec;
    const int2* pairs[2];                       // [kind] = conflict list, LoS list
    long long cap[2];
    const unsigned long long* npairs;
    int nstep;
};

__host__ __device__ __forceinline__ int64_t ev_table_cap(int64_t pairs) {
    int64_t t = 64;
    while (t < 2 * pairs) t <<= 1;
    return t;
}

__device__ __forceinline__ unsigned long long ev_hash(unsigned long long k) {      // splitmix64 finaliser
    k ^= k >> 30; k *= 0xbf58476d1ce4e5b9ULL;
    k ^= k >> 27; k *= 0x94d049bb133111ebULL;
    return k ^ (k >> 31);
}

// linear probing; the tables are at most half full, so an empty slot ends every search
__device__ __forceinline__ bool ev_find(const EvSlot* tab, const unsigned long long mask, const unsigned long long key, int& log) {
    for (unsigned long long s = ev_hash(key) & mask;; s = (s + 1) & mask) {
        const EvSlot e = tab[s];
        if (e.key == key) { log = e.log; return true; }
        if (e.key == 0ull) return false;
    }
}

__device__ __forceinline__ float ev_rec(const float* rec, const int j, const int field) {
    return rec[(size_t)(j / kEvTile) * (8 * kEvTile) + field * kEvTile + (j % kEvTile)];
}

// Horizontal distance and |dalt| of the pair (a, b) in this detection's CD records, cd_pair.cuh's algebra
// (dx = dlon-difference * (ch_a ch_b - sh_a sh_b), dy = lat-difference).  Every step is an explicitly rounded IEEE
// operation -- no contraction into FMAs -- so the value is exactly symmetric in a and b and a float32 restatement on the
// host reproduces it bit for bit.
__device__ __forceinline__ void ev_los_severity(const float* rec, const int a, const int b, float& d, float& dalt) {
    const float cav = __fsub_rn(__fmul_rn(ev_rec(rec, a, 2), ev_rec(rec, b, 2)), __fmul_rn(ev_rec(rec, a, 3), ev_rec(rec, b, 3)));
    const float dx = __fmul_rn(__fsub_rn(ev_rec(rec, b, 0), ev_rec(rec, a, 0)), cav);
    const float dy = __fsub_rn(ev_rec(rec, b, 1), ev_rec(rec, a, 1));
    d = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
    dalt = fabsf(__fsub_rn(ev_rec(rec, b, 6), ev_rec(rec, a, 6)));
}

__global__ void __launch_bounds__(kEvThreads) traf_ev_insert_kernel(const EvParams P) {
    const unsigned long long n0 = P.npairs[0], n1 = P.npairs[1];
    const long long m0 = n0 < (unsigned long long)P.cap[0] ? (long long)n0 : P.cap[0];
    const long long m1 = n1 < (unsigned long long)P.cap[1] ? (long long)n1 : P.cap[1];
    if (blockIdx.x == 0 && threadIdx.x == 0 && (m0 < (long long)n0 || m1 < (long long)n1))
        atomicAdd(&P.ctr[BSG_EV_CTR_TRUNCATED], 1ull);
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < m0 + m1; r += (long long)gridDim.x * blockDim.x) {
        const int kind = r >= m0;
        const int2 p = P.pairs[kind][kind ? r - m0 : r];
        const int a = min(p.x, p.y), b = max(p.x, p.y);
        if (a < 0 || a == b) continue;          // not a pair: a detection never lists one, a hand-made list might
        const unsigned long long key = (unsigned long long)kind << 62 | (unsigned long long)a << 31 | (unsigned long long)b;
        unsigned long long s = ev_hash(key) & P.mask;
        bool won = false;
        for (;; s = (s + 1) & P.mask) {
            const unsigned long long old = atomicCAS(&P.cur[s].key, 0ull, key);
            if (old == 0ull) { won = true; break; }
            if (old == key) break;
        }
        if (!won) continue;                     // the other orientation (or a duplicate row) speaks for the pair
        P.cur_slots[atomicAdd(P.cur_count, 1u)] = (int)s;
        float d = 0.0f, dalt = 0.0f;
        if (kind) ev_los_severity(P.rec, a, b, d, dalt);
        int log;
        if (ev_find(P.prev, P.mask, key, log)) {
            // the event goes on.  This thread is the only one that touches the event's row in this detection, and
            // detections are ordered on the stream, so the minima need no atomics.
            if (kind && log >= 0) {
                const float2 v = P.sev[log];
                P.sev[log] = make_float2(fminf(v.x, d), fminf(v.y, dalt));
            }
        } else {                                // a new event: its number is also its log row
            const unsigned long long idx = atomicAdd(&P.ctr[BSG_EV_CTR_NCONF_TOTAL + kind], 1ull);
            atomicAdd(&P.ctr[BSG_EV_CTR_NCONF_ACTIVE + kind], 1ull);
            log = idx < (unsigned long long)P.log_cap[kind] ? (int)idx : -1;
            if (log < 0) {
                atomicAdd(&P.ctr[BSG_EV_CTR_LOG_OVERFLOW], 1ull);
            } else {
                P.log[kind][log] = make_int4(a, b, P.nstep, -1);
                if (kind) P.sev[log] = make_float2(d, dalt);
            }
        }
        P.cur[s].log = log;
    }
}

__global__ void __launch_bounds__(kEvThreads) traf_ev_retire_kernel(const EvParams P) {
    const long long m = *P.prev_count;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < m; r += (long long)gridDim.x * blockDim.x) {
        const int s = P.prev_slots[r];
        const EvSlot e = P.prev[s];
        int log;
        if (!ev_find(P.cur, P.mask, e.key, log)) {
            const int kind = (int)(e.key >> 62);
            atomicAdd(&P.ctr[BSG_EV_CTR_NCONF_ACTIVE + kind], ~0ull);        // - 1
            if (e.log >= 0) P.log[kind][e.log].w = P.nstep;
        }
        P.prev[s] = EvSlot{0ull, 0, 0};
    }
}

}  // namespace bsg

using namespace bsg;

extern "C" int64_t bsg_traf_events_workspace(int64_t conf_cap, int64_t los_cap) {
    if (conf_cap < 0 || los_cap < 0 || conf_cap + los_cap > kEvMaxPairs) return 0;
    const int64_t pairs = conf_cap + los_cap;
    return kEvHeader + (int64_t)sizeof(EvSlot) * ev_table_cap(pairs) + (int64_t)sizeof(int) * pairs;
}

extern "C" int bsg_traf_events_update(const bsg_traf_events* ev, const float* d_rec, const bsg_cd_lists* lists, int64_t nstep,
                                      void* stream) {
    if (!ev || !lists) return bsg_fail(BSG_EINVAL, "bsg_traf_events_update: null argument");
    if (!lists->d_npairs) return bsg_fail(BSG_EINVAL, "bsg_traf_events_update: lists->d_npairs is null");
    if (lists->conf_cap < 0 || lists->los_cap < 0 || lists->conf_cap + lists->los_cap > kEvMaxPairs)
        return bsg_fail(BSG_EINVAL, "bsg_traf_events_update: list capacities must be >= 0 and add up to at most 2^28");
    if ((lists->conf_cap > 0 && !lists->d_conf_pairs) || (lists->los_cap > 0 && !lists->d_los_pairs))
        return bsg_fail(BSG_EINVAL, "bsg_traf_events_update: a pair list with a capacity is null");
    if (lists->los_cap > 0 && !d_rec) return bsg_fail(BSG_EINVAL, "bsg_traf_events_update: LoS severity needs the CD records d_rec");
    if (!ev->d_cur || !ev->d_prev || ev->d_cur == ev->d_prev)
        return bsg_fail(BSG_EINVAL, "bsg_traf_events_update: d_cur and d_prev must be two distinct sets");
    if (((uintptr_t)ev->d_cur | (uintptr_t)ev->d_prev) % 16) return bsg_fail(BSG_EINVAL, "bsg_traf_events_update: sets must be 16-byte aligned");
    if (ev->set_bytes < bsg_traf_events_workspace(lists->conf_cap, lists->los_cap))
        return bsg_fail(BSG_EINVAL, "bsg_traf_events_update: set_bytes is smaller than bsg_traf_events_workspace(conf_cap, los_cap)");
    if (ev->conf_log_cap < 0 || ev->los_log_cap < 0 || ev->conf_log_cap > 0x7fffffffLL || ev->los_log_cap > 0x7fffffffLL)
        return bsg_fail(BSG_EINVAL, "bsg_traf_events_update: log capacities must be in [0, 2^31)");
    if ((ev->conf_log_cap > 0 && !ev->d_conf_log) || (ev->los_log_cap > 0 && (!ev->d_los_log || !ev->d_los_sev)))
        return bsg_fail(BSG_EINVAL, "bsg_traf_events_update: a log with a capacity is null");
    if (!ev->d_counters) return bsg_fail(BSG_EINVAL, "bsg_traf_events_update: d_counters is null");
    if (nstep < 0 || nstep > 0x7fffffffLL) return bsg_fail(BSG_EINVAL, "bsg_traf_events_update: nstep must be in [0, 2^31)");

    const int64_t pairs = lists->conf_cap + lists->los_cap;
    const int64_t tcap = ev_table_cap(pairs);
    EvParams P;
    P.cur = (EvSlot*)((char*)ev->d_cur + kEvHeader);
    P.prev = (EvSlot*)((char*)ev->d_prev + kEvHeader);
    P.cur_count = (unsigned*)ev->d_cur;
    P.prev_count = (const unsigned*)ev->d_prev;
    P.cur_slots = (int*)(P.cur + tcap);
    P.prev_slots = (const int*)(P.prev + tcap);
    P.mask = (unsigned long long)(tcap - 1);
    P.log[0] = (int4*)ev->d_conf_log; P.log[1] = (int4*)ev->d_los_log; P.sev = (float2*)ev->d_los_sev;
    P.log_cap[0] = ev->conf_log_cap; P.log_cap[1] = ev->los_log_cap;
    P.ctr = ev->d_counters;
    P.rec = d_rec;
    P.pairs[0] = (const int2*)lists->d_conf_pairs; P.pairs[1] = (const int2*)lists->d_los_pairs;
    P.cap[0] = lists->conf_cap; P.cap[1] = lists->los_cap;
    P.npairs = lists->d_npairs;
    P.nstep = (int)nstep;
    if (pairs == 0) return BSG_OK;

    cudaStream_t st = (cudaStream_t)stream;
    int dev = 0, sms = 0;
    BSG_CUDA(cudaGetDevice(&dev));
    BSG_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    // grid sized on the capacity (the counts live on the device), capped at one full wave: threads stride over the rows
    const int64_t want = (pairs + kEvThreads - 1) / kEvThreads, wave = (int64_t)sms * (2048 / kEvThreads);
    const unsigned blocks = (unsigned)(want < wave ? want : wave);
    BSG_CUDA(cudaMemsetAsync(P.cur_count, 0, sizeof(unsigned), st));     // the current set's table is empty already
    traf_ev_insert_kernel<<<blocks, kEvThreads, 0, st>>>(P);
    traf_ev_retire_kernel<<<blocks, kEvThreads, 0, st>>>(P);
    return bsg_cuda_check(cudaGetLastError(), "bsg_traf_events_update launch");
}
