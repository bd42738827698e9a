// gcra_kernels.cuh -- the sm_100a kernels of the batched GCRA engine.
//
//   K1a ingest  : bulk-async (TMA, UBLKCP) staging of a request tile into shared memory, per-request
//                 validation + parameter derivation (rate_limiter.rs:111-122), key -> slot probe/claim
//   K1b order   : stable one-sweep LSD radix sort of (slot, index) so that requests on one key are adjacent and
//                 in index order -- the reference applies requests strictly one at a time
//                 (throttlecrab-server/src/actor.rs:217-236)
//   K1c decide  : warp-cooperative GCRA compare-and-update (rate_limiter.rs:150-248); duplicates of a
//                 key inside a batch are resolved exactly by speculate-and-commit over warp ballots
//   K2  sweep   : HashMap::retain(expiry > now) (adaptive_cleanup.rs:176-182) as a streaming scan
//   K3  route   : stable partition of a batch by owner shard for the multi-GPU all-to-all
#pragma once
#include <cooperative_groups.h>

#include "gcra_device.cuh"
#include "../../include/gcra_b200.h"

namespace gcra {

constexpr int TILE_THREADS = 256;

// ---------------------------------------------------------------------------------------------
// mbarrier + 1-D bulk async copy (TMA) helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ u32 smem_u32(const void *p) {
    return (u32)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(u64 *bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(u64 *bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, u32 bytes, u64 *bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ void mbar_wait(u64 *bar, u32 parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra.uni WAIT_DONE;\n"
        "bra.uni WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// ---------------------------------------------------------------------------------------------
// K1a: ingest
// ---------------------------------------------------------------------------------------------
struct PolicyDerived { i64 ei, dvt; int status; int pad; };

__device__ __forceinline__ void write_result(gcra_result *out, i64 remaining, i64 reset, i64 retry,
                                             int status, int allowed) {
    longlong2 a = make_longlong2(remaining, reset);
    longlong2 b;
    b.x = retry;
    b.y = (i64)(u32)status | ((i64)(allowed & 0xff) << 32);
    reinterpret_cast<longlong2 *>(out)[0] = a;
    reinterpret_cast<longlong2 *>(out)[1] = b;
}

// validation (rate_limiter.rs:111-117) + parameter derivation of ONE request record (shared or global memory):
// returns the status the reference would return before touching the store, fills the key hash and the
// derived request.
template <bool COMPACT>
__device__ __forceinline__ int parse_request(const unsigned char *rec, const PolicyDerived *__restrict__ pol, u32 npol,
                                             i64 now_batch, u64 &key_hash, Req &r) {
    int status = 0;
    if (COMPACT) {
        ulonglong2 w = *reinterpret_cast<const ulonglong2 *>(rec);
        key_hash = w.x;
        int qty = (int)(u32)(w.y & 0xffffffffULL);
        u32 p = (u32)(w.y >> 32);
        r.q = qty;
        r.now = now_batch;
        r.ei = 0;
        r.dvt = 0;
        if (qty < 0) status = GCRA_NEGATIVE_QUANTITY;          // rate_limiter.rs:111-113
        else if (p >= npol) status = GCRA_INTERNAL;
        else {
            PolicyDerived pd = pol[p];
            status = pd.status;
            r.ei = pd.ei;
            r.dvt = pd.dvt;
        }
    } else {
        const ulonglong2 *q = reinterpret_cast<const ulonglong2 *>(rec);
        ulonglong2 w0 = q[0], w1 = q[1], w2 = q[2];
        key_hash = w0.x;
        i64 max_burst = (i64)w0.y, count = (i64)w1.x, period = (i64)w1.y;
        r.q = (i64)w2.x;
        r.now = (i64)w2.y;
        r.ei = 0;
        r.dvt = 0;
        if (r.q < 0) status = GCRA_NEGATIVE_QUANTITY;          // :111-113
        else if (max_burst <= 0 || count <= 0 || period <= 0) status = GCRA_INVALID_RATE_LIMIT;  // :115-117
        else status = derive_params(max_burst, count, period, &r.ei, &r.dvt);
    }
    // a pre-epoch `now` makes the reference read the wall clock (:128-143): not reproducible
    if (status == 0 && r.now < 0) status = GCRA_INTERNAL;
    return status;
}

// validation, parameter derivation, key probe/claim for ONE request whose record sits at `rec` (shared or
// global memory).  Writes the derived request, the error result if any, and returns the sort key
// (slot << 32 | i).  Must be called by all 32 lanes of a warp (warp-aggregated counters).
template <bool COMPACT>
__device__ __forceinline__ u64 ingest_one(const Table &t, const unsigned char *rec, bool in_range,
                                          const PolicyDerived *__restrict__ pol, u32 npol, i64 now_batch, u32 i,
                                          Req *__restrict__ drec, gcra_result *__restrict__ out) {
    int status = 0;
    u64 key_hash = 0;
    Req r = {0, 0, 0, 0};
    if (in_range) status = parse_request<COMPACT>(rec, pol, npol, now_batch, key_hash, r);
    u32 slot = t.null_slot;
    bool fresh = false;
    if (in_range && status == 0) {
        slot = find_or_claim(t, stored_key(key_hash), fresh);
        if (slot == t.null_slot) status = GCRA_INTERNAL;   // table full
    }
    if (in_range) {
        reinterpret_cast<longlong2 *>(drec + i)[0] = make_longlong2(r.now, r.ei);
        reinterpret_cast<longlong2 *>(drec + i)[1] = make_longlong2(r.dvt, r.q);
        if (status != 0) write_result(out + i, 0, 0, 0, status, 0);
    }
    // warp-aggregated counters
    u32 mf = __ballot_sync(0xffffffffu, fresh);
    u32 me = __ballot_sync(0xffffffffu, in_range && status != 0);
    if ((threadIdx.x & 31) == 0) {
        if (mf) atomicAdd(&t.counters[C_OCCUPIED], (u64)__popc(mf));
        if (me) atomicAdd(&t.counters[C_ERRORS], (u64)__popc(me));
    }
    return ((u64)slot << 32) | i;
}

template <bool COMPACT>
__global__ void __launch_bounds__(TILE_THREADS)
ingest_kernel(Table t, const void *__restrict__ req_base, const PolicyDerived *__restrict__ pol,
              u32 npol, i64 now_batch, u32 n, Req *__restrict__ drec, u64 *__restrict__ sortkeys,
              gcra_result *__restrict__ out) {
    constexpr u32 RSZ = COMPACT ? sizeof(gcra_request16) : sizeof(gcra_request);
    __shared__ __align__(128) unsigned char stage[TILE_THREADS * RSZ];
    __shared__ __align__(8) u64 bar;

    const u32 base = blockIdx.x * TILE_THREADS;
    const u32 cnt = min((u32)TILE_THREADS, n - base);
    if (threadIdx.x == 0) {
        mbar_init(&bar, 1);
        fence_barrier_init();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(&bar, cnt * RSZ);
        bulk_g2s(stage, (const unsigned char *)req_base + (size_t)base * RSZ, cnt * RSZ, &bar);
    }
    mbar_wait(&bar, 0);

    const u32 i = base + threadIdx.x;
    const bool in_range = threadIdx.x < cnt;
    const u64 key = ingest_one<COMPACT>(t, stage + (size_t)threadIdx.x * RSZ, in_range, pol, npol, now_batch, i, drec, out);
    if (in_range) sortkeys[i] = key;
}

// ---------------------------------------------------------------------------------------------
// K1b: stable LSD radix sort on the slot bits of (slot << 32 | index), one sweep per pass
// ---------------------------------------------------------------------------------------------
// One launch reads the keys once and builds the digit histograms of every pass (sort_digits_hist_kernel).  Then
// one launch per pass (sort_onesweep_kernel): a CTA ranks one tile of keys in shared memory, publishes the tile's
// count of every digit, finds the counts of all tiles before it by decoupled look-back, and scatters.  A CTA takes
// its tile from a ticket counter, so tiles are handed out in the order CTAs start: a tile only ever waits on tiles
// that running (or finished) CTAs hold, and those publish their counts before they wait on anything.  No grid
// barrier, no assumption about how many CTAs are resident.
#ifndef GCRA_SORT_ITEMS
#define GCRA_SORT_ITEMS 16
#endif
constexpr int SORT_ITEMS = GCRA_SORT_ITEMS;                // items per thread
constexpr int SORT_TILE = TILE_THREADS * SORT_ITEMS;       // 4096 keys per tile
// CTAs per SM of the one-sweep kernel: 2 x 148 SMs hold all 256 tiles of a 2^20-key sort at once, with registers
// for every thread's 16 keys (no spills)
constexpr int SORT_MIN_CTAS = 2;
constexpr int SORT_MAX_BITS = 9;
constexpr int SORT_MAX_DIGITS = 1 << SORT_MAX_BITS;
constexpr int SORT_MAX_PASSES = 4;                         // slot_bits <= 32: at most 4 passes of 8 bits
constexpr int SORT_HIST_KEYS = 2 * SORT_TILE;              // keys per CTA of the histogram kernel
constexpr int SORT_LOOKBACK = 4;                           // predecessor words read per look-back step

// digit width of pass p: `bits` slot bits over `passes` passes, the first bits % passes passes one bit wider
__host__ __device__ __forceinline__ u32 sort_pass_bits(u32 bits, u32 passes, u32 p) {
    return bits / passes + (p < bits % passes ? 1u : 0u);
}

// block-wide exclusive scan of one value per thread (warp shuffles + one shared-memory hop);
// returns the exclusive prefix, the block total in *total
__device__ __forceinline__ u32 block_exclusive_scan(u32 v, u32 *part, u32 *total) {
    const u32 lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u32 inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        u32 t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (u32)o) inc += t;
    }
    if (lane == 31) part[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        u32 w = lane < TILE_THREADS / 32 ? part[lane] : 0;
#pragma unroll
        for (int o = 1; o < TILE_THREADS / 32; o <<= 1) {
            u32 t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= (u32)o) w += t;
        }
        if (lane < TILE_THREADS / 32) part[lane] = w;          // inclusive over warps
    }
    __syncthreads();
    const u32 before = warp > 0 ? part[warp - 1] : 0;
    *total = part[TILE_THREADS / 32 - 1];
    return before + inc - v;
}

// The sort kernels take the element count either from the host (`n`) or -- when `n_dev` is given -- from device
// memory: the residue of the index-order pipeline is only known on the device, its launches are sized for the
// largest residue and the tiles beyond the count exit.
__device__ __forceinline__ u32 sort_count(u32 n, const u32 *__restrict__ n_dev) { return n_dev ? *n_dev : n; }

// tot: this sort's digit totals [SORT_MAX_PASSES][SORT_MAX_DIGITS], zero on entry.  clear: the other half of the
// double buffer, the totals of the previous sort on this scratch set (every pass of it has finished): zeroed here
// for the next sort, so no memset is needed.
__global__ void __launch_bounds__(TILE_THREADS)
sort_digits_hist_kernel(const u64 *__restrict__ in, u32 n_host, const u32 *__restrict__ n_dev, u32 bits, u32 passes,
                        u32 *__restrict__ tot, u32 *__restrict__ clear) {
    __shared__ u32 h[SORT_MAX_PASSES * SORT_MAX_DIGITS];
    for (u32 i = threadIdx.x; i < SORT_MAX_PASSES * SORT_MAX_DIGITS; i += TILE_THREADS) {
        h[i] = 0;
        if (blockIdx.x == 0) clear[i] = 0;
    }
    u32 shift[SORT_MAX_PASSES], mask[SORT_MAX_PASSES];
    {
        u32 s = 32;
#pragma unroll
        for (int p = 0; p < SORT_MAX_PASSES; p++) {
            const u32 pb = (u32)p < passes ? sort_pass_bits(bits, passes, p) : 0;
            shift[p] = s;
            mask[p] = (1u << pb) - 1;
            s += pb;
        }
    }
    __syncthreads();
    const u32 n = sort_count(n_host, n_dev);
    for (u32 base = blockIdx.x * SORT_TILE; base < n; base += gridDim.x * SORT_TILE) {
        u64 key[SORT_ITEMS];
#pragma unroll
        for (int k = 0; k < SORT_ITEMS; k++) {
            const u32 i = base + k * TILE_THREADS + threadIdx.x;
            key[k] = i < n ? in[i] : 0;
        }
#pragma unroll
        for (int k = 0; k < SORT_ITEMS; k++) {
            if (base + k * TILE_THREADS + threadIdx.x >= n) continue;
#pragma unroll
            for (int p = 0; p < SORT_MAX_PASSES; p++)
                if ((u32)p < passes) atomicAdd(&h[p * SORT_MAX_DIGITS + ((u32)(key[k] >> shift[p]) & mask[p])], 1u);
        }
    }
    __syncthreads();
    for (u32 i = threadIdx.x; i < passes * SORT_MAX_DIGITS; i += TILE_THREADS)
        if (h[i]) atomicAdd(&tot[i], h[i]);
}

// Look-back status of (tile, digit) in one 64-bit word: [63:33] the pass's sequence number, [32] 1 = inclusive
// prefix over tiles 0..tile, 0 = this tile's count only, [31:0] the count.  Every pass of every sort on a scratch
// set gets a new sequence number (never 0), so words left by earlier passes read as "not published yet" and the
// array is never cleared between passes.
constexpr u64 SORT_STATUS_INCL = 1ULL << 32;
constexpr u32 SORT_SEQ_LIMIT = 1u << 31;
__device__ __forceinline__ u64 sort_status(u32 seq, bool incl, u32 count) {
    return ((u64)seq << 33) | (incl ? SORT_STATUS_INCL : 0) | count;
}
__device__ __forceinline__ u64 ld_relaxed_gpu(const u64 *p) {
    u64 v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_gpu(u64 *p, u64 v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

struct SortOnesweepSmem {
    u32 cnt[TILE_THREADS / 32][SORT_MAX_DIGITS];   // per-warp digit counters -> per-warp offsets inside the tile
    u32 gbase[SORT_MAX_DIGITS];                    // output position of (digit, this tile)
    u32 part[TILE_THREADS / 32];
    u32 tile;
};

// One pass.  tot: the digit totals of this pass (sort_digits_hist_kernel); status: [tiles][SORT_MAX_DIGITS] look-back
// words; the CTA's tile is atomicAdd(ticket) - ticket_base (the host knows how many tickets earlier launches took).
__global__ void __launch_bounds__(TILE_THREADS, SORT_MIN_CTAS)
sort_onesweep_kernel(const u64 *__restrict__ in, u64 *__restrict__ outk, u32 n_host, const u32 *__restrict__ n_dev,
                     u32 shift, u32 bits, const u32 *__restrict__ tot, u64 *__restrict__ status, u32 *__restrict__ ticket,
                     u32 ticket_base, u32 seq) {
    constexpr int NW = TILE_THREADS / 32;
    __shared__ SortOnesweepSmem sm;
    if (threadIdx.x == 0) sm.tile = atomicAdd(ticket, 1u) - ticket_base;
    const u32 nd = 1u << bits, mask = nd - 1;
    for (u32 d = threadIdx.x; d < nd; d += TILE_THREADS) {
#pragma unroll
        for (int x = 0; x < NW; x++) sm.cnt[x][d] = 0;
    }
    __syncthreads();
    const u32 n = sort_count(n_host, n_dev);
    const u32 tile = sm.tile;
    if ((u64)tile * SORT_TILE >= n) return;       // uniform over the CTA
    const u32 w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const u32 lt = (1u << lane) - 1;
    // warp w owns the tile elements [w * 32 * SORT_ITEMS, (w + 1) * 32 * SORT_ITEMS): item k, lane l -> k * 32 + l,
    // in index order, and ranks them in that order: the sort is stable
    const u32 base = tile * SORT_TILE + w * (32 * SORT_ITEMS);
    u64 key[SORT_ITEMS];
    u32 dig[SORT_ITEMS], rank[SORT_ITEMS];
#pragma unroll
    for (int k = 0; k < SORT_ITEMS; k++) {
        const u32 i = base + k * 32 + lane;
        key[k] = i < n ? in[i] : 0;
    }
#pragma unroll
    for (int k = 0; k < SORT_ITEMS; k++) {
        const bool valid = base + k * 32 + lane < n;
        dig[k] = (u32)(key[k] >> shift) & mask;
        const u32 peers = __match_any_sync(0xffffffffu, valid ? dig[k] : (0x80000000u | lane));
        const u32 before = valid ? sm.cnt[w][dig[k]] : 0;
        rank[k] = before + __popc(peers & lt);
        __syncwarp();
        if (valid && (peers & lt) == 0) sm.cnt[w][dig[k]] = before + __popc(peers);
        __syncwarp();
    }
    // global start of every digit: exclusive scan of the digit totals, two consecutive digits per thread
    // (nd <= 512); the scan's barriers also complete the per-warp counters
    const u32 d0 = 2 * threadIdx.x, d1 = d0 + 1;
    const u32 t0 = d0 < nd ? tot[d0] : 0, t1 = d1 < nd ? tot[d1] : 0;
    u32 total;
    const u32 ex = block_exclusive_scan(t0 + t1, sm.part, &total);
    // per digit: exclusive scan over the warps -> the tile's count, published at once
    u32 agg0 = 0, agg1 = 0;
    if (d0 < nd) {
#pragma unroll
        for (int x = 0; x < NW; x++) { const u32 v = sm.cnt[x][d0]; sm.cnt[x][d0] = agg0; agg0 += v; }
    }
    if (d1 < nd) {
#pragma unroll
        for (int x = 0; x < NW; x++) { const u32 v = sm.cnt[x][d1]; sm.cnt[x][d1] = agg1; agg1 += v; }
    }
    u64 *row = status + (size_t)tile * SORT_MAX_DIGITS;
    if (d0 < nd) st_relaxed_gpu(&row[d0], sort_status(seq, tile == 0, agg0));
    if (d1 < nd) st_relaxed_gpu(&row[d1], sort_status(seq, tile == 0, agg1));
    // look-back: add the predecessors' counts until one has published its inclusive prefix.  SORT_LOOKBACK words
    // of both digits are read at once: a tile that starts with hundreds of others before it reaches an inclusive
    // prefix in a few L2 round trips instead of one per predecessor.
    u32 pre0 = 0, pre1 = 0;
    if (tile > 0) {
        bool done0 = d0 >= nd, done1 = d1 >= nd;
        u32 next0 = tile, next1 = tile;            // tiles [next, tile) are summed
        while (!(done0 && done1)) {
            u64 s0[SORT_LOOKBACK], s1[SORT_LOOKBACK];
#pragma unroll
            for (int j = 0; j < SORT_LOOKBACK; j++) {
                s0[j] = !done0 && (u32)j < next0 ? ld_relaxed_gpu(status + (size_t)(next0 - 1 - j) * SORT_MAX_DIGITS + d0) : 0;
                s1[j] = !done1 && (u32)j < next1 ? ld_relaxed_gpu(status + (size_t)(next1 - 1 - j) * SORT_MAX_DIGITS + d1) : 0;
            }
            bool go0 = !done0, go1 = !done1;       // stop at the first word not published yet, retry from there
#pragma unroll
            for (int j = 0; j < SORT_LOOKBACK; j++) {
                go0 = go0 && (u32)(s0[j] >> 33) == seq;
                if (go0) {
                    pre0 += (u32)s0[j];
                    next0--;
                    if (s0[j] & SORT_STATUS_INCL) { done0 = true; go0 = false; }
                }
                go1 = go1 && (u32)(s1[j] >> 33) == seq;
                if (go1) {
                    pre1 += (u32)s1[j];
                    next1--;
                    if (s1[j] & SORT_STATUS_INCL) { done1 = true; go1 = false; }
                }
            }
        }
        if (d0 < nd) st_relaxed_gpu(&row[d0], sort_status(seq, true, pre0 + agg0));
        if (d1 < nd) st_relaxed_gpu(&row[d1], sort_status(seq, true, pre1 + agg1));
    }
    if (d0 < nd) sm.gbase[d0] = ex + pre0;
    if (d1 < nd) sm.gbase[d1] = ex + t0 + pre1;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < SORT_ITEMS; k++) {
        if (base + k * 32 + lane < n) outk[sm.gbase[dig[k]] + sm.cnt[w][dig[k]] + rank[k]] = key[k];
    }
}

// ---------------------------------------------------------------------------------------------
// A batch as the kernels see it: one segment of n rows (host-known count), or -- multi-GPU, rows written
// by peer GPUs straight into this GPU's inbox -- up to MAX_SEGS segments whose row counts live in device
// memory.  Row id = (segment << cap_shift) | row-in-segment; results of a row go to its segment's result
// array (for a peer's segment that is a peer-mapped pointer: the result travels back over NVLink as it is
// written).
// ---------------------------------------------------------------------------------------------
constexpr int MAX_SEGS = 16;
struct SegDesc {
    const unsigned char *req;
    gcra_result *res;
};
struct BatchView {
    const unsigned char *req0;   // nseg == 1
    gcra_result *res0;
    const SegDesc *segs;         // device array [nseg], nseg > 1
    const u32 *dev_counts;       // device array [nseg], nseg > 1
    u32 n;                       // nseg == 1: number of rows
    u32 nseg;
    u32 cap_shift;               // nseg > 1: log2 of the per-segment row capacity

    __device__ __forceinline__ gcra_result *res_at(u32 i) const {
        if (nseg == 1) return res0 + i;
        return (gcra_result *)__ldg((const u64 *)&segs[i >> cap_shift].res) + (i & ((1u << cap_shift) - 1));
    }
    __device__ __forceinline__ const unsigned char *req_at(u32 i, u32 rsz) const {
        if (nseg == 1) return req0 + (size_t)i * rsz;
        return (const unsigned char *)__ldg((const u64 *)&segs[i >> cap_shift].req) + (size_t)(i & ((1u << cap_shift) - 1)) * rsz;
    }
};

// What the payload `i` of a sorted key stands for.  Sort pipeline: the batch index -- the derived request is
// drec[i], the result goes to out + i.  Residue of the index-order pipeline: the row id -- the request is parsed
// from the batch itself (req_at(i)), the result goes to the row's own place (res_at(i)).
struct OutMap {
    gcra_result *out;
    int by_row;                  // 0: sort pipeline, 1: residue of the index-order pipeline
    int compact;                 // by_row: the batch holds gcra_request16 rows
    BatchView view;
    const PolicyDerived *pol;
    u32 npol;
    i64 now_batch;
    template <bool BY_ROW>
    __device__ __forceinline__ gcra_result *at(u32 i) const { return BY_ROW ? view.res_at(i) : out + i; }
};

// ---------------------------------------------------------------------------------------------
// K1c: decide -- the GCRA theoretical-arrival-time compare-and-update
// ---------------------------------------------------------------------------------------------
// Sorted positions are cut into chunks of 32, one warp per chunk.  A run of equal slots (all
// requests of one key, in index order) is owned by the warp whose chunk holds the run's first
// element; when a run crosses the chunk end that warp keeps walking it chunk by chunk, carrying
// the key's state in registers, and the warps of the following chunks skip those lanes.
//
// Inside a chunk every lane evaluates its request against the state its run currently has.
// A request that is denied (or leaves the entry bit-for-bit unchanged) does not alter what later
// requests see, so all lanes up to and including the first state-changing lane of a run are final;
// that lane's new state is shuffled to the lanes behind it and only they re-evaluate.  The loop
// runs (state changes in the busiest run of the chunk + 1) times, and yields exactly the results
// of applying the requests one after another.
struct RunState { i64 tat, exp, ei; };   // ei: informational column only, never part of a decision

__device__ __forceinline__ void run_chunk(u32 lane, bool mine, u32 gmask, const Req &r, RunState &s,
                                          Decision &fin, bool &changed_any, u32 &n_exp_hits) {
    // on return: fin = this lane's decision; s = state after this lane (its run's state)
    const u32 lt = (1u << lane) - 1;
    bool pending = mine;
    bool mflag = false;
    for (;;) {
        Decision d;
        bool mut = false;
        i64 so_tat = s.tat, so_exp = s.exp;
        if (pending) {
            d = decide(s.tat, s.exp, r);
            if (d.allowed) {
                so_tat = d.new_tat; so_exp = d.new_exp;
                mut = (so_tat != s.tat) | (so_exp != s.exp);
            }
        }
        const u32 M = __ballot_sync(0xffffffffu, pending && mut);
        const u32 prior = M & gmask & lt;                  // state-changing lanes of my run before me
        const bool final_now = pending && prior == 0;
        const u32 behind = __ballot_sync(0xffffffffu, pending && prior != 0);
        if (final_now) {
            fin = d;
            // a write over an entry that exists but is expired (adaptive_cleanup.rs:233,267)
            if (d.allowed && !d.live && s.exp >= 0) n_exp_hits++;
            if (mut) { s.tat = so_tat; s.exp = so_exp; mflag = true; }
            pending = false;
        }
        if (behind == 0) break;                            // common case: one pass, no shuffles
        const int src = prior ? (__ffs(prior) - 1) : (int)lane;
        const i64 sn_tat = __shfl_sync(0xffffffffu, so_tat, src);
        const i64 sn_exp = __shfl_sync(0xffffffffu, so_exp, src);
        if (pending) { s.tat = sn_tat; s.exp = sn_exp; }
    }
    changed_any = mflag;
}

// A run of LONG_RUN_MIN or more requests on one key (a hot key) is not walked by its warp: the warp
// appends (first position, length) to a work list and decide_long_kernel gives it a whole CTA.
#ifndef GCRA_LONG_MIN
#define GCRA_LONG_MIN 256
#endif
#ifndef GCRA_GIANT_MIN
#define GCRA_GIANT_MIN 4096
#endif
#ifndef GCRA_CLUSTER
#define GCRA_CLUSTER 8
#endif
constexpr u32 LONG_RUN_MIN = GCRA_LONG_MIN;     // >= this: one CTA per run (decide_runs_kernel<1>)
constexpr u32 GIANT_RUN_MIN = GCRA_GIANT_MIN;   // >= this: one cluster per run (decide_runs_kernel<CLUSTER_CTAS>)
constexpr int LONG_THREADS = 512;
constexpr int CLUSTER_CTAS = GCRA_CLUSTER;
struct LongRun { u32 start, len; };

template <bool BY_ROW>
__device__ __forceinline__ void load_req(const Req *__restrict__ drec, const OutMap &om, u32 idx, Req &r) {
    if (BY_ROW) {
        // (rows in the residue passed validation in pass A: the status is 0)
        u64 key_hash;
        if (om.compact) parse_request<true>(om.view.req_at(idx, sizeof(gcra_request16)), om.pol, om.npol, om.now_batch, key_hash, r);
        else parse_request<false>(om.view.req_at(idx, sizeof(gcra_request)), nullptr, 0, 0, key_hash, r);
        return;
    }
    longlong2 a = reinterpret_cast<const longlong2 *>(drec + idx)[0];
    longlong2 b = reinterpret_cast<const longlong2 *>(drec + idx)[1];
    r.now = a.x; r.ei = a.y; r.dvt = b.x; r.q = b.y;
}

// first position >= lo whose slot differs from run_slot; sorted[lo] is known to be in the run.
// Warp-cooperative 32-ary search (all lanes call it; result uniform).
__device__ __forceinline__ u32 run_end(const u64 *__restrict__ sorted, u32 n, u32 lo, u32 run_slot, u32 lane) {
    u32 hi = n;   // sorted[hi] (if any) is outside the run
    while (hi - lo > 1) {
        u32 p = lo + (u32)(((u64)(hi - lo) * (lane + 1)) / 33);
        bool in = (u32)(sorted[p] >> 32) == run_slot;    // lo <= p < hi <= n
        u32 m = __ballot_sync(0xffffffffu, in);          // monotone: a prefix of lanes
        int k = __popc(m);
        u32 plo = __shfl_sync(0xffffffffu, p, k > 0 ? k - 1 : 0);
        u32 phi = __shfl_sync(0xffffffffu, p, k < 32 ? k : 31);
        if (k > 0) lo = plo;
        if (k < 32) hi = phi;
    }
    return hi;
}

__device__ __forceinline__ void load_state(const Table &t, u32 slot, RunState &s) {
    const longlong2 v = *reinterpret_cast<const longlong2 *>(&t.state[slot]);   // LDG.128
    s.tat = v.x;
    s.exp = (i64)((u64)v.x + (u64)v.y);
    s.ei = 0;
}

__device__ __forceinline__ void store_state(const Table &t, u32 slot, const RunState &s, bool created) {
    *reinterpret_cast<longlong2 *>(&t.state[slot]) =
        make_longlong2(s.tat, (i64)((u64)s.exp - (u64)s.tat));                                 // STG.128
    if (created) t.ei[slot] = s.ei;
}

#ifndef GCRA_DECIDE_THREADS
#define GCRA_DECIDE_THREADS 256
#endif
constexpr int DECIDE_THREADS = GCRA_DECIDE_THREADS;   // warps are independent: the CTA size only sets scheduling granularity

// one warp, one chunk of 32 sorted positions (see the comment above run_chunk); BY_ROW: the sorted payload is a row
// id of the batch (residue of the index-order pipeline), else a batch index into drec / out
template <bool BY_ROW>
__device__ __forceinline__ void decide_chunk(const Table &t, const u64 *sorted, const Req *__restrict__ drec, u32 n,
                                             const OutMap &out, LongRun *__restrict__ long_runs,
                                             LongRun *__restrict__ giant_runs, u32 *__restrict__ long_count,
                                             u32 warp_global, u32 lane, int mode = 0) {
    // mode 0: find the hot runs (work lists) and decide everything else; 1: only find the hot runs; 2: only
    // decide (the lists were written by a mode-1 launch, the hot-run kernels already work on them)
    const u32 base = warp_global * 32;
    if (base >= n) return;   // whole warp

    const u32 pos = base + lane;
    const u64 e = pos < n ? sorted[pos] : ~0ULL;
    const u32 slot = (u32)(e >> 32);
    const bool valid = pos < n && slot != t.null_slot;
    // slot of the element just before this chunk, and just after it
    const u32 prev_last = base > 0 ? (u32)(sorted[base - 1] >> 32) : 0xffffffffu;
    const u32 next_first = base + 32 < n ? (u32)(sorted[base + 32] >> 32) : 0xffffffffu;
    u32 prev = __shfl_up_sync(0xffffffffu, slot, 1);
    if (lane == 0) prev = prev_last;
    // lanes continuing a run that started in an earlier chunk belong to that chunk's warp
    const u32 slot0 = __shfl_sync(0xffffffffu, slot, 0);
    const u32 same0 = __ballot_sync(0xffffffffu, valid && slot == slot0);   // sorted => a prefix
    const u32 foreign = (base > 0 && slot0 == prev_last) ? same0 : 0;
    bool mine = valid && !((foreign >> lane) & 1);
    const bool head = mine && slot != prev;
    const u32 heads = __ballot_sync(0xffffffffu, head);
    const u32 le = (lane == 31) ? 0xffffffffu : ((2u << lane) - 1);
    const int hl = mine ? (31 - __clz(heads & le)) : (int)lane;
    // lanes of my run: from my head lane up to (not including) the next head, among `mine` lanes
    u32 gmask = 1u << lane;
    {
        const u32 mine_m = __ballot_sync(0xffffffffu, mine);
        if (mine) {
            const u32 above = heads & ~((hl == 31) ? 0xffffffffu : ((2u << hl) - 1));   // heads after mine
            const u32 upto = above ? ((1u << (__ffs(above) - 1)) - 1) : 0xffffffffu;     // lanes below the next head
            gmask = mine_m & upto & ~((1u << hl) - 1);
        }
    }

    // does the chunk's last run continue past the chunk?  (uniform)
    const u32 slot31 = __shfl_sync(0xffffffffu, slot, 31);
    const bool mine31 = __shfl_sync(0xffffffffu, mine ? 1 : 0, 31) != 0;
    bool cont = mine31 && next_first == slot31;
    const u32 gmask31 = __shfl_sync(0xffffffffu, gmask, 31);
    if (cont) {
        const u32 run_start = base + (u32)(__ffs(gmask31) - 1);
        const u32 end = run_end(sorted, n, base + 32, slot31, lane);
        if (end - run_start >= LONG_RUN_MIN) {
            // hot key: hand the whole run (including its lanes here) to decide_long_kernel
            if (lane == 0 && mode != 2) {
                const bool giant = end - run_start >= GIANT_RUN_MIN;
                u32 w = atomicAdd(long_count + (giant ? 1 : 0), 1u);
                LongRun *dst = giant ? giant_runs : long_runs;
                dst[w].start = run_start;
                dst[w].len = end - run_start;
            }
            if ((gmask31 >> lane) & 1) mine = false;
            cont = false;
        }
    }
    if (mode == 1) return;

    Req r = {0, 0, 0, 0};
    const u32 idx = (u32)e;
    if (mine) load_req<BY_ROW>(drec, out, idx, r);
    // run heads read the entry; the run's lanes get it by shuffle
    RunState s = {0, EXP_EMPTY, 0};
    if (head && mine) load_state(t, slot, s);
    s.tat = __shfl_sync(0xffffffffu, s.tat, hl);
    s.exp = __shfl_sync(0xffffffffu, s.exp, hl);
    const bool was_phantom = s.exp < 0;              // the key has no entry yet (same for every lane of the run)

    Decision fin;
    bool changed = false;
    u32 exp_hits = 0;
    run_chunk(lane, mine, gmask, r, s, fin, changed, exp_hits);

    u32 n_allowed = 0, n_denied = 0;
    if (mine) {
        Outputs o = outputs_of(fin, r);
        write_result(out.template at<BY_ROW>(idx), o.remaining, o.reset_after, o.retry_after, 0, fin.allowed ? 1 : 0);
        n_allowed += fin.allowed ? 1 : 0;
        n_denied += fin.allowed ? 0 : 1;
    }
    // run tails: last lane of each run inside this chunk writes the run's state back
    const u32 run_changed_mask = __ballot_sync(0xffffffffu, mine && changed);
    const bool run_changed = (run_changed_mask & gmask) != 0;
    const u32 next_slot_in = __shfl_down_sync(0xffffffffu, slot, 1);
    const u32 mine_mask = __ballot_sync(0xffffffffu, mine);
    const bool next_mine = lane < 31 && ((mine_mask >> (lane + 1)) & 1);
    const bool tail = mine && (!next_mine || next_slot_in != slot);

    u32 real_inc = 0;
    // informational ei column: emission interval of the run's first request in the creating batch
    s.ei = __shfl_sync(0xffffffffu, r.ei, hl);
    if (tail && !(cont && lane == 31) && run_changed) {
        store_state(t, slot, s, was_phantom);
        if (was_phantom) real_inc++;
    }

    if (cont) {
        // walk the rest of lane 31's run (< LONG_RUN_MIN requests), next chunk prefetched
        RunState cs;
        cs.tat = __shfl_sync(0xffffffffu, s.tat, 31);
        cs.exp = __shfl_sync(0xffffffffu, s.exp, 31);
        cs.ei = __shfl_sync(0xffffffffu, s.ei, 31);   // (set below: ei of the run's first request)
        bool c_changed = __shfl_sync(0xffffffffu, run_changed ? 1 : 0, 31) != 0;
        const bool c_phantom = __shfl_sync(0xffffffffu, was_phantom ? 1 : 0, 31) != 0;
        u32 b2 = base + 32;
        u64 e2 = b2 + lane < n ? sorted[b2 + lane] : ~0ULL;
        bool in_run = (u32)(e2 >> 32) == slot31 && b2 + lane < n;
        Req r2 = {0, 0, 0, 0};
        if (in_run) load_req<BY_ROW>(drec, out, (u32)e2, r2);
        for (;;) {
            const u32 rm = __ballot_sync(0xffffffffu, in_run);   // a prefix (sorted)
            if (rm == 0) break;
            // prefetch the following chunk while this one is decided
            const u32 b3 = b2 + 32;
            u64 e3 = ~0ULL;
            bool in3 = false;
            Req r3 = {0, 0, 0, 0};
            if (rm == 0xffffffffu) {
                e3 = b3 + lane < n ? sorted[b3 + lane] : ~0ULL;
                in3 = (u32)(e3 >> 32) == slot31 && b3 + lane < n;
                if (in3) load_req<BY_ROW>(drec, out, (u32)e3, r3);
            }
            RunState s2 = cs;
            Decision f2;
            bool ch2 = false;
            run_chunk(lane, in_run, rm, r2, s2, f2, ch2, exp_hits);
            if (in_run) {
                Outputs o = outputs_of(f2, r2);
                write_result(out.template at<BY_ROW>((u32)e2), o.remaining, o.reset_after, o.retry_after, 0, f2.allowed ? 1 : 0);
                n_allowed += f2.allowed ? 1 : 0;
                n_denied += f2.allowed ? 0 : 1;
            }
            c_changed |= __ballot_sync(0xffffffffu, in_run && ch2) != 0;
            const int last = 31 - __clz(rm);
            cs.tat = __shfl_sync(0xffffffffu, s2.tat, last);
            cs.exp = __shfl_sync(0xffffffffu, s2.exp, last);
            if (rm != 0xffffffffu) break;
            b2 = b3; e2 = e3; in_run = in3; r2 = r3;
        }
        cs.ei = __shfl_sync(0xffffffffu, s.ei, 31);
        if (lane == 31 && c_changed) {
            store_state(t, slot31, cs, c_phantom);
            if (c_phantom) real_inc++;
        }
    }

    // warp-aggregated counters
    n_allowed = __reduce_add_sync(0xffffffffu, n_allowed);
    n_denied = __reduce_add_sync(0xffffffffu, n_denied);
    real_inc = __reduce_add_sync(0xffffffffu, real_inc);
    exp_hits = __reduce_add_sync(0xffffffffu, exp_hits);
    if (lane == 0) {
        if (n_allowed) atomicAdd(&t.counters[C_ALLOWED], (u64)n_allowed);
        if (n_denied) atomicAdd(&t.counters[C_DENIED], (u64)n_denied);
        if (real_inc) atomicAdd(&t.counters[C_REAL], (u64)real_inc);
        if (exp_hits) atomicAdd(&t.counters[C_EXPIRED_HITS], (u64)exp_hits);
    }
}

#ifndef GCRA_DECIDE_MINBLOCKS
#define GCRA_DECIDE_MINBLOCKS (1024 / GCRA_DECIDE_THREADS)
#endif
template <bool BY_ROW>
__global__ void __launch_bounds__(DECIDE_THREADS, GCRA_DECIDE_MINBLOCKS)
decide_kernel(Table t, const u64 *__restrict__ sorted, const Req *__restrict__ drec, u32 n_host,
              const u32 *__restrict__ n_dev, OutMap out, LongRun *__restrict__ long_runs,
              LongRun *__restrict__ giant_runs, u32 *__restrict__ long_count, int mode) {
    const u32 n = sort_count(n_host, n_dev);
    const u32 warps_total = gridDim.x * (DECIDE_THREADS / 32);
    for (u32 wg = (blockIdx.x * DECIDE_THREADS + threadIdx.x) >> 5; wg * 32 < n; wg += warps_total)
        decide_chunk<BY_ROW>(t, sorted, drec, n, out, long_runs, giant_runs, long_count, wg, threadIdx.x & 31, mode);
}

// Small batches (n < LONG_RUN_MIN, e.g. one RateLimiter::rate_limit call or a lightly loaded actor): ONE CTA
// does everything -- ingest, a bitonic sort of the (slot, index) keys in shared memory, and the warp-chunk
// compare-and-update -- instead of 13 launches.  No run can reach LONG_RUN_MIN, so no work list is produced.
constexpr u32 SMALL_MAX = 255;
static_assert(SMALL_MAX < GCRA_LONG_MIN && SMALL_MAX < TILE_THREADS, "small path must not create long runs");

template <bool COMPACT>
__global__ void __launch_bounds__(TILE_THREADS)
small_batch_kernel(Table t, const void *__restrict__ req_base, const PolicyDerived *__restrict__ pol, u32 npol,
                   i64 now_batch, u32 n, Req *__restrict__ drec, gcra_result *__restrict__ out) {
    constexpr u32 RSZ = COMPACT ? sizeof(gcra_request16) : sizeof(gcra_request);
    __shared__ u64 keys[TILE_THREADS];
    const u32 tid = threadIdx.x;
    const bool in_range = tid < n;
    const u64 key = ingest_one<COMPACT>(t, (const unsigned char *)req_base + (size_t)(in_range ? tid : 0) * RSZ, in_range,
                                        pol, npol, now_batch, tid, drec, out);
    keys[tid] = in_range ? key : ~0ULL;
    __syncthreads();
    // bitonic sort of 256 keys; (slot << 32 | index) is a total order, so equal slots stay in index order
    for (u32 k = 2; k <= TILE_THREADS; k <<= 1) {
        for (u32 j = k >> 1; j > 0; j >>= 1) {
            const u32 partner = tid ^ j;
            if (partner > tid) {
                const u64 a = keys[tid], b = keys[partner];
                const bool up = (tid & k) == 0;
                if ((a > b) == up) { keys[tid] = b; keys[partner] = a; }
            }
            __syncthreads();
        }
    }
    __threadfence_block();   // drec / state written above are read below by other warps of this CTA
    OutMap om;
    om.out = out;
    om.by_row = 0;
    decide_chunk<false>(t, keys, drec, n, om, nullptr, nullptr, nullptr, tid >> 5, tid & 31);
}

// ---------------------------------------------------------------------------------------------
// Hot keys: runs of >= LONG_RUN_MIN requests get one CTA, runs of >= GIANT_RUN_MIN one 8-CTA cluster.
// ---------------------------------------------------------------------------------------------
// The run is consumed in strides (one request per thread of the group).  Two kinds of round:
//
//  * plain round: every pending thread evaluates its request against the run's current state; the
//    group finds the first state-changing request (min-reduction); everything up to it is final and
//    its new state becomes current.  One round per state change -- fine while changes are rare.
//
//  * finite-state round (after FSM_AFTER state changes in the run): some keys flip between a few
//    states all the time (max_burst = 1: every zero-quantity request toggles the entry, SURVEY V8), which
//    would cost one round per flip.  The threads keep the last K distinct states of the run as
//    candidates, each request becomes a map "candidate in -> candidate out" (a nibble per candidate,
//    0xF = leaves the candidate set), the maps are composed with an inclusive prefix scan (shuffles,
//    shared memory, distributed shared memory across the cluster), and every request reads its TRUE
//    input state off the scan.  A round is only repeated when a request creates a state that is not a
//    candidate yet.  Still exact: each decision is decide(true input state, request).
constexpr int FSM_K = 4;
constexpr u32 FSM_NEW = 0xF;
constexpr u32 FSM_IDENT = 0x3210;
constexpr u32 FSM_AFTER = 4;

__device__ __forceinline__ u32 fsm_compose(u32 f, u32 g) {   // first f, then g
    const u64 gg = (u64)g | (0xFULL << 60);
    u32 r = 0;
#pragma unroll
    for (int c = 0; c < FSM_K; c++) {
        const u32 x = (f >> (4 * c)) & 0xF;
        r |= ((u32)(gg >> (4 * x)) & 0xF) << (4 * c);
    }
    return r;
}

struct Cands {
    i64 tat[FSM_K], exp[FSM_K];
    __device__ __forceinline__ void get(u32 i, i64 &t, i64 &e) const {
        t = tat[0]; e = exp[0];
#pragma unroll
        for (int c = 1; c < FSM_K; c++) if (i == (u32)c) { t = tat[c]; e = exp[c]; }
    }
    __device__ __forceinline__ void set(u32 i, i64 t, i64 e) {
#pragma unroll
        for (int c = 0; c < FSM_K; c++) if (i == (u32)c) { tat[c] = t; exp[c] = e; }
    }
    __device__ __forceinline__ u32 find(u32 nc, i64 t, i64 e) const {
        u32 j = FSM_NEW;
#pragma unroll
        for (int c = 0; c < FSM_K; c++) if ((u32)c < nc && tat[c] == t && exp[c] == e) j = c;
        return j;
    }
};

struct PubState { i64 tat, exp; };

template <int CTAS, bool BY_ROW>
__global__ void __launch_bounds__(LONG_THREADS, 1)
decide_runs_kernel(Table t, const u64 *__restrict__ sorted, const Req *__restrict__ drec,
                   OutMap out, const LongRun *__restrict__ runs,
                   const u32 *__restrict__ count_ptr) {
    namespace cg = cooperative_groups;
    constexpr int NW = LONG_THREADS / 32;
    constexpr u32 STRIDE = CTAS * LONG_THREADS;
    __shared__ u32 sm_warp[2][NW];       // per-warp first-change position / composed map
    __shared__ u32 sm_cta[2];            // this CTA's value, read by the other CTAs of the cluster
    __shared__ PubState sm_pub[2];       // state created in this round (written into every CTA)
    const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    u32 rank = 0, group_id = blockIdx.x, num_groups = gridDim.x;
    if (CTAS > 1) {
        rank = cg::this_cluster().block_rank();
        group_id = blockIdx.x / CTAS;
        num_groups = gridDim.x / CTAS;
    }
    auto group_sync = [&]() {
        if (CTAS > 1) cg::this_cluster().sync(); else __syncthreads();
    };
    const u32 gpos = rank * LONG_THREADS + tid;          // position inside a stride
    const u32 count = *count_ptr;
    u32 n_allowed = 0, n_denied = 0, exp_hits = 0, real_inc = 0;
    u32 par = 0;
    for (u32 item = group_id; item < count; item += num_groups) {
        const u32 start = runs[item].start, len = runs[item].len;
        const u32 slot = (u32)(sorted[start] >> 32);
        RunState s0;
        load_state(t, slot, s0);
        const bool was_phantom = s0.exp < 0;           // the key has no entry yet
        Cands cd;
#pragma unroll
        for (int c = 0; c < FSM_K; c++) { cd.tat[c] = s0.tat; cd.exp[c] = s0.exp; }
        u32 nc = 1, cur = 0, victim = 0, n_changes = 0;
        // software pipeline: the next stride's request is loaded while this one is decided
        bool active = gpos < len;
        u32 idx = 0;
        Req r = {0, 0, 0, 0};
        if (active) { idx = (u32)sorted[start + gpos]; load_req<BY_ROW>(drec, out, idx, r); }
        for (u32 off = 0; off < len; off += STRIDE) {
            const u32 noff = off + STRIDE;
            const bool nactive = noff + gpos < len;
            u32 nidx = 0;
            Req nr = {0, 0, 0, 0};
            if (nactive) { nidx = (u32)sorted[start + noff + gpos]; load_req<BY_ROW>(drec, out, nidx, nr); }
            bool pending = active;
            for (;;) {
                const bool fsm = n_changes >= FSM_AFTER;
                u32 in_idx = cur;            // candidate this thread's request really starts from
                bool has_new;                // some request of this round created a new state
                u32 total = FSM_IDENT;       // composed map of the whole round (fsm rounds)
                u32 my_map = FSM_IDENT;
                if (!fsm) {
                    // ---- plain round: first state-changing request by min-reduction
                    i64 ct, ce;
                    cd.get(cur, ct, ce);
                    bool mut = false;
                    if (pending) {
                        const Decision d = decide(ct, ce, r);
                        mut = d.allowed && ((d.new_tat != ct) | (d.new_exp != ce));
                    }
                    const u32 wmin = __reduce_min_sync(0xffffffffu, (pending && mut) ? gpos : 0xffffffffu);
                    if (lane == 0) sm_warp[par][warp] = wmin;
                    __syncthreads();
                    u32 first = __reduce_min_sync(0xffffffffu, lane < NW ? sm_warp[par][lane] : 0xffffffffu);
                    if (CTAS > 1) {
                        if (tid == 0) sm_cta[par] = first;
                        cg::this_cluster().sync();
                        u32 v = 0xffffffffu;
                        if (lane < CTAS) v = *cg::this_cluster().map_shared_rank(&sm_cta[par], lane);
                        first = __reduce_min_sync(0xffffffffu, v);
                    }
                    has_new = first != 0xffffffffu;
                    if (pending && gpos > first) in_idx = FSM_NEW;       // behind the change: retry
                    if (pending && gpos == first) my_map = (FSM_IDENT & ~(0xFu << (4 * cur))) | (FSM_NEW << (4 * cur));
                } else {
                    // ---- finite-state round
                    if (pending) {
                        my_map = 0;
#pragma unroll
                        for (int c = 0; c < FSM_K; c++) {
                            u32 o = FSM_NEW;
                            if ((u32)c < nc) {
                                const Decision d = decide(cd.tat[c], cd.exp[c], r);
                                o = c;
                                if (d.allowed && ((d.new_tat != cd.tat[c]) | (d.new_exp != cd.exp[c])))
                                    o = cd.find(nc, d.new_tat, d.new_exp);
                            }
                            my_map |= o << (4 * c);
                        }
                    }
                    u32 incl = my_map;
#pragma unroll
                    for (int d = 1; d < 32; d <<= 1) {
                        const u32 o = __shfl_up_sync(0xffffffffu, incl, d);
                        if (lane >= (u32)d) incl = fsm_compose(o, incl);
                    }
                    u32 lane_excl = __shfl_up_sync(0xffffffffu, incl, 1);
                    if (lane == 0) lane_excl = FSM_IDENT;
                    if (lane == 31) sm_warp[par][warp] = incl;
                    __syncthreads();
                    u32 wt = lane < NW ? sm_warp[par][lane] : FSM_IDENT;
#pragma unroll
                    for (int d = 1; d < NW; d <<= 1) {
                        const u32 o = __shfl_up_sync(0xffffffffu, wt, d);
                        if (lane >= (u32)d) wt = fsm_compose(o, wt);
                    }
                    u32 cta_total = __shfl_sync(0xffffffffu, wt, NW - 1);
                    u32 excl = __shfl_sync(0xffffffffu, wt, warp > 0 ? warp - 1 : 0);
                    if (warp == 0) excl = FSM_IDENT;
                    total = cta_total;
                    if (CTAS > 1) {
                        if (tid == 0) sm_cta[par] = cta_total;
                        cg::this_cluster().sync();
                        u32 ctv = FSM_IDENT;
                        if (lane < CTAS) ctv = *cg::this_cluster().map_shared_rank(&sm_cta[par], lane);
#pragma unroll
                        for (int d = 1; d < CTAS; d <<= 1) {
                            const u32 o = __shfl_up_sync(0xffffffffu, ctv, d);
                            if (lane >= (u32)d) ctv = fsm_compose(o, ctv);
                        }
                        total = __shfl_sync(0xffffffffu, ctv, CTAS - 1);
                        u32 cexcl = __shfl_sync(0xffffffffu, ctv, rank > 0 ? rank - 1 : 0);
                        if (rank == 0) cexcl = FSM_IDENT;
                        excl = fsm_compose(cexcl, excl);
                    }
                    excl = fsm_compose(excl, lane_excl);
                    in_idx = (excl >> (4 * cur)) & 0xF;
                    has_new = ((total >> (4 * cur)) & 0xF) == FSM_NEW;
                }
                // ---- finalize every pending request whose true input state is known
                if (pending && in_idx != FSM_NEW) {
                    i64 ct, ce;
                    cd.get(in_idx, ct, ce);
                    const Decision d = decide(ct, ce, r);
                    const Outputs o = outputs_of(d, r);
                    write_result(out.template at<BY_ROW>(idx), o.remaining, o.reset_after, o.retry_after, 0, d.allowed ? 1 : 0);
                    n_allowed += d.allowed ? 1 : 0;
                    n_denied += d.allowed ? 0 : 1;
                    if (d.allowed && !d.live && ce >= 0) exp_hits++;
                    pending = false;
                    if (((my_map >> (4 * in_idx)) & 0xF) == FSM_NEW) {
                        // this request created a state outside the candidate set: publish it
                        PubState ps = {d.new_tat, d.new_exp};
                        if (CTAS > 1) {
                            for (int c = 0; c < CTAS; c++) *cg::this_cluster().map_shared_rank(&sm_pub[par], c) = ps;
                        } else {
                            sm_pub[par] = ps;
                        }
                    }
                }
                if (!has_new) {
                    if (fsm) cur = (total >> (4 * cur)) & 0xF;
                    par ^= 1;
                    break;                                   // uniform over the group: stride done
                }
                group_sync();
                const PubState ps = sm_pub[par];
                par ^= 1;
                u32 v = cd.find(nc, ps.tat, ps.exp);          // plain rounds may return to a known state
                if (v == FSM_NEW) {
                    if (nc < FSM_K) { v = nc; nc++; }
                    else { v = victim; victim = (victim + 1) % FSM_K; }
                    cd.set(v, ps.tat, ps.exp);
                }
                cur = v;
                n_changes++;
            }
            active = nactive; idx = nidx; r = nr;
        }
        if (rank == 0 && tid == 0) {
            RunState fs;
            cd.get(cur, fs.tat, fs.exp);
            if (fs.tat != s0.tat || fs.exp != s0.exp) {
                Req first;
                load_req<BY_ROW>(drec, out, (u32)sorted[start], first);
                fs.ei = first.ei;
                store_state(t, slot, fs, was_phantom);
                if (was_phantom) real_inc++;
            }
        }
        __syncthreads();
    }
    if (CTAS > 1) cg::this_cluster().sync();   // nobody leaves while its shared memory may be accessed remotely
    n_allowed = __reduce_add_sync(0xffffffffu, n_allowed);
    n_denied = __reduce_add_sync(0xffffffffu, n_denied);
    real_inc = __reduce_add_sync(0xffffffffu, real_inc);
    exp_hits = __reduce_add_sync(0xffffffffu, exp_hits);
    if (lane == 0) {
        if (n_allowed) atomicAdd(&t.counters[C_ALLOWED], (u64)n_allowed);
        if (n_denied) atomicAdd(&t.counters[C_DENIED], (u64)n_denied);
        if (real_inc) atomicAdd(&t.counters[C_REAL], (u64)real_inc);
        if (exp_hits) atomicAdd(&t.counters[C_EXPIRED_HITS], (u64)exp_hits);
    }
}

// ---------------------------------------------------------------------------------------------
// K2: sweep -- retain(expiry > now)
// ---------------------------------------------------------------------------------------------
// One thread per slot: a coalesced 128-bit load of the (tat, off) pair (L1 bypass), expiry = tat + off, and
// only the slots whose entry has expired are touched again: the pair is reset to the empty pattern with one
// 128-bit store into the sector that was just read.  The KEY word is left in place (no scattered 8-byte
// writes into sectors the sweep never reads): a key without an entry behaves exactly like an absent key
// (Store::get sees nothing, the next allowed request creates the entry), it just keeps its slot -- which is
// what a key that comes back wants anyway.  purge_kernel reclaims such slots when the table gets crowded.
__device__ __forceinline__ ulonglong2 ld_stream(const void *p) {
    ulonglong2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u64 {%0, %1}, [%2];" : "=l"(v.x), "=l"(v.y) : "l"(p));
    return v;
}

constexpr int SWEEP_UNROLL = 4;

// One thread per 32-byte SECTOR of the state array (two slots): two 128-bit loads, and when either entry has
// expired the whole sector is written back (two 128-bit stores), so DRAM only ever sees full-sector writes.
// `mode` (tuning, GCRA_SWEEP_MODE): 0 plain stores; 1 streaming stores (st.global.cs: the reset pairs are not read
// again soon, they need not displace the scan's lines in L2); 2 only the expired 16-byte pair is written.
__device__ __forceinline__ void st_stream(void *p, longlong2 v) {
    asm volatile("st.global.cs.v2.s64 [%0], {%1, %2};" ::"l"(p), "l"(v.x), "l"(v.y) : "memory");
}

__global__ void __launch_bounds__(TILE_THREADS)
sweep_kernel(Table t, u64 total_slots, i64 now, int mode) {
    u32 removed = 0;
    const u64 total_pairs = total_slots >> 1;            // the slot count is a power of two >= 64
    const u64 stride = (u64)gridDim.x * TILE_THREADS;
    u64 i = (u64)blockIdx.x * TILE_THREADS + threadIdx.x;
    while (i < total_pairs) {
        ulonglong2 a[SWEEP_UNROLL], b[SWEEP_UNROLL];
#pragma unroll
        for (int u = 0; u < SWEEP_UNROLL; u++) {
            const u64 p = i + (u64)u * stride;
            a[u] = make_ulonglong2(0, (u64)EXP_EMPTY);
            b[u] = a[u];
            if (p < total_pairs) { a[u] = ld_stream(&t.state[2 * p]); b[u] = ld_stream(&t.state[2 * p + 1]); }
        }
#pragma unroll
        for (int u = 0; u < SWEEP_UNROLL; u++) {
            const u64 p = i + (u64)u * stride;
            const i64 ea = (i64)(a[u].x + a[u].y), eb = (i64)(b[u].x + b[u].y);
            const bool xa = ea >= 0 && ea <= now, xb = eb >= 0 && eb <= now;   // entries Store::get no longer shows
            if (xa | xb) {
                longlong2 *dst = reinterpret_cast<longlong2 *>(&t.state[2 * p]);
                const longlong2 va = xa ? make_longlong2(0, EXP_EMPTY) : make_longlong2((i64)a[u].x, (i64)a[u].y);
                const longlong2 vb = xb ? make_longlong2(0, EXP_EMPTY) : make_longlong2((i64)b[u].x, (i64)b[u].y);
                if (mode == 1) { st_stream(dst, va); st_stream(dst + 1, vb); }
                else if (mode == 2) { if (xa) dst[0] = va; if (xb) dst[1] = vb; }
                else { dst[0] = va; dst[1] = vb; }
                removed += (xa ? 1 : 0) + (xb ? 1 : 0);
            }
        }
        i += (u64)SWEEP_UNROLL * stride;
    }
    removed = __reduce_add_sync(0xffffffffu, removed);
    if ((threadIdx.x & 31) == 0 && removed) {
        atomicAdd(&t.counters[C_REAL], (u64)(0 - (u64)removed));
        atomicAdd(&t.counters[C_SWEPT], (u64)removed);
    }
}

// Reclaim the slots of keys that hold no entry (swept, or only ever denied): exclusive pass run by the host
// before it would otherwise grow the table.  Reads key + state of every slot, clears such keys
// (stash: tombstone, so probing continues past them).
__global__ void __launch_bounds__(TILE_THREADS)
purge_kernel(Table t, u64 total_slots) {
    u32 freed = 0, freed_stash = 0;
    const u64 stride = (u64)gridDim.x * TILE_THREADS;
    for (u64 k = (u64)blockIdx.x * TILE_THREADS + threadIdx.x; k < total_slots; k += stride) {
        const ulonglong2 v = ld_stream(&t.state[k]);
        if ((i64)(v.x + v.y) >= 0) continue;
        if (t.keys[k] < 2) continue;
        const bool stash = k >= (u64)t.nb_main * 4;
        t.keys[k] = stash ? KEY_TOMB : KEY_EMPTY;
        freed++;
        if (stash) freed_stash++;
    }
    freed = __reduce_add_sync(0xffffffffu, freed);
    freed_stash = __reduce_add_sync(0xffffffffu, freed_stash);
    if ((threadIdx.x & 31) == 0 && freed) {
        atomicAdd(&t.counters[C_OCCUPIED], (u64)(0 - (u64)freed));
        if (freed_stash) atomicAdd(&t.counters[C_STASH], (u64)(0 - (u64)freed_stash));
    }
}

// fill slots [first, first+count) with the empty pattern (also resets an emptied stash)
__global__ void __launch_bounds__(TILE_THREADS)
clear_slots_kernel(Table t, u64 first, u64 count) {
    const u64 stride = (u64)gridDim.x * TILE_THREADS;
    for (u64 i = (u64)blockIdx.x * TILE_THREADS + threadIdx.x; i < count; i += stride) {
        t.keys[first + i] = KEY_EMPTY;
        *reinterpret_cast<longlong2 *>(&t.state[first + i]) = make_longlong2(0, EXP_EMPTY);
        t.ei[first + i] = 0;
    }
}

// re-insert every entry of `src` into the (empty, larger) table `dst` -- HashMap growth
__global__ void __launch_bounds__(TILE_THREADS)
rehash_kernel(Table src, u64 src_slots, Table dst) {
    const u64 stride = (u64)gridDim.x * TILE_THREADS;
    for (u64 i = (u64)blockIdx.x * TILE_THREADS + threadIdx.x; i < src_slots; i += stride) {
        u64 k = src.keys[i];
        if (k < 2) continue;
        TatOff st = src.state[i];
        if ((i64)((u64)st.tat + st.off) < 0) continue;   // keys without an entry are not carried over
        bool fresh;
        u32 s = find_or_claim(dst, k, fresh);
        if (s == dst.null_slot) { atomicAdd(&dst.counters[C_INSERT_FAIL], 1ULL); continue; }
        dst.state[s] = st;
        dst.ei[s] = src.ei[i];
        atomicAdd(&dst.counters[C_OCCUPIED], 1ULL);
        atomicAdd(&dst.counters[C_REAL], 1ULL);
    }
}

// ---------------------------------------------------------------------------------------------
// Store-trait single operations (core/store/mod.rs:85-133): one thread, results in `res`
// ---------------------------------------------------------------------------------------------
struct StoreOpResult { i64 value; int flag; int status; };

// op: 0 get (adaptive_cleanup.rs:246-252), 1 cas (:221-244), 2 set_nx (:254-278),
//     3 peek (entry as stored: res[0].value = tat, res[1].value = expiry)
__device__ __forceinline__ i64 expiry_of(i64 now, u64 ttl) {
    u64 e = (u64)now + ttl;
    return (e < ttl || e > (u64)I64_MAX) ? I64_MAX : (i64)e;
}

__global__ void store_op_kernel(Table t, int op, u64 key, i64 a, i64 b, u64 ttl, i64 now,
                                StoreOpResult *res) {
    StoreOpResult r = {0, 0, 0};
    if (op == 2) {
        bool fresh;
        u32 s = find_or_claim(t, key, fresh);
        if (s == t.null_slot) {
            r.status = GCRA_INTERNAL;
        } else {
            TatOff *l = t.state + s;
            if (fresh) atomicAdd(&t.counters[C_OCCUPIED], 1ULL);
            i64 ex = (i64)((u64)l->tat + l->off);   // EXP_EMPTY for a fresh or entry-less key
            if (ex > now) {
                r.flag = 0;                                  // live entry: :264-265
            } else {
                l->tat = a;
                l->off = (u64)expiry_of(now, ttl) - (u64)a;
                r.flag = 1;
                atomicAdd(&t.counters[C_ALLOWED], 1ULL);     // one mutating op
                if (ex < 0) atomicAdd(&t.counters[C_REAL], 1ULL);
                else atomicAdd(&t.counters[C_EXPIRED_HITS], 1ULL);   // :267
            }
        }
    } else {
        u32 s = find_slot(t, key);
        if (s != t.null_slot) {
            TatOff *l = t.state + s;
            i64 tat = l->tat;
            i64 ex = (i64)((u64)tat + l->off);
            if (op == 3) {
                if (ex >= 0) { r.flag = 1; r.value = tat; res[1].value = ex; }
            } else if (ex > now) {
                if (op == 0) { r.flag = 1; r.value = tat; }
                else if (tat == a) {                         // :236-240
                    l->tat = b;
                    l->off = (u64)expiry_of(now, ttl) - (u64)b;
                    r.flag = 1;
                    atomicAdd(&t.counters[C_ALLOWED], 1ULL);
                }
            } else if (op == 1 && ex >= 0) {
                atomicAdd(&t.counters[C_EXPIRED_HITS], 1ULL);        // :232-235
            }
        }
    }
    res[0] = r;
}

// ---------------------------------------------------------------------------------------------
// K3: routing for the hash-sharded multi-GPU engine -- stable partition by owner shard
// ---------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ u32 owner_of(u64 key_hash, u32 n_shards) {
    // bits independent of the in-table bucket choices (those use mix64's low/high words directly)
    u64 m = mix64(key_hash ^ 0xA24BAED4963EE407ULL);
    return (u32)(((m >> 32) * (u64)n_shards) >> 32);
}

constexpr int ROUTE_MAX_SHARDS = 16;

__global__ void __launch_bounds__(TILE_THREADS)
route_count_kernel(const gcra_request *__restrict__ req, u32 n, u32 n_shards, u32 num_tiles,
                   u32 *__restrict__ tile_counts) {
    __shared__ u32 c[ROUTE_MAX_SHARDS];
    if (threadIdx.x < ROUTE_MAX_SHARDS) c[threadIdx.x] = 0;
    __syncthreads();
    u32 i = blockIdx.x * TILE_THREADS + threadIdx.x;
    if (i < n) atomicAdd(&c[owner_of(req[i].key_hash, n_shards)], 1u);
    __syncthreads();
    if (threadIdx.x < n_shards) tile_counts[threadIdx.x * num_tiles + blockIdx.x] = c[threadIdx.x];
}

// single CTA: exclusive scan of tile_counts in (shard, tile) order; per-shard totals to counts
__global__ void __launch_bounds__(TILE_THREADS)
route_scan_kernel(u32 *__restrict__ tile_counts, u32 n_shards, u32 num_tiles, u32 *__restrict__ counts) {
    __shared__ u32 part[TILE_THREADS];
    __shared__ u32 carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (u32 s = 0; s < n_shards; s++) {
        u32 shard_start = carry;
        u32 *row = tile_counts + s * num_tiles;
        for (u32 b = 0; b < num_tiles; b += TILE_THREADS) {
            u32 i = b + threadIdx.x;
            u32 v = i < num_tiles ? row[i] : 0;
            part[threadIdx.x] = v;
            __syncthreads();
            for (u32 off = 1; off < TILE_THREADS; off <<= 1) {
                u32 x = threadIdx.x >= off ? part[threadIdx.x - off] : 0;
                __syncthreads();
                part[threadIdx.x] += x;
                __syncthreads();
            }
            if (i < num_tiles) row[i] = carry + part[threadIdx.x] - v;
            __syncthreads();
            if (threadIdx.x == 0) carry += part[TILE_THREADS - 1];
            __syncthreads();
        }
        if (threadIdx.x == 0) counts[s] = carry - shard_start;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(TILE_THREADS)
route_scatter_kernel(const gcra_request *__restrict__ req, u32 n, u32 n_shards, u32 num_tiles,
                     const u32 *__restrict__ tile_offsets, gcra_request *__restrict__ out,
                     u32 *__restrict__ src_index) {
    constexpr int NW = TILE_THREADS / 32;
    __shared__ u32 wc[NW][ROUTE_MAX_SHARDS];
    const u32 w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x < NW * ROUTE_MAX_SHARDS) (&wc[0][0])[threadIdx.x] = 0;
    __syncthreads();
    u32 i = blockIdx.x * TILE_THREADS + threadIdx.x;
    bool valid = i < n;
    u32 own = valid ? owner_of(req[i].key_hash, n_shards) : 0;
    u32 peers = __match_any_sync(0xffffffffu, valid ? own : (0x80000000u | lane));
    u32 rank = __popc(peers & ((1u << lane) - 1));
    if (valid && rank == 0) wc[w][own] = __popc(peers);
    __syncthreads();
    if (threadIdx.x < n_shards) {
        u32 acc = 0;
        for (int x = 0; x < NW; x++) { u32 v = wc[x][threadIdx.x]; wc[x][threadIdx.x] = acc; acc += v; }
    }
    __syncthreads();
    if (valid) {
        u32 pos = tile_offsets[own * num_tiles + blockIdx.x] + wc[w][own] + rank;
        const ulonglong2 *s = reinterpret_cast<const ulonglong2 *>(req + i);
        ulonglong2 *d = reinterpret_cast<ulonglong2 *>(out + pos);
        d[0] = s[0]; d[1] = s[1]; d[2] = s[2];
        src_index[pos] = i;
    }
}

__global__ void __launch_bounds__(TILE_THREADS)
route_unpermute_kernel(const gcra_result *__restrict__ routed, const u32 *__restrict__ src_index, u32 n,
                       gcra_result *__restrict__ out) {
    u32 i = blockIdx.x * TILE_THREADS + threadIdx.x;
    if (i < n) {
        const ulonglong2 *s = reinterpret_cast<const ulonglong2 *>(routed + i);
        ulonglong2 *d = reinterpret_cast<ulonglong2 *>(out + src_index[i]);
        d[0] = s[0]; d[1] = s[1];
    }
}


// ---------------------------------------------------------------------------------------------
// metrics bridge: denied requests per key, from the kernels' own outputs
// ---------------------------------------------------------------------------------------------
// The reference counts denials per key string in a HashMap and keeps the top N (throttlecrab-server/src/
// metrics.rs:24-64,162-173).  Here a pass over a finished batch (request rows + result rows) counts the denied rows
// per key hash: every 256-row tile aggregates in a shared-memory hash set, then adds each distinct key's count to an
// open-addressed table in HBM -- a key already in the table costs a load and a posted add, only a new key a CAS.
// A full table drops new keys (counted); gcra_top_denied prunes it to the top entries like the reference's cleanup.
struct DeniedTable {
    u64 *keys;      // 0 = empty
    u64 *counts;
    u32 mask;       // capacity - 1
    u64 *dropped;
};
constexpr u32 DENIED_HASH = 512;

template <bool COMPACT>
__global__ void __launch_bounds__(TILE_THREADS)
denied_count_kernel(const unsigned char *__restrict__ req, const gcra_result *__restrict__ res, u32 n, DeniedTable t) {
    constexpr u32 RSZ = COMPACT ? sizeof(gcra_request16) : sizeof(gcra_request);
    __shared__ u64 hkey[DENIED_HASH];
    __shared__ u32 hcnt[DENIED_HASH];
    for (u32 i = threadIdx.x; i < DENIED_HASH; i += TILE_THREADS) { hkey[i] = 0; hcnt[i] = 0; }
    __syncthreads();
    const u32 i = blockIdx.x * TILE_THREADS + threadIdx.x;
    if (i < n) {
        const longlong2 tail = reinterpret_cast<const longlong2 *>(res + i)[1];      // retry_after, status | allowed << 32
        const bool denied = (u32)tail.y == GCRA_OK && ((tail.y >> 32) & 0xff) == 0;
        if (denied) {
            u64 k = *reinterpret_cast<const u64 *>(req + (size_t)i * RSZ);
            if (k == 0) k = 1;                                                          // 0 marks an empty entry
            u32 h = (u32)(mix64(k) >> 55);                                              // 9 bits
            for (;;) {
                const u64 old = atomicCAS(&hkey[h], 0ULL, k);
                if (old == 0 || old == k) { atomicAdd(&hcnt[h], 1u); break; }
                h = (h + 1) & (DENIED_HASH - 1);
            }
        }
    }
    __syncthreads();
    for (u32 e = threadIdx.x; e < DENIED_HASH; e += TILE_THREADS) {
        const u64 k = hkey[e];
        if (k == 0) continue;
        u32 h = (u32)(mix64(k ^ 0x9E3779B97F4A7C15ULL)) & t.mask;
        bool done = false;
        for (u32 probe = 0; probe < 64 && !done; probe++) {
            u64 cur = t.keys[h];                                    // (a stale L1 line shows "empty": then the CAS decides)
            if (cur == 0) { const u64 old = atomicCAS(&t.keys[h], 0ULL, k); cur = old == 0 ? k : old; }
            if (cur == k) { atomicAdd(&t.counts[h], (u64)hcnt[e]); done = true; }
            else h = (h + 1) & t.mask;
        }
        if (!done) atomicAdd(t.dropped, (u64)hcnt[e]);
    }
}

}  // namespace gcra
