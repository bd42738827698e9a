// gcra_b200.cu -- host side of the engine and the C ABI declared in include/gcra_b200.h.
//
// Host responsibilities: table allocation/growth (HashMap::with_capacity / growth), the sweep
// policies of the three reference stores (adaptive_cleanup.rs:138-211, periodic.rs:128-142,
// probabilistic.rs:110-125) driving the sweep kernel, kernel sequencing on CUDA streams, and the
// pinned host ring.  All decisions are made by the kernels in gcra_kernels.cuh; there is no CPU
// decision path.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <dlfcn.h>
#include <cstring>
#include <string>
#include <vector>

#include "gcra_kernels.cuh"
#include "gcra_index_path.cuh"
#include "gcra_p2p.cuh"

using namespace gcra;

#define CK(call)                                                                         \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess) {                                                         \
            h->err = std::string(#call) + ": " + cudaGetErrorString(e_);                 \
            return GCRA_INTERNAL;                                                        \
        }                                                                                \
    } while (0)

#define RC(call)                                  \
    do {                                          \
        int rc_ = (call);                         \
        if (rc_ != GCRA_OK) return rc_;           \
    } while (0)

namespace {
const __int128 NS_PER_S = 1000000000;

struct RingSlot {
    void *h_req = nullptr;
    gcra_result *h_res = nullptr;
    void *d_req = nullptr;
    gcra_result *d_res = nullptr;
    cudaEvent_t ev_in = nullptr, ev_comp = nullptr, ev_done = nullptr;
    bool in_flight = false;
};
}  // namespace

// ---- NCCL, resolved at run time (dlopen) so that single-GPU users do not need it ---------------------
// Minimal declarations of the public NCCL API used here (nccl.h: ncclUniqueId is 128 opaque bytes,
// ncclUint8 = 1, ncclUint32 = 3).
namespace nccl_rt {
struct UniqueId { char internal[128]; };
typedef void *Comm;
typedef int (*GetUniqueId_t)(UniqueId *);
typedef int (*CommInitRank_t)(Comm *, int, UniqueId, int);
typedef int (*CommDestroy_t)(Comm);
typedef int (*Group_t)();
typedef int (*Send_t)(const void *, size_t, int, int, Comm, cudaStream_t);
typedef int (*Recv_t)(void *, size_t, int, int, Comm, cudaStream_t);
typedef const char *(*ErrStr_t)(int);
struct Api {
    void *lib = nullptr;
    GetUniqueId_t GetUniqueId = nullptr;
    CommInitRank_t CommInitRank = nullptr;
    CommDestroy_t CommDestroy = nullptr;
    Group_t GroupStart = nullptr, GroupEnd = nullptr;
    Send_t Send = nullptr;
    Recv_t Recv = nullptr;
    ErrStr_t GetErrorString = nullptr;
};
static Api g_api;
static bool load() {
    if (g_api.lib) return true;
    void *l = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!l) l = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!l) return false;
    Api a;
    a.lib = l;
    a.GetUniqueId = (GetUniqueId_t)dlsym(l, "ncclGetUniqueId");
    a.CommInitRank = (CommInitRank_t)dlsym(l, "ncclCommInitRank");
    a.CommDestroy = (CommDestroy_t)dlsym(l, "ncclCommDestroy");
    a.GroupStart = (Group_t)dlsym(l, "ncclGroupStart");
    a.GroupEnd = (Group_t)dlsym(l, "ncclGroupEnd");
    a.Send = (Send_t)dlsym(l, "ncclSend");
    a.Recv = (Recv_t)dlsym(l, "ncclRecv");
    a.GetErrorString = (ErrStr_t)dlsym(l, "ncclGetErrorString");
    if (!a.GetUniqueId || !a.CommInitRank || !a.CommDestroy || !a.GroupStart || !a.GroupEnd || !a.Send || !a.Recv) return false;
    g_api = a;
    return true;
}
const int kUint8 = 1, kUint32 = 3;
}  // namespace nccl_rt

// one tick in flight through the sharded pipeline
struct ShardSlot {
    gcra_request *routed = nullptr, *recv_req = nullptr;
    gcra_result *recv_res = nullptr, *back_res = nullptr;
    u32 *src_index = nullptr;
    u32 *counts_dev = nullptr;     // [2*W]: rows I send to every peer, rows every peer sends me
    u32 *counts_host = nullptr;    // pinned copy
    cudaEvent_t ev_ready = nullptr, ev_counts = nullptr, ev_routed = nullptr, ev_done = nullptr;
    bool used = false;
    uint32_t n = 0, n_recv = 0;
    gcra_result *d_res_user = nullptr;
    std::vector<size_t> send, recv, send_off, recv_off;
};

struct Shard {
    static const int DEPTH = 4;
    int rank = 0, world = 0;
    uint32_t max_rows = 0;
    nccl_rt::Comm comm_counts = nullptr, comm_req = nullptr, comm_res = nullptr;
    cudaStream_t s_part = nullptr, s_route = nullptr, s_return = nullptr;   // partition+counts | request all-to-all | way back
    ShardSlot slots[DEPTH];
    uint32_t next = 0;
    int pending = -1;              // slot whose decide + return stages have not been issued yet
    cudaEvent_t ev_tmp = nullptr;
};

// ---- multi-GPU over NVLink peer memory (gcra_p2p.cuh) ------------------------------------------------------
struct P2PSlot {
    u32 *res_loc = nullptr;            // [cap] where the result of my row i arrives in my outbox
    u32 *counts_dev = nullptr;         // [world] rows I routed to every owner in this tick
    SegDesc *segs_dev = nullptr;       // [world] segment r of this inbox slot: sender r's rows, sender r's outbox
    cudaEvent_t ev_ready = nullptr, ev_wait = nullptr, ev_done = nullptr;
    bool used = false;
    uint32_t n = 0;
};

struct P2P {
    int rank = 0, world = 0;
    uint32_t cap = 0, cap_shift = 0;
    void *window = nullptr;
    size_t window_bytes = 0, inbox_off = 0, outbox_off = 0;
    void *peer_base[P2P_MAX_WORLD] = {};
    bool opened[P2P_MAX_WORLD] = {};
    bool connected = false, routed_pending = false;
    P2PPeers *peers_dev = nullptr;
    u32 *tile_counts = nullptr;
    cudaStream_t s_part = nullptr, s_wait = nullptr, s_sig = nullptr, s_return = nullptr;
    P2PSlot slots[P2P_DEPTH];
    uint64_t next_tick = 0;
    bool timed = false, timed_valid = false;
    cudaEvent_t ev_t[6] = {};
};

// per-batch scratch; several sets so that the front halves of the next batches can overlap the back half of
// the current one
struct Scratch {
    Req *drec = nullptr;
    u64 *keys_a = nullptr, *keys_b = nullptr;
    // one-sweep sort: look-back words [tiles][SORT_MAX_DIGITS]; digit totals, double-buffered by sort
    // [2][SORT_MAX_PASSES][SORT_MAX_DIGITS], then the tile ticket counter
    u64 *sort_status = nullptr;
    u32 *sort_tot = nullptr, *sort_ticket = nullptr;
    uint32_t sort_seq = 0, sort_tickets = 0, sort_parity = 0;   // last pass sequence number, tickets taken, totals half
    LongRun *long_runs = nullptr, *giant_runs = nullptr;
    u32 *long_count = nullptr;
    cudaEvent_t ev_front = nullptr, ev_mid = nullptr, ev_back = nullptr, ev_fork = nullptr, ev_join = nullptr, ev_join2 = nullptr;
    bool back_recorded = false;
    // index-order pipeline (gcra_index_path.cuh)
    u32 *slot_arr = nullptr;            // [rows] slot of every row (null slot: the row failed validation)
    unsigned char *flags = nullptr;     // [rows] pass-B verdict of rows on shared slots
    u32 *bitmap = nullptr;              // [bm_words] 16-bit occurrence counters of the batch, hashed by slot
    u32 *pend = nullptr;                // [pend_words] 1 bit per entry: the PREVIOUS batch's tail owns a slot of the entry
    u64 *ctrl_block = nullptr;          // word 0: {tile ticket, residue count}; then one status word per tile
    uint32_t rows_alloc = 0;
    u32 *h_nres = nullptr;              // pinned: residue size of the set's latest index-order batch (valid after ev_mid)
    bool mid_recorded = false, nres_counted = true;
    uint32_t nres_rows = 0;             // rows of that batch
};

struct gcra_engine {
    int device = 0;
    cudaStream_t stream = nullptr, in_stream = nullptr, out_stream = nullptr, aux_stream = nullptr, aux2_stream = nullptr;
    Table tab{};
    uint32_t total_lines = 0;
    uint64_t capacity = 0;
    bool tight = false;              // GCRA_FLAG_TIGHT_TABLE: tests only, exercises stash + growth
    // scratch for one batch
    uint32_t max_batch = 0;
#ifndef GCRA_PIPE_SETS
#define GCRA_PIPE_SETS 4
#endif
    static const int N_SCR = GCRA_PIPE_SETS;
    Scratch scr[N_SCR];
    uint32_t scr_next = 0;
    // pipelined submission: three stages on three streams (front: probe | mid: decide + resolve | tail: the
    // sorted residue); the sort pipeline uses front (ingest + sort) and mid (decide)
    cudaStream_t front_stream[N_SCR] = {}, back_stream = nullptr, tail_stream = nullptr;
    int pend_set = -1;               // scratch set whose bitmap holds the PEND bits of the batch submitted last (-1: none)
    cudaEvent_t ev_ready = nullptr;
    void *d_req = nullptr;
    gcra_result *d_res = nullptr;
    u32 *route_counts = nullptr;
    PolicyDerived *d_pol = nullptr;
    uint32_t npol = 0;
    StoreOpResult *d_op = nullptr, *h_op = nullptr;
    u64 *h_counters = nullptr;       // pinned snapshot, refreshed after every batch
    cudaEvent_t ev_counters = nullptr;
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t evd[8] = {};         // index-order pipeline, serial timed batch: after each kernel group
    bool evd_valid = false;
    cudaEvent_t ev_sweep[2] = {nullptr, nullptr};
    bool sweep_timed = false;
    bool ev_valid = false;
    uint64_t launches = 0;
    uint64_t occupied_ub = 0;        // host-side upper bound of claimed slots
    // asynchronous occupancy snapshots: counters copied after every batch, read when their event is done
    static const int N_SNAP = 8;
    u64 *h_snap = nullptr;           // pinned [N_SNAP][C_COUNT]
    cudaEvent_t ev_snap[N_SNAP] = {};
    uint64_t snap_rows_after[N_SNAP] = {};   // rows launched up to and including the snapshot's batch
    bool snap_used[N_SNAP] = {};
    uint32_t snap_next = 0;
    uint64_t rows_launched = 0;
    // store policy (mirrors the reference stores' fields)
    int kind = GCRA_STORE_ADAPTIVE;
    __int128 next_cleanup = 0, cleanup_interval = 0;
    __int128 min_interval = 0, max_interval = 0, cur_interval = 0;
    uint64_t expired_count = 0, ops_since_cleanup = 0, max_ops = 0;
    uint64_t last_removed = 0, last_total = 0;
    uint64_t ops_count = 0, cleanup_modulo = 0;
    uint64_t seen_allowed = 0, seen_expired_hits = 0;
    uint64_t n_sweeps = 0, n_grows = 0, n_purges = 0;
    Shard *shard = nullptr;          // multi-GPU: native NCCL pipeline (gcra_shard_*)
    P2P *p2p = nullptr;              // multi-GPU: NVLink peer-memory pipeline (gcra_p2p_*)
    // index-order pipeline
    uint32_t epoch = 0;              // batch epoch of the slot marks (never 0)
    uint32_t bm_mask = 0;            // bitmap entries - 1
    size_t bm_words = 0, pend_words = 0;
    uint32_t index_min = 0;          // batches of at least this many rows take the index-order pipeline (0: never)
    int prefetch_state = 0;
    uint32_t max_tiles = 0;
    uint32_t grid_probe[2] = {592, 592}, grid_decide[2] = {444, 444};   // resident CTAs of the persistent kernels [compact]
    uint32_t dbg = 0;                // timing experiments only (gcra_debug_set): skips parts of pass B
    uint32_t last_nres = 0, last_nres_rows = 0;   // newest residue size that has reached the host (and its batch's rows)
    bool adaptive = true;            // choose the pipeline from the residue feedback (off when a test / env forces one)
    uint64_t n_path_switches = 0;
    uint32_t sort_hold = 0;          // > 0: the residue was large, this many more batches take the sort pipeline
    uint32_t since_drain = 0;        // index-order batches submitted since stage 2 last waited for every tail
    uint64_t n_drains = 0, n_index_batches = 0, residue_seen = 0, residue_batches_seen = 0;
    // ring
    std::vector<RingSlot> ring;
    uint32_t ring_cap = 0;
    bool ring_compact = false;
    // denied requests per key (gcra_track_denied): device table, updated by a pass over every finished batch
    DeniedTable denied{};
    uint32_t denied_max = 0, denied_cap = 0;
    uint64_t hash_seed[2] = {0, 0};  // SipHash key of the string-keyed entry points ((0,0): the unkeyed gcra_hash_key)
    std::string err;
};

static int alloc_index_scratch(gcra_engine *h, Scratch &sc, uint32_t rows);

static uint32_t ceil_log2(uint64_t x) {
    uint32_t b = 0;
    while ((1ULL << b) < x) b++;
    return b;
}

static void table_geometry(uint64_t capacity, bool tight, uint32_t &total_lines, uint32_t &nb_main, uint32_t &stash_slots) {
    // first-fit two-choice buckets of 4 stay below ~0.4 % stash traffic up to load 0.5
    uint64_t slots = 1ULL << ceil_log2(std::max<uint64_t>(tight ? capacity : capacity * 2, tight ? 64 : 256));
    total_lines = (uint32_t)(slots / 4);
    uint32_t ns = std::max<uint32_t>(tight ? total_lines / 4 : total_lines / 64, 8);
    nb_main = total_lines - ns;
    stash_slots = (ns - 1) * 4;   // the last line is reserved (null slot)
}

static int alloc_table(gcra_engine *h, uint64_t capacity, Table &t, uint32_t &total_lines, u64 *counters) {
    uint32_t nb, ss;
    table_geometry(capacity, h->tight, total_lines, nb, ss);
    const size_t slots = (size_t)total_lines * 4;
    CK(cudaMalloc(&t.keys, slots * sizeof(u64)));
    CK(cudaMalloc(&t.state, slots * sizeof(TatOff)));
    CK(cudaMalloc(&t.ei, slots * sizeof(i64)));
    CK(cudaMalloc(&t.mark, slots * sizeof(u64)));
    CK(cudaMemsetAsync(t.mark, 0xff, slots * sizeof(u64), h->stream));   // no batch epoch matches
    t.nb_main = nb;
    t.stash_slots = ss;
    t.null_slot = total_lines * 4 - 1;
    t.slot_bits = ceil_log2((uint64_t)total_lines * 4);
    t.counters = counters;
    uint32_t grid = (uint32_t)std::min<size_t>((slots + TILE_THREADS - 1) / TILE_THREADS, 148 * 16);
    clear_slots_kernel<<<grid, TILE_THREADS, 0, h->stream>>>(t, 0, slots);
    h->launches++;
    CK(cudaGetLastError());
    return GCRA_OK;
}

static uint64_t load_limit(const gcra_engine *h) {
    uint64_t main_slots = (uint64_t)h->tab.nb_main * 4;
    return h->tight ? main_slots * 13 / 16 : main_slots / 2;
}

static uint64_t load_limit_for(uint64_t capacity, bool tight) {
    uint32_t tl, nb, ss;
    table_geometry(capacity, tight, tl, nb, ss);
    uint64_t main_slots = (uint64_t)nb * 4;
    return tight ? main_slots * 13 / 16 : main_slots / 2;
}

static int refresh_counters(gcra_engine *h, bool wait) {
    CK(cudaMemcpyAsync(h->h_counters, h->tab.counters, C_COUNT * sizeof(u64), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaEventRecord(h->ev_counters, h->stream));
    if (wait) CK(cudaEventSynchronize(h->ev_counters));
    return GCRA_OK;
}

static int do_sweep(gcra_engine *h, int64_t now_ns, uint64_t *removed) {
    CK(cudaSetDevice(h->device));
    CK(cudaDeviceSynchronize());   // the sweep is exclusive: batches may be in flight on caller streams
    RC(refresh_counters(h, true));
    uint64_t before = h->h_counters[C_SWEPT];
    uint32_t grid = (uint32_t)std::min<uint64_t>(((uint64_t)h->total_lines * 2 + TILE_THREADS * SWEEP_UNROLL - 1) / (TILE_THREADS * SWEEP_UNROLL), 148 * 16);
    CK(cudaEventRecord(h->ev_sweep[0], h->stream));
    static const int sweep_mode = getenv("GCRA_SWEEP_MODE") ? atoi(getenv("GCRA_SWEEP_MODE")) : 0;
    sweep_kernel<<<grid, TILE_THREADS, 0, h->stream>>>(h->tab, (u64)h->total_lines * 4, now_ns, sweep_mode);
    CK(cudaEventRecord(h->ev_sweep[1], h->stream));
    h->sweep_timed = true;
    h->launches++;
    CK(cudaGetLastError());
    RC(refresh_counters(h, true));
    h->occupied_ub = h->h_counters[C_OCCUPIED];
    for (int i = 0; i < gcra_engine::N_SNAP; i++) h->snap_used[i] = false;
    h->n_sweeps++;
    if (removed) *removed = h->h_counters[C_SWEPT] - before;
    return GCRA_OK;
}

// reclaim the slots of keys without an entry (exclusive); returns with fresh counters
static int purge(gcra_engine *h) {
    CK(cudaDeviceSynchronize());
    const uint64_t slots = (uint64_t)h->total_lines * 4;
    uint32_t grid = (uint32_t)std::min<uint64_t>((slots + TILE_THREADS - 1) / TILE_THREADS, 148 * 16);
    purge_kernel<<<grid, TILE_THREADS, 0, h->stream>>>(h->tab, slots);
    h->launches++;
    CK(cudaGetLastError());
    RC(refresh_counters(h, true));
    if (h->h_counters[C_STASH] == 0) {
        // no key lives in the stash any more: drop its tombstones
        uint64_t first = (uint64_t)h->tab.nb_main * 4, cnt = slots - first;
        clear_slots_kernel<<<(uint32_t)((cnt + TILE_THREADS - 1) / TILE_THREADS), TILE_THREADS, 0, h->stream>>>(
            h->tab, first, cnt);
        h->launches++;
        CK(cudaGetLastError());
    }
    h->occupied_ub = h->h_counters[C_OCCUPIED];
    for (int i = 0; i < gcra_engine::N_SNAP; i++) h->snap_used[i] = false;
    h->n_purges++;
    return GCRA_OK;
}

// HashMap growth: rebuild into a table twice the size
static int grow(gcra_engine *h, uint64_t need) {
    CK(cudaStreamSynchronize(h->stream));
    uint64_t newcap = std::max<uint64_t>(h->capacity * 2, 256);
    while (load_limit_for(newcap, h->tight) < need) newcap *= 2;
    Table nt{};
    uint32_t nl = 0;
    u64 *ncounters = nullptr;
    CK(cudaMalloc(&ncounters, C_COUNT * sizeof(u64)));
    CK(cudaMemsetAsync(ncounters, 0, C_COUNT * sizeof(u64), h->stream));
    int rc = alloc_table(h, newcap, nt, nl, ncounters);
    if (rc) return rc;
    uint32_t grid = std::min<uint32_t>((h->total_lines + TILE_THREADS - 1) / TILE_THREADS, 148 * 8);
    rehash_kernel<<<grid, TILE_THREADS, 0, h->stream>>>(h->tab, (u64)h->total_lines * 4, nt);
    h->launches++;
    CK(cudaGetLastError());
    // carry the running totals over
    RC(refresh_counters(h, true));
    u64 keep[C_COUNT];
    memcpy(keep, h->h_counters, sizeof(keep));
    u64 fresh[C_COUNT];
    CK(cudaMemcpyAsync(fresh, ncounters, sizeof(fresh), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (fresh[C_INSERT_FAIL]) { h->err = "table growth lost entries"; return GCRA_INTERNAL; }
    keep[C_OCCUPIED] = fresh[C_OCCUPIED];
    keep[C_REAL] = fresh[C_REAL];
    keep[C_STASH] = fresh[C_STASH];
    CK(cudaMemcpyAsync(ncounters, keep, sizeof(keep), cudaMemcpyHostToDevice, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    cudaFree(h->tab.keys); cudaFree(h->tab.state); cudaFree(h->tab.ei); cudaFree(h->tab.mark);
    cudaFree(h->tab.counters);
    h->tab = nt;
    h->total_lines = nl;
    h->capacity = newcap;
    h->occupied_ub = keep[C_OCCUPIED];
    for (int i = 0; i < gcra_engine::N_SNAP; i++) h->snap_used[i] = false;
    h->n_grows++;
    return GCRA_OK;
}

static int ensure_room(gcra_engine *h, uint64_t n) {
    if (h->occupied_ub + n <= load_limit(h)) { h->occupied_ub += n; return GCRA_OK; }
    // the bound is stale (it assumes every request claimed a slot): tighten it from the newest
    // counter snapshot that has already arrived, without stalling the stream
    for (int back = 1; back <= gcra_engine::N_SNAP; back++) {
        int k = (int)((h->snap_next + gcra_engine::N_SNAP - back) % gcra_engine::N_SNAP);
        if (!h->snap_used[k]) break;
        if (cudaEventQuery(h->ev_snap[k]) != cudaSuccess) continue;
        uint64_t ub = h->h_snap[(size_t)k * C_COUNT + C_OCCUPIED] + (h->rows_launched - h->snap_rows_after[k]);
        if (ub < h->occupied_ub) h->occupied_ub = ub;
        break;
    }
    if (h->occupied_ub + n <= load_limit(h)) { h->occupied_ub += n; return GCRA_OK; }
    int rc = refresh_counters(h, true);
    if (rc) return rc;
    CK(cudaDeviceSynchronize());   // batches may be in flight on caller streams
    rc = refresh_counters(h, true);
    if (rc) return rc;
    h->occupied_ub = h->h_counters[C_OCCUPIED];
    if (h->occupied_ub + n > load_limit(h) && h->h_counters[C_OCCUPIED] > h->h_counters[C_REAL]) {
        // crowded: first give back the slots of keys that hold no entry (swept or only ever denied)
        rc = purge(h);
        if (rc) return rc;
    }
    if (h->occupied_ub + n > load_limit(h)) {
        rc = grow(h, (h->occupied_ub + n));
        if (rc) return rc;
    }
    h->occupied_ub += n;
    return GCRA_OK;
}

static int snapshot_async(gcra_engine *h, uint64_t n, cudaStream_t st) {
    h->rows_launched += n;
    int k = (int)h->snap_next;
    h->snap_next = (h->snap_next + 1) % gcra_engine::N_SNAP;
    CK(cudaMemcpyAsync(h->h_snap + (size_t)k * C_COUNT, h->tab.counters, C_COUNT * sizeof(u64), cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(h->ev_snap[k], st));
    h->snap_rows_after[k] = h->rows_launched;
    h->snap_used[k] = true;
    return GCRA_OK;
}

// ---- sweep policies ------------------------------------------------------------------------
static bool adaptive_should_clean(const gcra_engine *h, __int128 now, uint64_t len) {   // adaptive_cleanup.rs:138-171
    if (now >= h->next_cleanup) return true;
    if (h->ops_since_cleanup >= h->max_ops) return true;
    if (h->expired_count > 50) {
        double ratio = (double)h->expired_count / (double)(len ? len : 1);
        double threshold = (h->last_removed > h->last_total / 4) ? 0.2 / 2.0 : 0.2 * 1.25;
        if (ratio > threshold) return true;
    }
    if (len > load_limit(h) * 3 / 4) return true;
    return false;
}

// called at batch boundaries with the counters of the batches finished so far
static int apply_policy(gcra_engine *h, int64_t now_ns) {
    if (h->kind == GCRA_STORE_MANUAL) return GCRA_OK;
    uint64_t allowed = h->h_counters[C_ALLOWED], hits = h->h_counters[C_EXPIRED_HITS];
    uint64_t d_ops = allowed - h->seen_allowed, d_hits = hits - h->seen_expired_hits;
    h->seen_allowed = allowed;
    h->seen_expired_hits = hits;
    __int128 now = now_ns;
    uint64_t removed = 0;
    if (h->kind == GCRA_STORE_PERIODIC) {                       // periodic.rs:128-142
        if (now >= h->next_cleanup) {
            int rc = do_sweep(h, now_ns, &removed);
            if (rc) return rc;
            h->expired_count = removed;
            h->next_cleanup = now + h->cleanup_interval;
        }
    } else if (h->kind == GCRA_STORE_PROBABILISTIC) {           // probabilistic.rs:110-125
        // sweep when some op count k in (ops, ops + d_ops] has k * 2654435761 % modulo == 0
        const uint64_t c = 2654435761ULL, m = h->cleanup_modulo;
        uint64_t a = h->ops_count + 1, b = h->ops_count + d_ops;
        bool hit = false;
        if (d_ops) {
            if (b < (~0ULL) / c) {
                uint64_t g = m, x = c % m;
                while (x) { uint64_t tmp = g % x; g = x; x = tmp; }
                uint64_t step = m / g;
                hit = (b / step) > ((a - 1) / step);
            } else {
                for (uint64_t k = a; k <= b && !hit; k++) hit = ((k * c) % m) == 0;
            }
        }
        h->ops_count = b;
        if (hit) { int rc = do_sweep(h, now_ns, &removed); if (rc) return rc; }
    } else {                                                    // adaptive_cleanup.rs:205-211
        h->ops_since_cleanup += d_ops;
        h->expired_count += d_hits;
        uint64_t len = h->h_counters[C_REAL];
        if (adaptive_should_clean(h, now, len)) {               // cleanup(): :173-203
            int rc = do_sweep(h, now_ns, &removed);
            if (rc) return rc;
            if (removed == 0 && h->expired_count == 0) {
                __int128 d = h->cur_interval * 2;
                h->cur_interval = d < h->max_interval ? d : h->max_interval;
            } else if ((double)removed > (double)len * 0.5) {
                __int128 d = h->cur_interval / 2;
                h->cur_interval = d > h->min_interval ? d : h->min_interval;
            }
            h->last_removed = removed;
            h->last_total = len;
            h->next_cleanup = now + h->cur_interval;
            h->expired_count = 0;
            h->ops_since_cleanup = 0;
        }
    }
    return GCRA_OK;
}

// the cluster kernel: cluster dimension given at launch (cudaLaunchKernelEx)
template <bool BY_ROW>
static int launch_giant(gcra_engine *h, Scratch &sc, const u64 *src, const OutMap &om, cudaStream_t st) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((128 / CLUSTER_CTAS) * CLUSTER_CTAS);
    cfg.blockDim = dim3(LONG_THREADS);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CLUSTER_CTAS;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (CLUSTER_CTAS > 8) {
        static bool once = false;
        if (!once) { cudaFuncSetAttribute(decide_runs_kernel<CLUSTER_CTAS, BY_ROW>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1); once = true; }
    }
    CK(cudaLaunchKernelEx(&cfg, decide_runs_kernel<CLUSTER_CTAS, BY_ROW>, h->tab, (const u64 *)src, (const Req *)sc.drec, om,
                          (const LongRun *)sc.giant_runs, (const u32 *)(sc.long_count + 1)));
    return GCRA_OK;
}

static BatchView single_view(const void *d_req, gcra_result *d_res, uint32_t n) {
    BatchView v{};
    v.req0 = (const unsigned char *)d_req;
    v.res0 = d_res;
    v.n = n;
    v.nseg = 1;
    v.cap_shift = 31;
    return v;
}

static uint32_t sort_tiles_max(const gcra_engine *h) { return (h->max_batch + SORT_TILE - 1) / SORT_TILE; }

// stable LSD radix sort of `n` (host count) or `*n_dev` (device count, at most n_max) keys on the slot bits: one
// histogram launch for every pass, then one launch per pass; returns the buffer that holds the sorted keys
static int enqueue_sort(gcra_engine *h, Scratch &sc, uint32_t n_max, const u32 *n_dev, cudaStream_t st, u64 **sorted_out) {
    const uint32_t bits = h->tab.slot_bits;
    const uint32_t passes = (bits + SORT_MAX_BITS - 1) / SORT_MAX_BITS;
    const uint32_t tiles = (n_max + SORT_TILE - 1) / SORT_TILE;
    if (passes > SORT_MAX_PASSES) { h->err = "slot bits beyond the sort's passes"; return GCRA_INTERNAL; }
    u32 *tot = sc.sort_tot + sc.sort_parity * SORT_MAX_PASSES * SORT_MAX_DIGITS;
    u32 *clear = sc.sort_tot + (sc.sort_parity ^ 1) * SORT_MAX_PASSES * SORT_MAX_DIGITS;
    sc.sort_parity ^= 1;
    const uint32_t hgrid = std::min<uint32_t>((n_max + SORT_HIST_KEYS - 1) / SORT_HIST_KEYS, 4 * 148);
    sort_digits_hist_kernel<<<hgrid, TILE_THREADS, 0, st>>>(sc.keys_a, n_max, n_dev, bits, passes, tot, clear);
    u64 *src = sc.keys_a, *dst = sc.keys_b;
    uint32_t shift = 32;
    for (uint32_t p = 0; p < passes; p++) {
        const uint32_t pb = sort_pass_bits(bits, passes, p);
        if (sc.sort_seq + 1 >= SORT_SEQ_LIMIT) {
            // the 31-bit pass sequence number wrapped (once per 2 G passes): forget every look-back word
            CK(cudaMemsetAsync(sc.sort_status, 0, (size_t)sort_tiles_max(h) * SORT_MAX_DIGITS * sizeof(u64), st));
            sc.sort_seq = 0;
        }
        // every CTA takes exactly one ticket, also those beyond a device count
        sort_onesweep_kernel<<<tiles, TILE_THREADS, 0, st>>>(src, dst, n_max, n_dev, shift, pb, tot + p * SORT_MAX_DIGITS,
                                                             sc.sort_status, sc.sort_ticket, sc.sort_tickets, ++sc.sort_seq);
        sc.sort_tickets += tiles;
        std::swap(src, dst);
        shift += pb;
    }
    h->launches += 1 + passes;
    *sorted_out = src;
    return GCRA_OK;
}

template <bool BY_ROW>
static int enqueue_decide_sorted_t(gcra_engine *h, Scratch &sc, uint32_t n_max, const u32 *n_dev, const u64 *src,
                                   const OutMap &om, cudaStream_t st) {
    // (sort pipeline: the work-list counters were cleared at the end of the front half, off this stream)
    if (BY_ROW) CK(cudaMemsetAsync(sc.long_count, 0, 2 * sizeof(u32), st));
    const uint32_t warps = (n_max + 31) / 32;
    uint32_t grid = (warps + DECIDE_THREADS / 32 - 1) / (DECIDE_THREADS / 32);
    if (n_dev) grid = std::min<uint32_t>(grid, 4 * 148);
    decide_kernel<BY_ROW><<<grid, DECIDE_THREADS, 0, st>>>(h->tab, src, sc.drec, n_max, n_dev, om, sc.long_runs, sc.giant_runs,
                                                           sc.long_count, 0);
    h->launches++;
    if (n_max >= GIANT_RUN_MIN) {
        // the two hot-run kernels work on disjoint runs: the one-CTA-per-run kernel goes to a side
        // stream and overlaps the cluster kernel (fork/join with events)
        CK(cudaEventRecord(sc.ev_fork, st));
        CK(cudaStreamWaitEvent(h->aux_stream, sc.ev_fork, 0));
        decide_runs_kernel<1, BY_ROW><<<148, LONG_THREADS, 0, h->aux_stream>>>(h->tab, src, sc.drec, om, sc.long_runs, sc.long_count);
        CK(cudaEventRecord(sc.ev_join, h->aux_stream));
        RC(launch_giant<BY_ROW>(h, sc, src, om, st));   // hottest keys: one cluster per run
        CK(cudaStreamWaitEvent(st, sc.ev_join, 0));
        h->launches += 2;
    } else if (n_max >= LONG_RUN_MIN) {
        decide_runs_kernel<1, BY_ROW><<<148, LONG_THREADS, 0, st>>>(h->tab, src, sc.drec, om, sc.long_runs, sc.long_count);
        h->launches++;
    }
    return GCRA_OK;
}

// the warp-cooperative compare-and-update over sorted keys + the hot-run kernels
static int enqueue_decide_sorted(gcra_engine *h, Scratch &sc, uint32_t n_max, const u32 *n_dev, const u64 *src,
                                 const OutMap &om, cudaStream_t st) {
    return om.by_row ? enqueue_decide_sorted_t<true>(h, sc, n_max, n_dev, src, om, st)
                     : enqueue_decide_sorted_t<false>(h, sc, n_max, n_dev, src, om, st);
}

// per-set buffers of the index-order pipeline for batches of up to `rows` row ids
static int alloc_index_scratch(gcra_engine *h, Scratch &sc, uint32_t rows) {
    cudaFree(sc.slot_arr); cudaFree(sc.flags); cudaFree(sc.ctrl_block);
    sc.slot_arr = nullptr; sc.flags = nullptr; sc.ctrl_block = nullptr;
    const uint32_t tiles = (rows + TILE_THREADS - 1) / TILE_THREADS;
    if (tiles > h->max_tiles) h->max_tiles = tiles;
    CK(cudaMalloc(&sc.slot_arr, (size_t)rows * sizeof(u32)));
    CK(cudaMalloc(&sc.flags, (size_t)rows));
    CK(cudaMalloc(&sc.ctrl_block, ((size_t)h->max_tiles + 1) * sizeof(u64)));
    if (!sc.h_nres) { CK(cudaMallocHost(&sc.h_nres, sizeof(u32))); *sc.h_nres = 0; }
    if (!sc.bitmap) {
        CK(cudaMalloc(&sc.bitmap, h->bm_words * sizeof(u32)));
        CK(cudaMalloc(&sc.pend, h->pend_words * sizeof(u32)));
        CK(cudaMemsetAsync(sc.bitmap, 0, h->bm_words * sizeof(u32), h->stream));   // from then on cleared after every use
        CK(cudaMemsetAsync(sc.pend, 0, h->pend_words * sizeof(u32), h->stream));
    }
    sc.rows_alloc = rows;
    return GCRA_OK;
}

// metrics bridge: count this batch's denied rows per key (single-segment batches: request and result rows local)
static int enqueue_denied(gcra_engine *h, const BatchView &v, bool compact, cudaStream_t st) {
    if (!h->denied_max || v.nseg != 1 || v.n == 0) return GCRA_OK;
    const uint32_t tiles = (v.n + TILE_THREADS - 1) / TILE_THREADS;
    if (compact) denied_count_kernel<true><<<tiles, TILE_THREADS, 0, st>>>(v.req0, v.res0, v.n, h->denied);
    else denied_count_kernel<false><<<tiles, TILE_THREADS, 0, st>>>(v.req0, v.res0, v.n, h->denied);
    h->launches++;
    CK(cudaGetLastError());
    return GCRA_OK;
}

static bool use_index_path(const gcra_engine *h, uint32_t n) {
    // The batch counters are 16-bit fields that receive at most 2 per distinct slot and 256-row tile.  Slots that
    // share a hashed entry add up: k slots that occur in EVERY tile reach 2 k x tiles.  Up to 2^21 rows (8192 tiles)
    // that stays below 65536 unless four such ultra-hot keys (each > 0.4 % of the traffic) hash to one of the 2^23+
    // entries; larger batches take the sort pipeline.
    return h->index_min != 0 && n >= h->index_min && n <= (1u << 21);
}

static uint32_t view_max_rows(const BatchView &v) { return v.nseg == 1 ? v.n : (v.nseg << v.cap_shift); }

// Stage 1 of a batch.  Independent of the later stages of EARLIER batches: it only claims empty slots (a CAS on
// the keys array; it never touches the state array), which no earlier batch's decide kernels touch.
//   sort pipeline         ingest (validate, derive, probe/claim) + stable sort by slot
//   index-order pipeline  pass A (probe) + pass A' (batch bitmap)
static int enqueue_front(gcra_engine *h, Scratch &sc, const BatchView &v, bool index_path, bool compact, int64_t now_batch,
                         cudaStream_t st, bool timed, u64 **sorted_out) {
    if (timed) CK(cudaEventRecord(h->ev[0], st));
    *sorted_out = nullptr;
    if (index_path) {
        const uint32_t rows = view_max_rows(v);
        const uint32_t tiles = (rows + TILE_THREADS - 1) / TILE_THREADS;
        const uint32_t grid = std::min<uint32_t>(tiles, h->grid_probe[compact ? 1 : 0]);    // persistent, software-pipelined CTAs
        CK(cudaMemsetAsync(sc.ctrl_block, 0, ((size_t)h->max_tiles + 1) * sizeof(u64), st));
        if (timed) CK(cudaEventRecord(h->evd[0], st));
        if (compact)
            probe_kernel<true><<<grid, TILE_THREADS, 0, st>>>(h->tab, v, h->d_pol, h->npol, now_batch, sc.slot_arr, sc.bitmap,
                                                              h->bm_mask, h->prefetch_state);
        else
            probe_kernel<false><<<grid, TILE_THREADS, 0, st>>>(h->tab, v, nullptr, 0, 0, sc.slot_arr, sc.bitmap, h->bm_mask,
                                                               h->prefetch_state);
        if (timed) CK(cudaEventRecord(h->evd[1], st));
        h->launches += 1;
        if (timed) { CK(cudaEventRecord(h->ev[1], st)); CK(cudaEventRecord(h->evd[2], st)); }
        return GCRA_OK;
    }
    const uint32_t n = v.n;
    const uint32_t tiles = (n + TILE_THREADS - 1) / TILE_THREADS;
    if (compact)
        ingest_kernel<true><<<tiles, TILE_THREADS, 0, st>>>(h->tab, v.req0, h->d_pol, h->npol, now_batch, n,
                                                            sc.drec, sc.keys_a, v.res0);
    else
        ingest_kernel<false><<<tiles, TILE_THREADS, 0, st>>>(h->tab, v.req0, nullptr, 0, 0, n, sc.drec,
                                                             sc.keys_a, v.res0);
    h->launches++;
    if (timed) CK(cudaEventRecord(h->ev[1], st));
    RC(enqueue_sort(h, sc, n, nullptr, st, sorted_out));
    if (timed) CK(cudaEventRecord(h->ev[2], st));
    CK(cudaMemsetAsync(sc.long_count, 0, 2 * sizeof(u32), st));   // hot-run work lists of this batch's decide kernels
    return GCRA_OK;
}

// Stage 2 of an index-order batch: pass B (decide in batch order) + pass C (resolve).  Batches' stages 2 run
// strictly in submission order.  `next` is the scratch set the NEXT batch will use: pass C leaves the PEND bits
// of this batch's residue keys in its bitmap.  This set's own bitmap is cleared for its next use afterwards.
static int enqueue_mid_index(gcra_engine *h, Scratch &sc, Scratch &next, const BatchView &v, bool compact, int64_t now_batch,
                             bool honour_pend, cudaStream_t st, bool timed) {
    const u32 hp = honour_pend ? 1u : 0u;
    if (++h->epoch == 0) {
        // the 32-bit batch epoch wrapped: forget every mark (once per 4 G batches)
        CK(cudaMemsetAsync(h->tab.mark, 0xff, (size_t)h->total_lines * 4 * sizeof(u64), st));
        h->epoch = 1;
    }
    const uint32_t rows = view_max_rows(v);
    const uint32_t grid = std::min<uint32_t>((rows + TILE_THREADS - 1) / TILE_THREADS, h->grid_decide[compact ? 1 : 0]);   // persistent CTAs
    const uint32_t rgrid = std::min<uint32_t>((rows + RES_TILE - 1) / RES_TILE + v.nseg, 6 * 148);
    u32 *ctrl = reinterpret_cast<u32 *>(sc.ctrl_block);
    u64 *status = sc.ctrl_block + 1;
    if (compact) {
        decide_index_kernel<true><<<grid, TILE_THREADS, 0, st>>>(h->tab, v, h->d_pol, h->npol, now_batch, sc.slot_arr,
                                                                 sc.bitmap, sc.pend, h->bm_mask, sc.flags, h->epoch, hp, h->dbg);
        if (timed) CK(cudaEventRecord(h->evd[3], st));
        resolve_kernel<true><<<rgrid, TILE_THREADS, 0, st>>>(h->tab, v, h->d_pol, h->npol, now_batch, sc.slot_arr,
                                                             h->bm_mask, sc.flags, h->epoch, ctrl, status, sc.keys_a,
                                                             next.pend, sc.h_nres, h->max_batch);
    } else {
        decide_index_kernel<false><<<grid, TILE_THREADS, 0, st>>>(h->tab, v, nullptr, 0, 0, sc.slot_arr, sc.bitmap, sc.pend,
                                                                  h->bm_mask, sc.flags, h->epoch, hp, h->dbg);
        if (timed) CK(cudaEventRecord(h->evd[3], st));
        resolve_kernel<false><<<rgrid, TILE_THREADS, 0, st>>>(h->tab, v, nullptr, 0, 0, sc.slot_arr, h->bm_mask,
                                                              sc.flags, h->epoch, ctrl, status, sc.keys_a,
                                                              next.pend, sc.h_nres, h->max_batch);
    }
    h->launches += 2;
    h->n_index_batches++;
    if (timed) CK(cudaEventRecord(h->evd[4], st));
    // (pass C wrote the residue size of this batch to sc.h_nres, mapped pinned host memory: read, once ev_mid has
    // completed, when later batches are submitted)
    sc.nres_rows = std::min<uint32_t>(rows, h->max_batch);
    sc.nres_counted = false;
    if (timed) CK(cudaEventRecord(h->ev[2], st));
    CK(cudaGetLastError());
    return GCRA_OK;
}

// Stage 3 of an index-order batch: the residue (requests behind the first state change of their key, and
// requests deferred because the previous batch's tail still owned their key) through the sort pipeline; its
// size only exists on the device.  Tails run strictly in submission order.
static int enqueue_tail_index(gcra_engine *h, Scratch &sc, const BatchView &v, bool compact, int64_t now_batch, cudaStream_t st,
                              bool timed) {
    const u32 *n_res = reinterpret_cast<const u32 *>(sc.ctrl_block) + RC_NRES;
    const uint32_t n_max = std::min<uint32_t>(view_max_rows(v), h->max_batch);
    u64 *rs = nullptr;
    // this set's bitmap has been read for the last time (pass C): cleared here, off stage 2's stream, for its next
    // use (pass A' of the batch that takes this set again, and the PEND bits the batch before that one leaves)
    CK(cudaMemsetAsync(sc.bitmap, 0, h->bm_words * sizeof(u32), st));
    CK(cudaMemsetAsync(sc.pend, 0, h->pend_words * sizeof(u32), st));   // (the bits the previous batch left: read by pass B)
    if (timed) CK(cudaEventRecord(h->evd[5], st));
    RC(enqueue_sort(h, sc, n_max, n_res, st, &rs));
    if (timed) CK(cudaEventRecord(h->evd[6], st));
    OutMap om{};
    om.out = nullptr;
    om.by_row = 1;
    om.compact = compact ? 1 : 0;
    om.view = v;
    om.pol = h->d_pol;
    om.npol = h->npol;
    om.now_batch = now_batch;
    RC(enqueue_decide_sorted(h, sc, n_max, n_res, rs, om, st));
    if (timed) { CK(cudaEventRecord(h->ev[3], st)); h->ev_valid = true; CK(cudaEventRecord(h->evd[7], st)); h->evd_valid = true; }
    CK(cudaGetLastError());
    return GCRA_OK;
}

// Stage 2 of a sort-pipeline batch: the compare-and-update kernels over the sorted keys
static int enqueue_back_sorted(gcra_engine *h, Scratch &sc, const BatchView &v, const u64 *sorted, cudaStream_t st, bool timed) {
    OutMap om{};
    om.out = v.res0;
    om.by_row = 0;
    RC(enqueue_decide_sorted(h, sc, v.n, nullptr, sorted, om, st));
    if (timed) { CK(cudaEventRecord(h->ev[3], st)); h->ev_valid = true; }
    CK(cudaGetLastError());
    return GCRA_OK;
}

static int check_batch(gcra_engine *h, uint32_t n, bool compact) {
    if (n > h->max_batch) { h->err = "batch larger than max_batch"; return GCRA_INTERNAL; }
    if (compact && h->npol == 0) { h->err = "no policy table registered"; return GCRA_INTERNAL; }
    return ensure_room(h, n);
}

// ---- one batch, everything on the caller's stream ------------------------------------------------
static int launch_batch(gcra_engine *h, uint32_t n, const void *d_req, bool compact, int64_t now_batch,
                        gcra_result *d_res, cudaStream_t st, bool timed) {
    if (n == 0) return GCRA_OK;
    RC(check_batch(h, n, compact));
    const uint32_t k = h->scr_next;
    Scratch &sc = h->scr[k];
    h->scr_next = (h->scr_next + 1) % gcra_engine::N_SCR;
    Scratch &next = h->scr[h->scr_next];
    // order after every earlier batch (they may have been submitted pipelined on the engine's streams),
    // which also frees this scratch set
    for (auto &o : h->scr) if (o.back_recorded) CK(cudaStreamWaitEvent(st, o.ev_back, 0));
    static const bool no_small = getenv("GCRA_NO_SMALL") && atoi(getenv("GCRA_NO_SMALL"));   // A/B switch for tools/latency_probe.py
    if (n <= SMALL_MAX && !no_small) {
        // small batch (a single rate_limit call, a lightly loaded actor): one CTA does ingest, ordering and
        // the compare-and-update in a single launch
        if (timed) { CK(cudaEventRecord(h->ev[0], st)); CK(cudaEventRecord(h->ev[1], st)); CK(cudaEventRecord(h->ev[2], st)); }
        if (compact)
            small_batch_kernel<true><<<1, TILE_THREADS, 0, st>>>(h->tab, d_req, h->d_pol, h->npol, now_batch, n, sc.drec, d_res);
        else
            small_batch_kernel<false><<<1, TILE_THREADS, 0, st>>>(h->tab, d_req, nullptr, 0, 0, n, sc.drec, d_res);
        h->launches++;
        if (timed) { CK(cudaEventRecord(h->ev[3], st)); h->ev_valid = true; }
        CK(cudaGetLastError());
    } else {
        u64 *sorted = nullptr;
        const BatchView v = single_view(d_req, d_res, n);
        const bool ip = use_index_path(h, n);
        RC(enqueue_front(h, sc, v, ip, compact, now_batch, st, timed, &sorted));
        if (ip) {
            RC(enqueue_mid_index(h, sc, next, v, compact, now_batch, false, st, timed));
            CK(cudaEventRecord(sc.ev_mid, st));
            sc.mid_recorded = true;
            RC(enqueue_tail_index(h, sc, v, compact, now_batch, st, timed));
        } else {
            RC(enqueue_back_sorted(h, sc, v, sorted, st, timed));
            sc.mid_recorded = false;
        }
    }
    RC(enqueue_denied(h, single_view(d_req, d_res, n), compact, st));
    CK(cudaEventRecord(sc.ev_back, st));
    sc.back_recorded = true;
    h->pend_set = -1;          // everything of this batch is ordered on `st`: the next batch waits for all of it
    return snapshot_async(h, n, st);
}

// ---- one batch, pipelined over the engine's streams --------------------------------------------------
// index-order pipeline: stage 1 (probe) of batch j+1 overlaps stage 2 (decide, resolve) of batch j and stage 3
// (the sorted residue) of batch j-1.  Stage 2 of batch j may run while the tail of batch j-1 is still at work
// because pass C of batch j-1 left PEND bits for exactly the keys that tail owns.  Sort pipeline: stage 1 =
// ingest + sort, stage 2 = decide, after every earlier batch has completely finished.
// `ready` (may be null) is an event after which the requests may be read; `*done` is set to an event after which
// the results are complete.
static int launch_pipelined_view(gcra_engine *h, const BatchView &v, uint32_t n_rows, bool compact, int64_t now_batch,
                                 cudaEvent_t ready, cudaEvent_t *done) {
    RC(check_batch(h, n_rows, compact));
    const uint32_t k = h->scr_next;
    Scratch &sc = h->scr[k];
    h->scr_next = (h->scr_next + 1) % gcra_engine::N_SCR;
    const uint32_t kn = h->scr_next;
    cudaStream_t fs = h->front_stream[k];                  // (all sets share one front stream, see gcra_create)
    if (ready) CK(cudaStreamWaitEvent(fs, ready, 0));
    if (sc.back_recorded) CK(cudaStreamWaitEvent(fs, sc.ev_back, 0));   // scratch set free again
    u64 *sorted = nullptr;
    // residue feedback: the newest pass-C count that has reached the host
    bool residue_large = false;
    for (int back = 1; back < gcra_engine::N_SCR; back++) {
        Scratch &os = h->scr[(k + gcra_engine::N_SCR - back) % gcra_engine::N_SCR];
        if (!os.mid_recorded || cudaEventQuery(os.ev_mid) != cudaSuccess) continue;
        if (!os.nres_counted) { h->residue_seen += *os.h_nres; h->residue_batches_seen++; os.nres_counted = true; }
        h->last_nres = *os.h_nres;
        h->last_nres_rows = os.nres_rows;
        residue_large = (uint64_t)*os.h_nres * 8 > os.nres_rows;
        break;
    }
    bool ip = v.nseg > 1 || use_index_path(h, n_rows);
    if (ip && v.nseg == 1 && h->adaptive) {
        // Which pipeline?  The index-order pipeline wins while most requests are decided in passes B and C; when
        // more than a quarter of a batch went through the sorted tail (keys spending a burst: every request
        // changes the state), sorting everything once is cheaper: the next 31 batches take the sort pipeline,
        // then the index-order pipeline is tried again.
        if (h->sort_hold > 0) { h->sort_hold--; ip = false; }
        else if (h->last_nres_rows && (uint64_t)h->last_nres * 4 > h->last_nres_rows) {
            h->sort_hold = 31; h->last_nres = 0; h->last_nres_rows = 0; ip = false; h->n_path_switches++;
        }
    }
    RC(enqueue_front(h, sc, v, ip, compact, now_batch, fs, false, &sorted));
    CK(cudaEventRecord(sc.ev_front, fs));
    cudaStream_t ms = h->back_stream;
    CK(cudaStreamWaitEvent(ms, sc.ev_front, 0));
    // May stage 2 of this batch overlap the tail of the batch submitted just before?  Only if that batch left its
    // PEND bits in this set's pend bitmap.  Keys the tail owns stay deferred for as long as they keep appearing
    // (their requests go from tail to tail), so the overlap is given up -- stage 2 waits for every tail and ignores
    // the PEND bits -- whenever the residue reported by an earlier batch has grown beyond 1/8 of its rows, and
    // every 64 batches.
    bool overlap = ip && h->pend_set == (int)k;
    if (ip) {
        if (residue_large && h->since_drain >= 2) overlap = false;
        if (h->since_drain >= 64) overlap = false;
        if (!overlap) { if (h->pend_set == (int)k) h->n_drains++; h->since_drain = 0; } else h->since_drain++;
    }
    for (int o = 0; o < gcra_engine::N_SCR; o++) {
        Scratch &os = h->scr[o];
        if (o == (int)k || !os.back_recorded) continue;
        const bool is_prev = o == (int)((k + gcra_engine::N_SCR - 1) % gcra_engine::N_SCR);
        if (overlap && is_prev) continue;
        CK(cudaStreamWaitEvent(ms, os.ev_back, 0));
    }
    if (ip) {
        RC(enqueue_mid_index(h, sc, h->scr[kn], v, compact, now_batch, overlap, ms, false));
        CK(cudaEventRecord(sc.ev_mid, ms));
        sc.mid_recorded = true;
        cudaStream_t ts = h->tail_stream;
        CK(cudaStreamWaitEvent(ts, sc.ev_mid, 0));
        RC(enqueue_tail_index(h, sc, v, compact, now_batch, ts, false));
        RC(enqueue_denied(h, v, compact, ts));
        CK(cudaEventRecord(sc.ev_back, ts));
        sc.back_recorded = true;
        h->pend_set = (int)kn;
        if (done) *done = sc.ev_back;
        return snapshot_async(h, n_rows, ts);
    }
    RC(enqueue_back_sorted(h, sc, v, sorted, ms, false));
    RC(enqueue_denied(h, v, compact, ms));
    sc.mid_recorded = false;   // (no residue count from this batch)
    CK(cudaEventRecord(sc.ev_back, ms));
    sc.back_recorded = true;
    h->pend_set = -1;
    if (done) *done = sc.ev_back;
    return snapshot_async(h, n_rows, ms);
}

static int launch_pipelined(gcra_engine *h, uint32_t n, const void *d_req, bool compact, int64_t now_batch,
                            gcra_result *d_res, cudaEvent_t ready, cudaEvent_t *done) {
    if (n == 0) { if (done) *done = nullptr; return GCRA_OK; }
    return launch_pipelined_view(h, single_view(d_req, d_res, n), n, compact, now_batch, ready, done);
}

// CUDA loads a kernel's code lazily, at its FIRST launch, and that load may wait for running kernels.  The
// multi-GPU pipelines keep kernels running that wait for work other launches deliver (flags in peer memory), so a
// first launch behind such a kernel would stall until the wait gives up: load everything when the engine is made.
template <typename K>
static void preload(K kernel) {
    cudaFuncAttributes a;
    cudaFuncGetAttributes(&a, kernel);
}

static void preload_kernels() {
    preload(ingest_kernel<false>); preload(ingest_kernel<true>);
    preload(small_batch_kernel<false>); preload(small_batch_kernel<true>);
    preload(sort_digits_hist_kernel); preload(sort_onesweep_kernel);
    preload(decide_kernel<false>); preload(decide_kernel<true>);
    preload(decide_runs_kernel<1, false>); preload(decide_runs_kernel<CLUSTER_CTAS, false>);
    preload(decide_runs_kernel<1, true>); preload(decide_runs_kernel<CLUSTER_CTAS, true>);
    preload(probe_kernel<false>); preload(probe_kernel<true>);
    preload(decide_index_kernel<false>); preload(decide_index_kernel<true>);
    preload(resolve_kernel<false>); preload(resolve_kernel<true>);
    preload(sweep_kernel); preload(purge_kernel); preload(clear_slots_kernel); preload(rehash_kernel); preload(store_op_kernel);
    preload(route_count_kernel); preload(route_scan_kernel); preload(route_scatter_kernel); preload(route_unpermute_kernel);
    preload(p2p_scan_kernel); preload(p2p_scatter_kernel); preload(p2p_signal_req_kernel); preload(p2p_signal_res_kernel);
    preload(p2p_wait_kernel); preload(p2p_unpermute_kernel);
    preload(denied_count_kernel<false>); preload(denied_count_kernel<true>);
}

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

int32_t gcra_create(const gcra_config *cfg, gcra_engine **out) {
    if (!cfg || !out) return GCRA_INTERNAL;
    *out = nullptr;
    gcra_engine *h = new gcra_engine();
    auto fail = [&](const char *what, cudaError_t e) {
        fprintf(stderr, "gcra_create: %s: %s\n", what, cudaGetErrorString(e));
        delete h;
        return (int32_t)GCRA_INTERNAL;
    };
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) return fail("no CUDA device (this engine has no CPU path)", e);
    if (cfg->device < 0 || cfg->device >= ndev) return fail("bad device ordinal", cudaErrorInvalidDevice);
    h->device = cfg->device;
    if ((e = cudaSetDevice(h->device)) != cudaSuccess) return fail("cudaSetDevice", e);
    if (const char *g = getenv("GCRA_L2_FETCH")) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)atoi(g));
    if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) return fail("stream", e);
    cudaStreamCreateWithFlags(&h->in_stream, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&h->out_stream, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&h->aux_stream, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&h->aux2_stream, cudaStreamNonBlocking);
    // ONE front stream shared by all scratch sets (front halves run one after another; since ingest only CASes
    // the keys array they could overlap as well -- not measured yet)
    cudaStreamCreateWithFlags(&h->front_stream[0], cudaStreamNonBlocking);
    for (int k = 1; k < gcra_engine::N_SCR; k++) h->front_stream[k] = h->front_stream[0];
    cudaStreamCreateWithFlags(&h->back_stream, cudaStreamNonBlocking);
    cudaStreamCreateWithFlags(&h->tail_stream, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&h->ev_ready, cudaEventDisableTiming);
    h->capacity = cfg->capacity ? cfg->capacity : 1000;      // DEFAULT_CAPACITY adaptive_cleanup.rs:10
    h->max_batch = cfg->max_batch ? cfg->max_batch : (1u << 20);
    h->tight = (cfg->flags & GCRA_FLAG_TIGHT_TABLE) != 0;
    h->hash_seed[0] = cfg->hash_seed[0];
    h->hash_seed[1] = cfg->hash_seed[1];
    if (cfg->flags & GCRA_FLAG_RANDOM_SEED) {
        FILE *ur = fopen("/dev/urandom", "rb");
        if (!ur || fread(h->hash_seed, sizeof(h->hash_seed), 1, ur) != 1) {
            if (ur) fclose(ur);
            fprintf(stderr, "gcra_create: cannot read /dev/urandom for the hash seed\n");
            delete h;
            return GCRA_INTERNAL;
        }
        fclose(ur);
        h->hash_seed[0] |= 1;      // never (0, 0)
    }
    u64 *counters = nullptr;
    if ((e = cudaMalloc(&counters, C_COUNT * sizeof(u64))) != cudaSuccess) return fail("counters", e);
    cudaMemsetAsync(counters, 0, C_COUNT * sizeof(u64), h->stream);
    if (alloc_table(h, h->capacity, h->tab, h->total_lines, counters)) {
        fprintf(stderr, "gcra_create: %s\n", h->err.c_str());
        delete h;
        return GCRA_INTERNAL;
    }
    const size_t mb = h->max_batch;
    const uint32_t stiles = sort_tiles_max(h);
    {
        // index-order pipeline: hashed batch counters (16 bits) and pend bits, 8 entries per row of the largest
        // batch (n distinct slots share their entry with probability ~1/8), 64 K .. 16 M entries
        uint32_t lg = ceil_log2(std::max<uint64_t>(8ULL * mb, 1ULL << 16));
        if (lg > 24) lg = 24;
        h->bm_mask = (1u << lg) - 1;
        h->bm_words = (size_t)1 << (lg - 1);      // 16-bit counters, 2 per word
        h->pend_words = (size_t)1 << (lg - 5);    // 1 bit per entry
        h->index_min = 32768;
        if (const char *g = getenv("GCRA_INDEX_MIN")) { h->index_min = (uint32_t)atoll(g); h->adaptive = false; }
        if (cfg->flags & GCRA_FLAG_INDEX_PATH) { h->index_min = SMALL_MAX + 1; h->adaptive = false; }
        if (cfg->flags & GCRA_FLAG_SORT_PATH) { h->index_min = 0; h->adaptive = false; }
        if (const char *g = getenv("GCRA_ADAPTIVE")) h->adaptive = atoi(g) != 0;
        h->prefetch_state = 0;
        if (const char *g = getenv("GCRA_PREFETCH")) h->prefetch_state = atoi(g);
        int sms = 148, nb = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, probe_kernel<false>, TILE_THREADS, 0) == cudaSuccess && nb > 0) h->grid_probe[0] = (uint32_t)(nb * sms);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, probe_kernel<true>, TILE_THREADS, 0) == cudaSuccess && nb > 0) h->grid_probe[1] = (uint32_t)(nb * sms);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, decide_index_kernel<false>, TILE_THREADS, 0) == cudaSuccess && nb > 0) h->grid_decide[0] = (uint32_t)(nb * sms);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, decide_index_kernel<true>, TILE_THREADS, 0) == cudaSuccess && nb > 0) h->grid_decide[1] = (uint32_t)(nb * sms);
        // tuning: CTAs per SM of the persistent kernels (fewer leave room for the other stages' kernels)
        if (const char *g = getenv("GCRA_CTAS_PROBE")) { uint32_t c = (uint32_t)atoi(g) * sms; if (c) { h->grid_probe[0] = std::min(h->grid_probe[0], c); h->grid_probe[1] = std::min(h->grid_probe[1], c); } }
        if (const char *g = getenv("GCRA_CTAS_DECIDE")) { uint32_t c = (uint32_t)atoi(g) * sms; if (c) { h->grid_decide[0] = std::min(h->grid_decide[0], c); h->grid_decide[1] = std::min(h->grid_decide[1], c); } }
    }
    bool ok = cudaMalloc(&h->d_req, mb * sizeof(gcra_request)) == cudaSuccess &&
              cudaMalloc(&h->d_res, mb * sizeof(gcra_result)) == cudaSuccess &&
              cudaMalloc(&h->route_counts, (size_t)ROUTE_MAX_SHARDS * ((mb + TILE_THREADS - 1) / TILE_THREADS) * sizeof(u32)) == cudaSuccess &&
              cudaMalloc(&h->d_op, 2 * sizeof(StoreOpResult)) == cudaSuccess &&
              cudaMallocHost(&h->h_op, 2 * sizeof(StoreOpResult)) == cudaSuccess &&
              cudaMallocHost(&h->h_counters, C_COUNT * sizeof(u64)) == cudaSuccess &&
              cudaMallocHost(&h->h_snap, (size_t)gcra_engine::N_SNAP * C_COUNT * sizeof(u64)) == cudaSuccess;
    for (int k = 0; k < gcra_engine::N_SCR && ok; k++) {
        Scratch &sc = h->scr[k];
        ok = cudaMalloc(&sc.drec, mb * sizeof(Req)) == cudaSuccess &&
             cudaMalloc(&sc.keys_a, mb * sizeof(u64)) == cudaSuccess &&
             cudaMalloc(&sc.keys_b, mb * sizeof(u64)) == cudaSuccess &&
             cudaMalloc(&sc.sort_status, (size_t)SORT_MAX_DIGITS * stiles * sizeof(u64)) == cudaSuccess &&
             cudaMemset(sc.sort_status, 0, (size_t)SORT_MAX_DIGITS * stiles * sizeof(u64)) == cudaSuccess &&
             cudaMalloc(&sc.sort_tot, (2 * SORT_MAX_PASSES * SORT_MAX_DIGITS + 1) * sizeof(u32)) == cudaSuccess &&
             cudaMemset(sc.sort_tot, 0, (2 * SORT_MAX_PASSES * SORT_MAX_DIGITS + 1) * sizeof(u32)) == cudaSuccess &&
             cudaMalloc(&sc.long_runs, (mb / LONG_RUN_MIN + 1) * sizeof(LongRun)) == cudaSuccess &&
             cudaMalloc(&sc.giant_runs, (mb / GIANT_RUN_MIN + 1) * sizeof(LongRun)) == cudaSuccess &&
             cudaMalloc(&sc.long_count, 2 * sizeof(u32)) == cudaSuccess &&
             cudaEventCreateWithFlags(&sc.ev_front, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&sc.ev_back, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&sc.ev_mid, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&sc.ev_fork, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&sc.ev_join, cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&sc.ev_join2, cudaEventDisableTiming) == cudaSuccess;
        if (ok) sc.sort_ticket = sc.sort_tot + 2 * SORT_MAX_PASSES * SORT_MAX_DIGITS;
        ok = ok && alloc_index_scratch(h, sc, h->max_batch) == GCRA_OK;
    }
    if (!ok) return fail("scratch allocation", cudaGetLastError());
    memset(h->h_counters, 0, C_COUNT * sizeof(u64));
    cudaEventCreateWithFlags(&h->ev_counters, cudaEventDisableTiming);
    for (int i = 0; i < gcra_engine::N_SNAP; i++) cudaEventCreateWithFlags(&h->ev_snap[i], cudaEventDisableTiming);
    for (int i = 0; i < 4; i++) cudaEventCreate(&h->ev[i]);
    for (int i = 0; i < 8; i++) cudaEventCreate(&h->evd[i]);
    cudaEventCreate(&h->ev_sweep[0]);
    cudaEventCreate(&h->ev_sweep[1]);
    // store policy, defaults as in the reference constructors
    h->kind = cfg->store_kind;
    __int128 created = cfg->created_ns;
    if (h->kind == GCRA_STORE_PERIODIC) {
        h->cleanup_interval = (__int128)(cfg->p0 ? cfg->p0 : 60) * NS_PER_S;       // periodic.rs:12
        h->next_cleanup = created + h->cleanup_interval;
    } else if (h->kind == GCRA_STORE_PROBABILISTIC) {
        h->cleanup_modulo = cfg->p0 ? cfg->p0 : 1000;                               // probabilistic.rs:12
    } else if (h->kind == GCRA_STORE_ADAPTIVE) {
        h->min_interval = (__int128)(cfg->p0 ? cfg->p0 : 1) * NS_PER_S;            // adaptive_cleanup.rs:12-15
        h->max_interval = (__int128)(cfg->p1 ? cfg->p1 : 300) * NS_PER_S;
        h->max_ops = cfg->p2 ? cfg->p2 : 100000;
        h->cur_interval = 5 * NS_PER_S;
        h->next_cleanup = created + 5 * NS_PER_S;
    }
    preload_kernels();
    if ((e = cudaStreamSynchronize(h->stream)) != cudaSuccess) return fail("init", e);
    *out = h;
    return GCRA_OK;
}

void gcra_destroy(gcra_engine *h) {
    if (!h) return;
    cudaSetDevice(h->device);
    cudaDeviceSynchronize();
    if (h->shard) {
        Shard *sh = h->shard;
        for (auto &sl : sh->slots) {
            cudaFree(sl.routed); cudaFree(sl.recv_req); cudaFree(sl.recv_res); cudaFree(sl.back_res); cudaFree(sl.src_index);
            cudaFree(sl.counts_dev); cudaFreeHost(sl.counts_host);
            cudaEventDestroy(sl.ev_ready); cudaEventDestroy(sl.ev_counts); cudaEventDestroy(sl.ev_routed); cudaEventDestroy(sl.ev_done);
        }
        if (nccl_rt::g_api.CommDestroy) { nccl_rt::g_api.CommDestroy(sh->comm_counts); nccl_rt::g_api.CommDestroy(sh->comm_req); nccl_rt::g_api.CommDestroy(sh->comm_res); }
        cudaStreamDestroy(sh->s_part); cudaStreamDestroy(sh->s_route); cudaStreamDestroy(sh->s_return); cudaEventDestroy(sh->ev_tmp);
        delete sh;
    }
    if (h->p2p) {
        P2P *p = h->p2p;
        for (int r = 0; r < p->world; r++) if (p->opened[r]) cudaIpcCloseMemHandle(p->peer_base[r]);
        for (auto &sl : p->slots) {
            cudaFree(sl.res_loc); cudaFree(sl.counts_dev); cudaFree(sl.segs_dev);
            cudaEventDestroy(sl.ev_ready); cudaEventDestroy(sl.ev_wait); cudaEventDestroy(sl.ev_done);
        }
        for (auto &e : p->ev_t) cudaEventDestroy(e);
        cudaFree(p->peers_dev); cudaFree(p->tile_counts); cudaFree(p->window);
        cudaStreamDestroy(p->s_part); cudaStreamDestroy(p->s_wait); cudaStreamDestroy(p->s_sig); cudaStreamDestroy(p->s_return);
        delete p;
    }
    for (auto &s : h->ring) {
        cudaFreeHost(s.h_req); cudaFreeHost(s.h_res); cudaFree(s.d_req); cudaFree(s.d_res);
        cudaEventDestroy(s.ev_in); cudaEventDestroy(s.ev_comp); cudaEventDestroy(s.ev_done);
    }
    cudaFree(h->tab.keys); cudaFree(h->tab.state); cudaFree(h->tab.ei); cudaFree(h->tab.mark); cudaFree(h->tab.counters);
    for (auto &sc : h->scr) {
        cudaFree(sc.drec); cudaFree(sc.keys_a); cudaFree(sc.keys_b); cudaFree(sc.sort_status); cudaFree(sc.sort_tot);
        cudaFree(sc.long_runs); cudaFree(sc.giant_runs); cudaFree(sc.long_count);
        cudaFree(sc.slot_arr); cudaFree(sc.flags); cudaFree(sc.bitmap); cudaFree(sc.pend); cudaFree(sc.ctrl_block);
        cudaFreeHost(sc.h_nres);
        cudaEventDestroy(sc.ev_front); cudaEventDestroy(sc.ev_mid); cudaEventDestroy(sc.ev_back); cudaEventDestroy(sc.ev_fork); cudaEventDestroy(sc.ev_join); cudaEventDestroy(sc.ev_join2);
    }
    cudaFree(h->denied.keys); cudaFree(h->denied.counts); cudaFree(h->denied.dropped);
    cudaFree(h->d_req); cudaFree(h->d_res); cudaFree(h->route_counts); cudaFree(h->d_pol); cudaFree(h->d_op);
    cudaFreeHost(h->h_op); cudaFreeHost(h->h_counters); cudaFreeHost(h->h_snap);
    for (int i = 0; i < gcra_engine::N_SNAP; i++) cudaEventDestroy(h->ev_snap[i]);
    cudaEventDestroy(h->ev_counters);
    for (int i = 0; i < 4; i++) cudaEventDestroy(h->ev[i]);
    for (int i = 0; i < 8; i++) cudaEventDestroy(h->evd[i]);
    cudaEventDestroy(h->ev_sweep[0]); cudaEventDestroy(h->ev_sweep[1]);
    cudaStreamDestroy(h->stream); cudaStreamDestroy(h->in_stream); cudaStreamDestroy(h->out_stream); cudaStreamDestroy(h->aux_stream); cudaStreamDestroy(h->aux2_stream);
    cudaStreamDestroy(h->front_stream[0]);
    cudaStreamDestroy(h->back_stream); cudaStreamDestroy(h->tail_stream); cudaEventDestroy(h->ev_ready);
    delete h;
}

const char *gcra_last_error(gcra_engine *h) { return h ? h->err.c_str() : "null handle"; }

uint64_t gcra_hash_key(const void *key, uint64_t len) {
    const unsigned char *p = (const unsigned char *)key;
    uint64_t hsh = 0x2545F4914F6CDD1DULL ^ (len * 0x9E3779B97F4A7C15ULL);
    while (len >= 8) {
        uint64_t w;
        memcpy(&w, p, 8);
        hsh = mix64(hsh ^ w) + 0xD1B54A32D192ED03ULL;
        p += 8; len -= 8;
    }
    if (len) {
        uint64_t w = 0;
        memcpy(&w, p, len);
        hsh = mix64(hsh ^ w ^ (len << 56));
    }
    return mix64(hsh);
}

// SipHash-2-4 (Aumasson & Bernstein), 64-bit output: the keyed hash for keys an adversary may choose
static inline uint64_t rotl64(uint64_t x, int b) { return (x << b) | (x >> (64 - b)); }
uint64_t gcra_hash_key_seeded(const void *key, uint64_t len, uint64_t k0, uint64_t k1) {
    uint64_t v0 = 0x736f6d6570736575ULL ^ k0, v1 = 0x646f72616e646f6dULL ^ k1;
    uint64_t v2 = 0x6c7967656e657261ULL ^ k0, v3 = 0x7465646279746573ULL ^ k1;
    const unsigned char *p = (const unsigned char *)key;
    const unsigned char *end = p + (len & ~7ULL);
#define GCRA_SIPROUND                                                                 \
    do {                                                                              \
        v0 += v1; v1 = rotl64(v1, 13); v1 ^= v0; v0 = rotl64(v0, 32);                \
        v2 += v3; v3 = rotl64(v3, 16); v3 ^= v2;                                      \
        v0 += v3; v3 = rotl64(v3, 21); v3 ^= v0;                                      \
        v2 += v1; v1 = rotl64(v1, 17); v1 ^= v2; v2 = rotl64(v2, 32);                \
    } while (0)
    for (; p != end; p += 8) {
        uint64_t m;
        memcpy(&m, p, 8);
        v3 ^= m; GCRA_SIPROUND; GCRA_SIPROUND; v0 ^= m;
    }
    uint64_t b = len << 56;
    for (uint64_t i = 0; i < (len & 7); i++) b |= (uint64_t)p[i] << (8 * i);
    v3 ^= b; GCRA_SIPROUND; GCRA_SIPROUND; v0 ^= b;
    v2 ^= 0xff;
    GCRA_SIPROUND; GCRA_SIPROUND; GCRA_SIPROUND; GCRA_SIPROUND;
#undef GCRA_SIPROUND
    return v0 ^ v1 ^ v2 ^ v3;
}

// the identity the engine's own string-keyed entry points give a key: keyed when the engine has a seed
static uint64_t engine_hash(const gcra_engine *h, const void *key, uint64_t len) {
    return (h->hash_seed[0] | h->hash_seed[1]) ? gcra_hash_key_seeded(key, len, h->hash_seed[0], h->hash_seed[1])
                                               : gcra_hash_key(key, len);
}

uint64_t gcra_engine_hash_key(gcra_engine *h, const void *key, uint64_t len) { return engine_hash(h, key, len); }

void gcra_get_hash_seed(gcra_engine *h, uint64_t out[2]) { out[0] = h->hash_seed[0]; out[1] = h->hash_seed[1]; }

void gcra_hash_key_ids(const void *prefix, uint64_t prefix_len, const uint64_t *ids, uint64_t n, uint64_t *out) {
    char buf[96];
    if (prefix_len > 64) prefix_len = 64;
    memcpy(buf, prefix, prefix_len);
    for (uint64_t i = 0; i < n; i++) {
        char tmp[24];
        int k = 0;
        uint64_t v = ids[i];
        do { tmp[k++] = (char)('0' + v % 10); v /= 10; } while (v);
        for (int j = 0; j < k; j++) buf[prefix_len + j] = tmp[k - 1 - j];
        out[i] = gcra_hash_key(buf, prefix_len + k);
    }
}

int32_t gcra_derive_params(int64_t max_burst, int64_t count, int64_t period, int64_t *ei, int64_t *dvt) {
    i64 a = 0, b = 0;
    int st = derive_params(max_burst, count, period, &a, &b);
    if (ei) *ei = a;
    if (dvt) *dvt = b;
    return st;
}

static int store_op(gcra_engine *h, int op, uint64_t key_hash, int64_t a, int64_t b, uint64_t ttl, int64_t now) {
    CK(cudaSetDevice(h->device));
    // the table encodes 'no state' as a negative expiry: times before the epoch are outside its domain
    if (op != 3 && now < 0) { h->err = "pre-epoch time is not supported"; return GCRA_INTERNAL; }
    if (op == 2) { int rc = ensure_room(h, 1); if (rc) return rc; }
    // a Store-trait call reads / writes a slot's state: after every batch still in flight on the engine's or a
    // caller's stream (launch_batch orders itself the same way)
    for (auto &o : h->scr) if (o.back_recorded) CK(cudaStreamWaitEvent(h->stream, o.ev_back, 0));
    store_op_kernel<<<1, 1, 0, h->stream>>>(h->tab, op, stored_key(key_hash), a, b, ttl, now, h->d_op);
    h->launches++;
    CK(cudaMemcpyAsync(h->h_op, h->d_op, 2 * sizeof(StoreOpResult), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return GCRA_OK;
}

static int policy_before_mutation(gcra_engine *h, int64_t now_ns) {
    // the reference's mutating ops start with maybe_clean_expired(now) (adaptive_cleanup.rs:229,261)
    int rc = refresh_counters(h, true);
    if (rc) return rc;
    return apply_policy(h, now_ns);
}

int32_t gcra_store_get(gcra_engine *h, const void *key, uint64_t len, int64_t now_ns, int64_t *value,
                       uint8_t *found) {
    int rc = store_op(h, 0, engine_hash(h, key, len), 0, 0, 0, now_ns);
    if (rc) return rc;
    if (found) *found = (uint8_t)h->h_op[0].flag;
    if (value) *value = h->h_op[0].value;
    return GCRA_OK;
}

int32_t gcra_store_cas(gcra_engine *h, const void *key, uint64_t len, int64_t old_value, int64_t new_value,
                       uint64_t ttl_ns, int64_t now_ns, uint8_t *swapped) {
    int rc = policy_before_mutation(h, now_ns);
    if (rc) return rc;
    rc = store_op(h, 1, engine_hash(h, key, len), old_value, new_value, ttl_ns, now_ns);
    if (rc) return rc;
    if (swapped) *swapped = (uint8_t)h->h_op[0].flag;
    return GCRA_OK;
}

int32_t gcra_store_set_nx(gcra_engine *h, const void *key, uint64_t len, int64_t value, uint64_t ttl_ns,
                          int64_t now_ns, uint8_t *stored) {
    int rc = policy_before_mutation(h, now_ns);
    if (rc) return rc;
    rc = store_op(h, 2, engine_hash(h, key, len), value, 0, ttl_ns, now_ns);
    if (rc) return rc;
    if (h->h_op[0].status) { h->err = "table full"; return GCRA_INTERNAL; }
    if (stored) *stored = (uint8_t)h->h_op[0].flag;
    return GCRA_OK;
}

int32_t gcra_rate_limit_batch_device(gcra_engine *h, uint64_t n, const gcra_request *d_req, gcra_result *d_res,
                                     void *stream) {
    CK(cudaSetDevice(h->device));
    return launch_batch(h, (uint32_t)n, d_req, false, 0, d_res, stream ? (cudaStream_t)stream : h->stream, true);
}

int32_t gcra_rate_limit_batch16_device(gcra_engine *h, uint64_t n, const gcra_request16 *d_req, int64_t now_ns,
                                       gcra_result *d_res, void *stream) {
    CK(cudaSetDevice(h->device));
    return launch_batch(h, (uint32_t)n, d_req, true, now_ns, d_res, stream ? (cudaStream_t)stream : h->stream, true);
}

int32_t gcra_rate_limit_batch_device_pipelined(gcra_engine *h, uint64_t n, const gcra_request *d_req,
                                               gcra_result *d_res, void *ready_stream) {
    CK(cudaSetDevice(h->device));
    cudaEvent_t ready = nullptr;
    if (ready_stream) {
        CK(cudaEventRecord(h->ev_ready, (cudaStream_t)ready_stream));
        ready = h->ev_ready;
    }
    return launch_pipelined(h, (uint32_t)n, d_req, false, 0, d_res, ready, nullptr);
}

int32_t gcra_pipeline_join(gcra_engine *h, void *stream) {
    CK(cudaSetDevice(h->device));
    for (auto &o : h->scr) {
        if (!o.back_recorded) continue;
        if (stream) CK(cudaStreamWaitEvent((cudaStream_t)stream, o.ev_back, 0));
        else CK(cudaEventSynchronize(o.ev_back));
    }
    return GCRA_OK;
}

static int host_batch(gcra_engine *h, uint64_t n, const void *req, size_t rsz, bool compact, int64_t now_batch,
                      gcra_result *res) {
    CK(cudaSetDevice(h->device));
    uint64_t done = 0;
    while (done < n) {
        uint32_t m = (uint32_t)std::min<uint64_t>(n - done, h->max_batch);
        const unsigned char *src = (const unsigned char *)req + done * rsz;
        // like the reference's mutating ops, sweep (if the store's policy says so) BEFORE the work
        // (adaptive_cleanup.rs:229,261), with the clock of the first request of the chunk
        int64_t now_hint = compact ? now_batch : ((const gcra_request *)req)[done].now_ns;
        int rc = apply_policy(h, now_hint);
        if (rc) return rc;
        CK(cudaMemcpyAsync(h->d_req, src, (size_t)m * rsz, cudaMemcpyHostToDevice, h->stream));
        rc = launch_batch(h, m, h->d_req, compact, now_batch, h->d_res, h->stream, true);
        if (rc) return rc;
        CK(cudaMemcpyAsync(res + done, h->d_res, (size_t)m * sizeof(gcra_result), cudaMemcpyDeviceToHost, h->stream));
        RC(refresh_counters(h, false));
        CK(cudaStreamSynchronize(h->stream));
        done += m;
    }
    return GCRA_OK;
}

int32_t gcra_rate_limit_batch(gcra_engine *h, uint64_t n, const gcra_request *req, gcra_result *res) {
    return host_batch(h, n, req, sizeof(gcra_request), false, 0, res);
}

int32_t gcra_rate_limit_batch16(gcra_engine *h, uint64_t n, const gcra_request16 *req, int64_t now_ns,
                                gcra_result *res) {
    return host_batch(h, n, req, sizeof(gcra_request16), true, now_ns, res);
}

int32_t gcra_rate_limit(gcra_engine *h, const void *key, uint64_t len, int64_t max_burst, int64_t count_per_period,
                        int64_t period, int64_t quantity, int64_t now_ns, gcra_result *out) {
    gcra_request r = {engine_hash(h, key, len), max_burst, count_per_period, period, quantity, now_ns};
    gcra_result tmp;
    int rc = host_batch(h, 1, &r, sizeof(r), false, 0, &tmp);
    if (rc) { if (out) { memset(out, 0, sizeof(*out)); out->status = GCRA_INTERNAL; } return rc; }
    if (out) *out = tmp;
    if (tmp.status == GCRA_INTERNAL) h->err = "rate_limit: internal (duration overflow, pre-epoch time or table full)";
    return tmp.status;
}

int32_t gcra_set_policies(gcra_engine *h, uint32_t n, const gcra_policy *policies) {
    CK(cudaSetDevice(h->device));
    std::vector<PolicyDerived> pd(n);
    for (uint32_t i = 0; i < n; i++) {
        const gcra_policy &p = policies[i];
        pd[i].ei = pd[i].dvt = 0; pd[i].pad = 0;
        if (p.max_burst <= 0 || p.count_per_period <= 0 || p.period <= 0) pd[i].status = GCRA_INVALID_RATE_LIMIT;
        else pd[i].status = derive_params(p.max_burst, p.count_per_period, p.period, &pd[i].ei, &pd[i].dvt);
    }
    CK(cudaStreamSynchronize(h->stream));
    cudaFree(h->d_pol);
    h->d_pol = nullptr;
    h->npol = 0;
    if (n) {
        CK(cudaMalloc(&h->d_pol, n * sizeof(PolicyDerived)));
        CK(cudaMemcpy(h->d_pol, pd.data(), n * sizeof(PolicyDerived), cudaMemcpyHostToDevice));
        h->npol = n;
    }
    return GCRA_OK;
}

// ---- ring --------------------------------------------------------------------------------------
int32_t gcra_ring_create(gcra_engine *h, uint32_t slots, uint32_t slot_capacity, int32_t compact) {
    CK(cudaSetDevice(h->device));
    if (!h->ring.empty()) { h->err = "ring already created"; return GCRA_INTERNAL; }
    if (slot_capacity == 0 || slot_capacity > h->max_batch) { h->err = "slot_capacity must be in 1..max_batch"; return GCRA_INTERNAL; }
    h->ring_cap = slot_capacity;
    h->ring_compact = compact != 0;
    size_t rsz = compact ? sizeof(gcra_request16) : sizeof(gcra_request);
    h->ring.resize(slots);
    for (auto &s : h->ring) {
        // request slots are only WRITTEN by the host: optionally write-combined pinned memory (GCRA_RING_WC=1)
        CK(cudaHostAlloc(&s.h_req, slot_capacity * rsz,
                         getenv("GCRA_RING_WC") && atoi(getenv("GCRA_RING_WC")) ? cudaHostAllocWriteCombined : cudaHostAllocDefault));
        CK(cudaMallocHost(&s.h_res, slot_capacity * sizeof(gcra_result)));
        CK(cudaMalloc(&s.d_req, slot_capacity * rsz));
        CK(cudaMalloc(&s.d_res, slot_capacity * sizeof(gcra_result)));
        CK(cudaEventCreateWithFlags(&s.ev_in, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&s.ev_comp, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&s.ev_done, cudaEventDisableTiming));
    }
    return GCRA_OK;
}

void *gcra_ring_requests(gcra_engine *h, uint32_t slot) { return slot < h->ring.size() ? h->ring[slot].h_req : nullptr; }
gcra_result *gcra_ring_results(gcra_engine *h, uint32_t slot) { return slot < h->ring.size() ? h->ring[slot].h_res : nullptr; }

int32_t gcra_ring_submit(gcra_engine *h, uint32_t slot, uint32_t n, int64_t now_ns) {
    CK(cudaSetDevice(h->device));
    if (slot >= h->ring.size() || n > h->ring_cap) { h->err = "bad ring slot / size"; return GCRA_INTERNAL; }
    RingSlot &s = h->ring[slot];
    if (s.in_flight) { h->err = "ring slot still in flight"; return GCRA_INTERNAL; }
    // sweep policy with the counters of the batches finished so far (no stall)
    if (cudaEventQuery(h->ev_counters) == cudaSuccess) { int rc = apply_policy(h, now_ns); if (rc) return rc; }
    size_t rsz = h->ring_compact ? sizeof(gcra_request16) : sizeof(gcra_request);
    CK(cudaMemcpyAsync(s.d_req, s.h_req, (size_t)n * rsz, cudaMemcpyHostToDevice, h->in_stream));
    CK(cudaEventRecord(s.ev_in, h->in_stream));
    // front half (ingest + order) of this slot overlaps the back half (decide) of the previous one
    cudaEvent_t done = nullptr;
    int rc = launch_pipelined(h, n, s.d_req, h->ring_compact, now_ns, s.d_res, s.ev_in, &done);
    if (rc) return rc;
    if (done) CK(cudaStreamWaitEvent(h->out_stream, done, 0));
    CK(cudaMemcpyAsync(h->h_counters, h->tab.counters, C_COUNT * sizeof(u64), cudaMemcpyDeviceToHost, h->out_stream));
    CK(cudaEventRecord(h->ev_counters, h->out_stream));
    CK(cudaMemcpyAsync(s.h_res, s.d_res, (size_t)n * sizeof(gcra_result), cudaMemcpyDeviceToHost, h->out_stream));
    CK(cudaEventRecord(s.ev_done, h->out_stream));
    s.in_flight = true;
    return GCRA_OK;
}

int32_t gcra_ring_wait(gcra_engine *h, uint32_t slot) {
    if (slot >= h->ring.size()) { h->err = "bad ring slot"; return GCRA_INTERNAL; }
    RingSlot &s = h->ring[slot];
    if (!s.in_flight) return GCRA_OK;
    CK(cudaEventSynchronize(s.ev_done));
    s.in_flight = false;
    return GCRA_OK;
}

int32_t gcra_ring_poll(gcra_engine *h, uint32_t slot, int32_t *done) {
    if (slot >= h->ring.size()) { h->err = "bad ring slot"; return GCRA_INTERNAL; }
    RingSlot &s = h->ring[slot];
    if (!s.in_flight) { *done = 1; return GCRA_OK; }
    cudaError_t e = cudaEventQuery(s.ev_done);
    if (e == cudaSuccess) { s.in_flight = false; *done = 1; return GCRA_OK; }
    if (e == cudaErrorNotReady) { *done = 0; return GCRA_OK; }
    h->err = cudaGetErrorString(e);
    return GCRA_INTERNAL;
}

// ---- sweep / introspection ---------------------------------------------------------------------
int32_t gcra_sweep(gcra_engine *h, int64_t now_ns, uint64_t *removed) { return do_sweep(h, now_ns, removed); }

// The store kind's own sweep policy (maybe_clean_expired: adaptive_cleanup.rs:205-211, periodic.rs:128-142,
// probabilistic.rs:110-125) evaluated against the counters of everything finished so far.  The host-buffer calls
// and the ring do this themselves before every batch; the device-resident, pipelined and sharded submissions
// cannot (the requests' clocks live on the device): their caller ticks the policy with its own clock.
int32_t gcra_policy_tick(gcra_engine *h, int64_t now_ns, uint64_t *swept) {
    CK(cudaSetDevice(h->device));
    if (swept) *swept = 0;
    if (h->kind == GCRA_STORE_MANUAL) return GCRA_OK;
    for (auto &o : h->scr) if (o.back_recorded) CK(cudaEventSynchronize(o.ev_back));
    RC(refresh_counters(h, true));
    const uint64_t before = h->h_counters[C_SWEPT];
    RC(apply_policy(h, now_ns));
    if (swept) { RC(refresh_counters(h, true)); *swept = h->h_counters[C_SWEPT] - before; }
    return GCRA_OK;
}

uint64_t gcra_len(gcra_engine *h) {
    cudaSetDevice(h->device);
    if (refresh_counters(h, true)) return 0;
    return h->h_counters[C_REAL];
}

int32_t gcra_get_stats(gcra_engine *h, gcra_stats *out) {
    CK(cudaSetDevice(h->device));
    int rc = refresh_counters(h, true);
    if (rc) return rc;
    const u64 *c = h->h_counters;
    out->len = c[C_REAL];
    out->occupied_slots = c[C_OCCUPIED];
    out->table_slots = (uint64_t)h->total_lines * 4;
    out->stash_entries = c[C_STASH];
    out->allowed = c[C_ALLOWED];
    out->denied = c[C_DENIED];
    out->errors = c[C_ERRORS];
    out->expired_hits = c[C_EXPIRED_HITS];
    out->sweeps = h->n_sweeps;
    out->swept = c[C_SWEPT];
    out->grows = h->n_grows;
    out->purges = h->n_purges;
    out->index_batches = h->n_index_batches;
    out->residue_rows = h->residue_seen;
    out->residue_batches = h->residue_batches_seen;
    out->drains = h->n_drains;
    out->path_switches = h->n_path_switches;
    return GCRA_OK;
}

int32_t gcra_peek(gcra_engine *h, uint64_t key_hash, int64_t *tat, int64_t *expiry_ns, uint8_t *found) {
    int rc = store_op(h, 3, key_hash, 0, 0, 0, 0);
    if (rc) return rc;
    *found = (uint8_t)h->h_op[0].flag;
    if (*found) { *tat = h->h_op[0].value; *expiry_ns = h->h_op[1].value; }
    return GCRA_OK;
}

// ---- metrics bridge: top denied keys (throttlecrab-server/src/metrics.rs:24-64,162-173) --------------------------
int32_t gcra_track_denied(gcra_engine *h, uint32_t max_keys) {
    CK(cudaSetDevice(h->device));
    CK(cudaDeviceSynchronize());
    cudaFree(h->denied.keys); cudaFree(h->denied.counts); cudaFree(h->denied.dropped);
    h->denied = DeniedTable{};
    h->denied_max = max_keys;
    h->denied_cap = 0;
    if (!max_keys) return GCRA_OK;
    h->denied_cap = 1u << ceil_log2(std::max<uint64_t>(16ULL * max_keys, 1024));
    CK(cudaMalloc(&h->denied.keys, (size_t)h->denied_cap * sizeof(u64)));
    CK(cudaMalloc(&h->denied.counts, (size_t)h->denied_cap * sizeof(u64)));
    CK(cudaMalloc(&h->denied.dropped, sizeof(u64)));
    CK(cudaMemset(h->denied.keys, 0, (size_t)h->denied_cap * sizeof(u64)));
    CK(cudaMemset(h->denied.counts, 0, (size_t)h->denied_cap * sizeof(u64)));
    CK(cudaMemset(h->denied.dropped, 0, sizeof(u64)));
    h->denied.mask = h->denied_cap - 1;
    return GCRA_OK;
}

// the k most denied keys (hash, count), most denied first; *dropped = denials of keys that found the table full.
// Like the reference's cleanup (metrics.rs:52-64) the table is pruned to its `max_keys` top entries when more than
// three times as many have accumulated.
int32_t gcra_top_denied(gcra_engine *h, uint32_t k, uint64_t *key_hashes, uint64_t *counts, uint32_t *n_out, uint64_t *dropped) {
    CK(cudaSetDevice(h->device));
    if (n_out) *n_out = 0;
    if (!h->denied_max) { h->err = "gcra_track_denied first"; return GCRA_INTERNAL; }
    for (auto &o : h->scr) if (o.back_recorded) CK(cudaEventSynchronize(o.ev_back));
    std::vector<u64> keys(h->denied_cap), cnts(h->denied_cap);
    CK(cudaMemcpy(keys.data(), h->denied.keys, keys.size() * sizeof(u64), cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(cnts.data(), h->denied.counts, cnts.size() * sizeof(u64), cudaMemcpyDeviceToHost));
    if (dropped) CK(cudaMemcpy(dropped, h->denied.dropped, sizeof(u64), cudaMemcpyDeviceToHost));
    std::vector<std::pair<u64, u64>> top;      // (count, key)
    for (uint32_t i = 0; i < h->denied_cap; i++) if (keys[i]) top.emplace_back(cnts[i], keys[i]);
    std::sort(top.begin(), top.end(), [](const std::pair<u64, u64> &a, const std::pair<u64, u64> &b) {
        return a.first != b.first ? a.first > b.first : a.second < b.second;
    });
    const uint32_t n = (uint32_t)std::min<size_t>(k, top.size());
    for (uint32_t i = 0; i < n; i++) { key_hashes[i] = top[i].second; counts[i] = top[i].first; }
    if (n_out) *n_out = n;
    if (top.size() > (size_t)3 * h->denied_max) {
        std::fill(keys.begin(), keys.end(), 0);
        std::fill(cnts.begin(), cnts.end(), 0);
        for (uint32_t i = 0; i < h->denied_max; i++) {
            uint32_t s = (uint32_t)(mix64(top[i].second ^ 0x9E3779B97F4A7C15ULL)) & h->denied.mask;
            while (keys[s]) s = (s + 1) & h->denied.mask;
            keys[s] = top[i].second;
            cnts[s] = top[i].first;
        }
        CK(cudaMemcpy(h->denied.keys, keys.data(), keys.size() * sizeof(u64), cudaMemcpyHostToDevice));
        CK(cudaMemcpy(h->denied.counts, cnts.data(), cnts.size() * sizeof(u64), cudaMemcpyHostToDevice));
    }
    return GCRA_OK;
}

int32_t gcra_sync(gcra_engine *h) {
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->in_stream));
    CK(cudaStreamSynchronize(h->front_stream[0]));
    CK(cudaStreamSynchronize(h->back_stream));
    CK(cudaStreamSynchronize(h->tail_stream));
    CK(cudaStreamSynchronize(h->aux_stream));
    CK(cudaStreamSynchronize(h->aux2_stream));
    CK(cudaStreamSynchronize(h->stream));
    CK(cudaStreamSynchronize(h->out_stream));
    return GCRA_OK;
}

int32_t gcra_last_kernel_ms(gcra_engine *h, float out[4]) {
    if (!h->ev_valid) { h->err = "no timed batch yet"; return GCRA_INTERNAL; }
    CK(cudaEventSynchronize(h->ev[3]));
    CK(cudaEventElapsedTime(&out[0], h->ev[0], h->ev[3]));
    CK(cudaEventElapsedTime(&out[1], h->ev[0], h->ev[1]));
    CK(cudaEventElapsedTime(&out[2], h->ev[1], h->ev[2]));
    CK(cudaEventElapsedTime(&out[3], h->ev[2], h->ev[3]));
    return GCRA_OK;
}

int32_t gcra_last_kernel_ms_detail(gcra_engine *h, float out[7]) {
    if (!h->evd_valid) { h->err = "no timed index-order batch yet"; return GCRA_INTERNAL; }
    CK(cudaEventSynchronize(h->evd[7]));
    for (int i = 0; i < 7; i++) CK(cudaEventElapsedTime(&out[i], h->evd[i], h->evd[i + 1]));
    return GCRA_OK;
}

void gcra_debug_set(gcra_engine *h, uint32_t mask) { h->dbg = mask; }

int32_t gcra_last_sweep_ms(gcra_engine *h, float *ms) {
    if (!h->sweep_timed) { h->err = "no sweep yet"; return GCRA_INTERNAL; }
    CK(cudaEventSynchronize(h->ev_sweep[1]));
    CK(cudaEventElapsedTime(ms, h->ev_sweep[0], h->ev_sweep[1]));
    return GCRA_OK;
}

uint64_t gcra_launch_count(gcra_engine *h) { return h->launches; }

// ---- snapshot / restore (absent in the reference: its state is lost on restart; SURVEY 8f #4) -----------
namespace {
struct SnapshotHeader {
    char magic[8];
    uint32_t version, total_lines, nb_main, stash_slots;
    uint64_t capacity;
    uint64_t counters[C_COUNT];
    uint64_t hash_seed[2];           // (version 2) the identities in the table were made with this seed
};
const char SNAP_MAGIC[8] = {'G', 'C', 'R', 'A', 'B', '2', '0', '0'};
const size_t SNAP_CHUNK = 32u << 20;
}  // namespace

static int copy_to_file(gcra_engine *h, FILE *f, const void *dptr, size_t bytes, std::vector<char> &buf) {
    for (size_t off = 0; off < bytes; off += SNAP_CHUNK) {
        size_t m = std::min(SNAP_CHUNK, bytes - off);
        CK(cudaMemcpy(buf.data(), (const char *)dptr + off, m, cudaMemcpyDeviceToHost));
        if (fwrite(buf.data(), 1, m, f) != m) { h->err = "snapshot: short write"; return GCRA_INTERNAL; }
    }
    return GCRA_OK;
}

static int copy_from_file(gcra_engine *h, FILE *f, void *dptr, size_t bytes, std::vector<char> &buf) {
    for (size_t off = 0; off < bytes; off += SNAP_CHUNK) {
        size_t m = std::min(SNAP_CHUNK, bytes - off);
        if (fread(buf.data(), 1, m, f) != m) { h->err = "snapshot: short read"; return GCRA_INTERNAL; }
        CK(cudaMemcpy((char *)dptr + off, buf.data(), m, cudaMemcpyHostToDevice));
    }
    return GCRA_OK;
}

int32_t gcra_snapshot_save(gcra_engine *h, const char *path) {
    CK(cudaSetDevice(h->device));
    CK(cudaDeviceSynchronize());
    FILE *f = fopen(path, "wb");
    if (!f) { h->err = std::string("snapshot: cannot open ") + path; return GCRA_INTERNAL; }
    SnapshotHeader hd{};
    memcpy(hd.magic, SNAP_MAGIC, 8);
    hd.version = 2; hd.hash_seed[0] = h->hash_seed[0]; hd.hash_seed[1] = h->hash_seed[1]; hd.total_lines = h->total_lines; hd.nb_main = h->tab.nb_main; hd.stash_slots = h->tab.stash_slots;
    hd.capacity = h->capacity;
    int rc = GCRA_OK;
    if (cudaMemcpy(hd.counters, h->tab.counters, sizeof(hd.counters), cudaMemcpyDeviceToHost) != cudaSuccess ||
        fwrite(&hd, sizeof(hd), 1, f) != 1) { h->err = "snapshot: header"; rc = GCRA_INTERNAL; }
    std::vector<char> buf(SNAP_CHUNK);
    const size_t slots = (size_t)h->total_lines * 4;
    if (!rc) rc = copy_to_file(h, f, h->tab.keys, slots * sizeof(u64), buf);
    if (!rc) rc = copy_to_file(h, f, h->tab.state, slots * sizeof(TatOff), buf);
    if (!rc) rc = copy_to_file(h, f, h->tab.ei, slots * sizeof(i64), buf);
    if (fclose(f) != 0 && !rc) { h->err = "snapshot: close"; rc = GCRA_INTERNAL; }
    return rc;
}

int32_t gcra_snapshot_load(gcra_engine *h, const char *path) {
    CK(cudaSetDevice(h->device));
    CK(cudaDeviceSynchronize());
    FILE *f = fopen(path, "rb");
    if (!f) { h->err = std::string("snapshot: cannot open ") + path; return GCRA_INTERNAL; }
    SnapshotHeader hd{};
    if (fread(&hd, sizeof(hd), 1, f) != 1 || memcmp(hd.magic, SNAP_MAGIC, 8) != 0 || hd.version != 2) {
        fclose(f); h->err = "snapshot: bad header"; return GCRA_INTERNAL;
    }
    int rc = GCRA_OK;
    if (hd.total_lines != h->total_lines || hd.nb_main != h->tab.nb_main || hd.stash_slots != h->tab.stash_slots) {
        // other geometry: replace the table by one of the snapshot's shape
        uint32_t tl, nb, ss;
        table_geometry(hd.capacity, h->tight, tl, nb, ss);
        if (tl != hd.total_lines || nb != hd.nb_main || ss != hd.stash_slots) {
            fclose(f); h->err = "snapshot: geometry not reproducible with this build/flags"; return GCRA_INTERNAL;
        }
        Table nt{};
        uint32_t nl = 0;
        rc = alloc_table(h, hd.capacity, nt, nl, h->tab.counters);
        if (rc) { fclose(f); return rc; }
        CK(cudaStreamSynchronize(h->stream));
        cudaFree(h->tab.keys); cudaFree(h->tab.state); cudaFree(h->tab.ei); cudaFree(h->tab.mark);
        h->tab = nt; h->total_lines = nl; h->capacity = hd.capacity;
    }
    std::vector<char> buf(SNAP_CHUNK);
    const size_t slots = (size_t)h->total_lines * 4;
    if (!rc) rc = copy_from_file(h, f, h->tab.keys, slots * sizeof(u64), buf);
    if (!rc) rc = copy_from_file(h, f, h->tab.state, slots * sizeof(TatOff), buf);
    if (!rc) rc = copy_from_file(h, f, h->tab.ei, slots * sizeof(i64), buf);
    fclose(f);
    if (rc) return rc;
    CK(cudaMemcpy(h->tab.counters, hd.counters, sizeof(hd.counters), cudaMemcpyHostToDevice));
    h->hash_seed[0] = hd.hash_seed[0];
    h->hash_seed[1] = hd.hash_seed[1];
    h->occupied_ub = hd.counters[C_OCCUPIED];
    h->seen_allowed = hd.counters[C_ALLOWED];
    h->seen_expired_hits = hd.counters[C_EXPIRED_HITS];
    for (int i = 0; i < gcra_engine::N_SNAP; i++) h->snap_used[i] = false;
    return GCRA_OK;
}


// ---- multi-GPU: the whole sharded tick in native code (one call per tick) ------------------------------
#define NK(call)                                                                              \
    do {                                                                                      \
        int r_ = (call);                                                                      \
        if (r_ != 0) {                                                                        \
            h->err = std::string(#call) + ": " + (nccl_rt::g_api.GetErrorString ? nccl_rt::g_api.GetErrorString(r_) : "nccl error"); \
            return GCRA_INTERNAL;                                                             \
        }                                                                                     \
    } while (0)

int32_t gcra_shard_unique_ids(void *out_3x128) {
    if (!nccl_rt::load()) return GCRA_INTERNAL;
    for (int i = 0; i < 3; i++)
        if (nccl_rt::g_api.GetUniqueId((nccl_rt::UniqueId *)((char *)out_3x128 + 128 * i)) != 0) return GCRA_INTERNAL;
    return GCRA_OK;
}

int32_t gcra_shard_init(gcra_engine *h, int32_t rank, int32_t world, const void *ids_3x128, uint32_t max_rows) {
    CK(cudaSetDevice(h->device));
    if (h->shard) { h->err = "shard already initialised"; return GCRA_INTERNAL; }
    if (world < 1 || world > ROUTE_MAX_SHARDS || rank < 0 || rank >= world) { h->err = "bad rank / world"; return GCRA_INTERNAL; }
    if (max_rows == 0 || max_rows > h->max_batch) { h->err = "max_rows must be in 1..max_batch"; return GCRA_INTERNAL; }
    if (!nccl_rt::load()) { h->err = "libnccl.so.2 not found"; return GCRA_INTERNAL; }
    Shard *sh = new Shard();
    sh->rank = rank; sh->world = world; sh->max_rows = max_rows;
    const nccl_rt::UniqueId *ids = (const nccl_rt::UniqueId *)ids_3x128;
    // one communicator per stage: NCCL runs the operations of ONE communicator in issue order
    NK(nccl_rt::g_api.CommInitRank(&sh->comm_counts, world, ids[0], rank));
    NK(nccl_rt::g_api.CommInitRank(&sh->comm_req, world, ids[1], rank));
    NK(nccl_rt::g_api.CommInitRank(&sh->comm_res, world, ids[2], rank));
    CK(cudaStreamCreateWithFlags(&sh->s_part, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&sh->s_route, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&sh->s_return, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&sh->ev_tmp, cudaEventDisableTiming));
    for (auto &sl : sh->slots) {
        CK(cudaMalloc(&sl.routed, (size_t)max_rows * sizeof(gcra_request)));
        // a shard can receive up to world x max_rows rows in one tick (every rank's whole tick): sized for that, so
        // no rank ever has to bail out of a tick its peers have already posted their sends for
        CK(cudaMalloc(&sl.recv_req, (size_t)world * max_rows * sizeof(gcra_request)));
        CK(cudaMalloc(&sl.recv_res, (size_t)world * max_rows * sizeof(gcra_result)));
        CK(cudaMalloc(&sl.back_res, (size_t)max_rows * sizeof(gcra_result)));
        CK(cudaMalloc(&sl.src_index, (size_t)max_rows * sizeof(u32)));
        CK(cudaMalloc(&sl.counts_dev, 2 * ROUTE_MAX_SHARDS * sizeof(u32)));
        CK(cudaMallocHost(&sl.counts_host, 2 * ROUTE_MAX_SHARDS * sizeof(u32)));
        CK(cudaEventCreateWithFlags(&sl.ev_ready, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&sl.ev_counts, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&sl.ev_routed, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&sl.ev_done, cudaEventDisableTiming));
        sl.send.resize(world); sl.recv.resize(world); sl.send_off.resize(world); sl.recv_off.resize(world);
    }
    h->shard = sh;
    return GCRA_OK;
}

// stages 3+4 of a tick: the engine's kernels (pipelined inside the engine) and the way back
static int shard_issue_decide_return(gcra_engine *h) {
    Shard *sh = h->shard;
    if (sh->pending < 0) return GCRA_OK;
    ShardSlot &sl = sh->slots[sh->pending];
    sh->pending = -1;
    const int W = sh->world;
    cudaEvent_t done = nullptr;
    // (more rows than one engine batch carries: several batches, cut anywhere -- the order is kept)
    for (uint32_t a = 0; a < sl.n_recv || a == 0; a += h->max_batch) {
        const uint32_t m = std::min<uint32_t>(sl.n_recv - a, h->max_batch);
        cudaEvent_t dn = nullptr;
        RC(launch_pipelined(h, m, sl.recv_req + a, false, 0, sl.recv_res + a, sl.ev_routed, &dn));
        if (dn) { done = dn; CK(cudaStreamWaitEvent(sh->s_return, dn, 0)); }
        if (sl.n_recv == 0) break;
    }
    if (!done) CK(cudaStreamWaitEvent(sh->s_return, sl.ev_routed, 0));
    NK(nccl_rt::g_api.GroupStart());
    for (int p = 0; p < W; p++) {
        // results of the rows peer p sent me go back to p; my own rows' results arrive in partition order
        NK(nccl_rt::g_api.Send(sl.recv_res + sl.recv_off[p], sl.recv[p] * sizeof(gcra_result), nccl_rt::kUint8, p, sh->comm_res, sh->s_return));
        NK(nccl_rt::g_api.Recv(sl.back_res + sl.send_off[p], sl.send[p] * sizeof(gcra_result), nccl_rt::kUint8, p, sh->comm_res, sh->s_return));
    }
    NK(nccl_rt::g_api.GroupEnd());
    if (sl.n) {
        route_unpermute_kernel<<<(sl.n + TILE_THREADS - 1) / TILE_THREADS, TILE_THREADS, 0, sh->s_return>>>(
            sl.back_res, sl.src_index, sl.n, sl.d_res_user);
        h->launches++;
    }
    CK(cudaEventRecord(sl.ev_done, sh->s_return));
    CK(cudaGetLastError());
    return GCRA_OK;
}

int32_t gcra_shard_submit(gcra_engine *h, uint64_t n64, const gcra_request *d_req, gcra_result *d_res, void *ready_stream) {
    CK(cudaSetDevice(h->device));
    Shard *sh = h->shard;
    if (!sh) { h->err = "gcra_shard_init first"; return GCRA_INTERNAL; }
    if (n64 > sh->max_rows) { h->err = "tick larger than max_rows"; return GCRA_INTERNAL; }
    const uint32_t n = (uint32_t)n64;
    const int W = sh->world;
    const int k = (int)(sh->next++ % Shard::DEPTH);
    ShardSlot &sl = sh->slots[k];
    if ((int)sh->pending == k) RC(shard_issue_decide_return(h));
    if (sl.used) CK(cudaStreamWaitEvent(sh->s_part, sl.ev_done, 0));     // the slot's buffers are free again
    sl.used = true; sl.n = n; sl.d_res_user = d_res;
    if (ready_stream) {
        CK(cudaEventRecord(sl.ev_ready, (cudaStream_t)ready_stream));
        CK(cudaStreamWaitEvent(sh->s_part, sl.ev_ready, 0));
    }
    // stage 1: stable partition by owner + count exchange
    if (n) {
        uint32_t tiles = (n + TILE_THREADS - 1) / TILE_THREADS;
        route_count_kernel<<<tiles, TILE_THREADS, 0, sh->s_part>>>(d_req, n, (u32)W, tiles, h->route_counts);
        route_scan_kernel<<<1, TILE_THREADS, 0, sh->s_part>>>(h->route_counts, (u32)W, tiles, sl.counts_dev);
        route_scatter_kernel<<<tiles, TILE_THREADS, 0, sh->s_part>>>(d_req, n, (u32)W, tiles, h->route_counts, sl.routed, sl.src_index);
        h->launches += 3;
    } else {
        CK(cudaMemsetAsync(sl.counts_dev, 0, W * sizeof(u32), sh->s_part));
    }
    NK(nccl_rt::g_api.GroupStart());
    for (int p = 0; p < W; p++) {
        NK(nccl_rt::g_api.Send(sl.counts_dev + p, 1, nccl_rt::kUint32, p, sh->comm_counts, sh->s_part));
        NK(nccl_rt::g_api.Recv(sl.counts_dev + W + p, 1, nccl_rt::kUint32, p, sh->comm_counts, sh->s_part));
    }
    NK(nccl_rt::g_api.GroupEnd());
    CK(cudaMemcpyAsync(sl.counts_host, sl.counts_dev, 2 * W * sizeof(u32), cudaMemcpyDeviceToHost, sh->s_part));
    CK(cudaEventRecord(sl.ev_counts, sh->s_part));
    // while this runs, enqueue the previous tick's engine kernels and its way back
    RC(shard_issue_decide_return(h));
    // stage 2: request all-to-all on its own stream (the partition + count exchange of the NEXT tick overlap
    // it); the counts are the only thing the host waits for
    CK(cudaEventSynchronize(sl.ev_counts));
    CK(cudaStreamWaitEvent(sh->s_route, sl.ev_counts, 0));
    size_t so = 0, ro = 0;
    for (int p = 0; p < W; p++) {
        sl.send[p] = sl.counts_host[p]; sl.recv[p] = sl.counts_host[W + p];
        sl.send_off[p] = so; sl.recv_off[p] = ro;
        so += sl.send[p]; ro += sl.recv[p];
    }
    sl.n_recv = (uint32_t)ro;             // <= world x max_rows, which the buffers hold
    NK(nccl_rt::g_api.GroupStart());
    for (int p = 0; p < W; p++) {
        NK(nccl_rt::g_api.Send(sl.routed + sl.send_off[p], sl.send[p] * sizeof(gcra_request), nccl_rt::kUint8, p, sh->comm_req, sh->s_route));
        NK(nccl_rt::g_api.Recv(sl.recv_req + sl.recv_off[p], sl.recv[p] * sizeof(gcra_request), nccl_rt::kUint8, p, sh->comm_req, sh->s_route));
    }
    NK(nccl_rt::g_api.GroupEnd());
    CK(cudaEventRecord(sl.ev_routed, sh->s_route));
    CK(cudaGetLastError());
    sh->pending = k;
    return GCRA_OK;
}

// make `stream` wait for the results of the tick submitted `ticks_back` submissions ago (0 = the latest);
// only the last DEPTH-1 ticks can be addressed
int32_t gcra_shard_wait_tick(gcra_engine *h, uint32_t ticks_back, void *stream) {
    CK(cudaSetDevice(h->device));
    Shard *sh = h->shard;
    if (!sh || ticks_back >= (uint32_t)Shard::DEPTH - 1 || ticks_back >= sh->next) { h->err = "bad tick"; return GCRA_INTERNAL; }
    const int k = (int)((sh->next - 1 - ticks_back) % Shard::DEPTH);
    if (sh->pending == k) RC(shard_issue_decide_return(h));
    if (stream) CK(cudaStreamWaitEvent((cudaStream_t)stream, sh->slots[k].ev_done, 0));
    else CK(cudaEventSynchronize(sh->slots[k].ev_done));
    return GCRA_OK;
}

int32_t gcra_shard_join(gcra_engine *h, void *stream) {
    CK(cudaSetDevice(h->device));
    Shard *sh = h->shard;
    if (!sh) { h->err = "gcra_shard_init first"; return GCRA_INTERNAL; }
    RC(shard_issue_decide_return(h));
    CK(cudaEventRecord(sh->ev_tmp, sh->s_return));
    if (stream) CK(cudaStreamWaitEvent((cudaStream_t)stream, sh->ev_tmp, 0));
    else CK(cudaEventSynchronize(sh->ev_tmp));
    return GCRA_OK;
}


// ---- multi-GPU over NVLink peer memory: the whole sharded tick without NCCL and without a host sync ------------
static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

int32_t gcra_p2p_prepare(gcra_engine *h, int32_t rank, int32_t world, uint32_t cap_rows, void *ipc_handle_out_64,
                         void **window_out) {
    CK(cudaSetDevice(h->device));
    if (h->p2p) { h->err = "p2p already prepared"; return GCRA_INTERNAL; }
    if (world < 1 || world > P2P_MAX_WORLD || rank < 0 || rank >= world) { h->err = "bad rank / world"; return GCRA_INTERNAL; }
    if (cap_rows == 0 || cap_rows > (1u << 24)) { h->err = "cap_rows must be in 1..2^24"; return GCRA_INTERNAL; }
    P2P *p = new P2P();
    p->rank = rank; p->world = world;
    p->cap_shift = std::max<uint32_t>(ceil_log2(cap_rows), 10);      // whole resolve tiles per segment
    p->cap = 1u << p->cap_shift;
    if (((uint64_t)world << p->cap_shift) >= (1ULL << 31)) { delete p; h->err = "world * cap_rows too large"; return GCRA_INTERNAL; }
    const size_t seg_rows = (size_t)P2P_DEPTH * world * p->cap;
    p->inbox_off = align_up(sizeof(P2PHeader), 256);
    p->outbox_off = align_up(p->inbox_off + seg_rows * sizeof(gcra_request), 256);
    p->window_bytes = align_up(p->outbox_off + seg_rows * sizeof(gcra_result), 256);
    CK(cudaMalloc(&p->window, p->window_bytes));
    CK(cudaMemset(p->window, 0, p->inbox_off));
    if (ipc_handle_out_64) {
        cudaIpcMemHandle_t hd;
        CK(cudaIpcGetMemHandle(&hd, p->window));
        static_assert(sizeof(hd) == 64, "cudaIpcMemHandle_t is 64 bytes");
        memcpy(ipc_handle_out_64, &hd, 64);
    }
    if (window_out) *window_out = p->window;
    CK(cudaStreamCreateWithFlags(&p->s_part, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&p->s_wait, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&p->s_sig, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&p->s_return, cudaStreamNonBlocking));
    for (auto &e : p->ev_t) CK(cudaEventCreate(&e));
    CK(cudaMalloc(&p->peers_dev, sizeof(P2PPeers)));
    CK(cudaMalloc(&p->tile_counts, (size_t)ROUTE_MAX_SHARDS * ((p->cap + TILE_THREADS - 1) / TILE_THREADS) * sizeof(u32)));
    for (auto &sl : p->slots) {
        CK(cudaMalloc(&sl.res_loc, (size_t)p->cap * sizeof(u32)));
        CK(cudaMalloc(&sl.counts_dev, P2P_MAX_WORLD * sizeof(u32)));
        CK(cudaMalloc(&sl.segs_dev, P2P_MAX_WORLD * sizeof(SegDesc)));
        CK(cudaEventCreateWithFlags(&sl.ev_ready, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&sl.ev_wait, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&sl.ev_done, cudaEventDisableTiming));
    }
    // the engine's per-row buffers now span the row-id space of a whole inbox slot
    CK(cudaDeviceSynchronize());
    for (auto &sc : h->scr) RC(alloc_index_scratch(h, sc, (uint32_t)world << p->cap_shift));
    h->p2p = p;
    return GCRA_OK;
}

// every rank's window: `ipc_handles` (world x 64 bytes, other processes) or `windows` (world pointers valid in THIS
// process: engines that share a process, e.g. the single-GPU loop-back test)
int32_t gcra_p2p_connect(gcra_engine *h, const void *ipc_handles, void *const *windows) {
    CK(cudaSetDevice(h->device));
    P2P *p = h->p2p;
    if (!p) { h->err = "gcra_p2p_prepare first"; return GCRA_INTERNAL; }
    if (!ipc_handles && !windows) { h->err = "need ipc handles or window pointers"; return GCRA_INTERNAL; }
    P2PPeers peers{};
    for (int r = 0; r < p->world; r++) {
        void *base = nullptr;
        if (r == p->rank) base = p->window;
        else if (windows) base = windows[r];
        else {
            cudaIpcMemHandle_t hd;
            memcpy(&hd, (const char *)ipc_handles + 64 * r, 64);
            CK(cudaIpcOpenMemHandle(&base, hd, cudaIpcMemLazyEnablePeerAccess));
            p->opened[r] = true;
        }
        p->peer_base[r] = base;
        peers.hdr[r] = (P2PHeader *)base;
        peers.inbox[r] = (unsigned char *)base + p->inbox_off;
        peers.outbox[r] = (unsigned char *)base + p->outbox_off;
    }
    CK(cudaMemcpy(p->peers_dev, &peers, sizeof(peers), cudaMemcpyHostToDevice));
    for (int d = 0; d < P2P_DEPTH; d++) {
        SegDesc segs[P2P_MAX_WORLD] = {};
        for (int r = 0; r < p->world; r++) {
            // segment r of MY inbox slot d holds sender r's rows; their results go to slot d, segment `rank` of
            // sender r's outbox
            segs[r].req = peers.inbox[p->rank] + (((size_t)d * p->world + r) << p->cap_shift) * sizeof(gcra_request);
            segs[r].res = (gcra_result *)(peers.outbox[r] + (((size_t)d * p->world + p->rank) << p->cap_shift) * sizeof(gcra_result));
        }
        CK(cudaMemcpy(p->slots[d].segs_dev, segs, sizeof(segs), cudaMemcpyHostToDevice));
    }
    p->connected = true;
    return GCRA_OK;
}

// first half of a tick: the sender's side (partition + transfer + flags)
int32_t gcra_p2p_submit_route(gcra_engine *h, uint64_t n64, const gcra_request *d_req, void *ready_stream) {
    CK(cudaSetDevice(h->device));
    P2P *p = h->p2p;
    if (!p || !p->connected) { h->err = "gcra_p2p_prepare / gcra_p2p_connect first"; return GCRA_INTERNAL; }
    if (p->routed_pending) { h->err = "gcra_p2p_submit_finish the previous tick first"; return GCRA_INTERNAL; }
    if (n64 > p->cap) { h->err = "tick larger than cap_rows"; return GCRA_INTERNAL; }
    const uint32_t n = (uint32_t)n64;
    const uint32_t W = (uint32_t)p->world, me = (uint32_t)p->rank;
    const uint64_t tick = ++p->next_tick;
    const uint32_t d = (uint32_t)((tick - 1) % P2P_DEPTH);
    P2PSlot &sl = p->slots[d];
    // slot d again: its previous tick has been un-permuted here, i.e. every owner is through with my rows of that
    // tick and with my outbox slot
    if (sl.used) CK(cudaStreamWaitEvent(p->s_part, sl.ev_done, 0));
    sl.used = true; sl.n = n;
    if (ready_stream) {
        CK(cudaEventRecord(sl.ev_ready, (cudaStream_t)ready_stream));
        CK(cudaStreamWaitEvent(p->s_part, sl.ev_ready, 0));
    }
    // stable partition by owner, rows stored straight into the owners' inboxes, then the flags
    const uint32_t tiles = (n + TILE_THREADS - 1) / TILE_THREADS;
    if (p->timed) CK(cudaEventRecord(p->ev_t[0], p->s_part));
    if (n) {
        route_count_kernel<<<tiles, TILE_THREADS, 0, p->s_part>>>(d_req, n, W, tiles, p->tile_counts);
        p2p_scan_kernel<<<W, TILE_THREADS, 0, p->s_part>>>(p->tile_counts, tiles, sl.counts_dev);
        p2p_scatter_kernel<<<tiles, TILE_THREADS, 0, p->s_part>>>(d_req, n, W, me, d, p->cap_shift, tiles, p->tile_counts,
                                                                 p->peers_dev, sl.res_loc);
        h->launches += 3;
    } else {
        CK(cudaMemsetAsync(sl.counts_dev, 0, W * sizeof(u32), p->s_part));
    }
    p2p_signal_req_kernel<<<1, 32, 0, p->s_part>>>(p->peers_dev, sl.counts_dev, W, me, d, tick);
    if (p->timed) CK(cudaEventRecord(p->ev_t[1], p->s_part));
    h->launches++;
    CK(cudaGetLastError());
    p->routed_pending = true;
    return GCRA_OK;
}

// second half: the owner's side (wait for every sender, decide, results into the senders' outboxes, flags) and the
// way back (wait for every owner, results into input order)
int32_t gcra_p2p_submit_finish(gcra_engine *h, gcra_result *d_res) {
    CK(cudaSetDevice(h->device));
    P2P *p = h->p2p;
    if (!p || !p->routed_pending) { h->err = "gcra_p2p_submit_route first"; return GCRA_INTERNAL; }
    p->routed_pending = false;
    const uint32_t W = (uint32_t)p->world, me = (uint32_t)p->rank;
    const uint64_t tick = p->next_tick;
    const uint32_t d = (uint32_t)((tick - 1) % P2P_DEPTH);
    P2PSlot &sl = p->slots[d];
    P2PHeader *hdr = (P2PHeader *)p->window;
    // owner: wait for every sender's rows of this tick, then the engine over the inbox slot as one batch of W
    // segments (row counts in the header); its kernels store the results into the senders' outboxes
    p2p_wait_kernel<<<1, 32, 0, p->s_wait>>>(hdr, 0, W, tick);
    CK(cudaEventRecord(sl.ev_wait, p->s_wait));
    BatchView v{};
    v.req0 = nullptr; v.res0 = nullptr;
    v.segs = sl.segs_dev;
    v.dev_counts = &hdr->counts[d][0];
    v.n = 0;
    v.nseg = W;
    v.cap_shift = p->cap_shift;
    cudaEvent_t done = nullptr;
    // Room in the table for the keys this tick may insert.  How many rows arrive is only known on the device; with a
    // hash-sharded key space it is about what this rank submitted itself, so 1.25 x that (+ slack) is reserved -- a
    // reservation of the full inbox would make the host wait for the device every tick.  Should a tick bring more
    // NEW keys than the table has room for, the surplus rows are answered with GCRA_INTERNAL ("table full"), as
    // find_or_claim always does; the next tick's check then sees the real occupancy and grows the table.
    const uint32_t n_rows = (uint32_t)std::min<uint64_t>((uint64_t)sl.n + sl.n / 4 + 4096, std::min<uint64_t>((uint64_t)W << p->cap_shift, h->max_batch));
    if (p->timed) CK(cudaEventRecord(p->ev_t[2], p->s_wait));
    RC(launch_pipelined_view(h, v, n_rows, false, 0, sl.ev_wait, &done));
    CK(cudaStreamWaitEvent(p->s_sig, done, 0));
    if (p->timed) CK(cudaEventRecord(p->ev_t[3], p->s_sig));
    p2p_signal_res_kernel<<<1, 32, 0, p->s_sig>>>(p->peers_dev, W, me, tick);
    // sender again: every owner's results of this tick are in my outbox -> input order, into the caller's buffer
    p2p_wait_kernel<<<1, 32, 0, p->s_return>>>(hdr, 1, W, tick);
    if (p->timed) CK(cudaEventRecord(p->ev_t[4], p->s_return));
    if (sl.n) {
        const uint32_t tiles = (sl.n + TILE_THREADS - 1) / TILE_THREADS;
        p2p_unpermute_kernel<<<tiles, TILE_THREADS, 0, p->s_return>>>((const unsigned char *)p->window + p->outbox_off, sl.res_loc,
                                                                     sl.n, W, d, p->cap_shift, d_res);
        h->launches++;
    }
    CK(cudaEventRecord(sl.ev_done, p->s_return));
    if (p->timed) { CK(cudaEventRecord(p->ev_t[5], p->s_return)); p->timed_valid = true; }
    h->launches += 3;
    CK(cudaGetLastError());
    return GCRA_OK;
}

// stage times (ms) of the most recent tick submitted with timing on (gcra_p2p_set_timing(h, 1)) -- meaningful when
// ticks are run one at a time (submit, join): [0] partition + transfer + flags, [1] until every sender's rows are
// here (includes the other ranks' skew), [2] the engine over the inbox, [3] until every owner's results are here,
// [4] un-permutation
int32_t gcra_p2p_set_timing(gcra_engine *h, int32_t on) {
    P2P *p = h->p2p;
    if (!p) { h->err = "gcra_p2p_prepare first"; return GCRA_INTERNAL; }
    p->timed = on != 0;
    return GCRA_OK;
}

int32_t gcra_p2p_last_tick_ms(gcra_engine *h, float out[5]) {
    CK(cudaSetDevice(h->device));
    P2P *p = h->p2p;
    if (!p || !p->timed_valid) { h->err = "no timed tick yet"; return GCRA_INTERNAL; }
    CK(cudaEventSynchronize(p->ev_t[5]));
    for (int i = 0; i < 5; i++) CK(cudaEventElapsedTime(&out[i], p->ev_t[i], p->ev_t[i + 1]));
    return GCRA_OK;
}

int32_t gcra_p2p_submit(gcra_engine *h, uint64_t n, const gcra_request *d_req, gcra_result *d_res, void *ready_stream) {
    RC(gcra_p2p_submit_route(h, n, d_req, ready_stream));
    return gcra_p2p_submit_finish(h, d_res);
}

// make `stream` wait for the results of the tick submitted `ticks_back` submissions ago (0 = the latest, < DEPTH)
int32_t gcra_p2p_wait_tick(gcra_engine *h, uint32_t ticks_back, void *stream) {
    CK(cudaSetDevice(h->device));
    P2P *p = h->p2p;
    if (!p || ticks_back >= (uint32_t)P2P_DEPTH || ticks_back >= p->next_tick) { h->err = "bad tick"; return GCRA_INTERNAL; }
    P2PSlot &sl = p->slots[(p->next_tick - 1 - ticks_back) % P2P_DEPTH];
    if (stream) CK(cudaStreamWaitEvent((cudaStream_t)stream, sl.ev_done, 0));
    else CK(cudaEventSynchronize(sl.ev_done));
    return GCRA_OK;
}

int32_t gcra_p2p_join(gcra_engine *h, void *stream) {
    CK(cudaSetDevice(h->device));
    P2P *p = h->p2p;
    if (!p) { h->err = "gcra_p2p_prepare first"; return GCRA_INTERNAL; }
    for (auto &sl : p->slots) {
        if (!sl.used) continue;
        if (stream) CK(cudaStreamWaitEvent((cudaStream_t)stream, sl.ev_done, 0));
        else CK(cudaEventSynchronize(sl.ev_done));
    }
    return GCRA_OK;
}

// 1 when a wait on this rank gave up (a peer never delivered a tick): results since then are not to be trusted
int32_t gcra_p2p_error(gcra_engine *h, uint32_t *error) {
    CK(cudaSetDevice(h->device));
    P2P *p = h->p2p;
    if (!p) { h->err = "gcra_p2p_prepare first"; return GCRA_INTERNAL; }
    CK(cudaMemcpy(error, (const char *)p->window + offsetof(P2PHeader, error), sizeof(u32), cudaMemcpyDeviceToHost));
    return GCRA_OK;
}

// ---- routing -------------------------------------------------------------------------------------
uint32_t gcra_owner_of(uint64_t key_hash, uint32_t n_shards) { return owner_of(key_hash, n_shards); }

int32_t gcra_route_partition(gcra_engine *h, uint64_t n, const gcra_request *d_req, uint32_t n_shards,
                             gcra_request *d_out, uint32_t *d_src_index, uint32_t *d_counts, void *stream) {
    CK(cudaSetDevice(h->device));
    if (n_shards == 0 || n_shards > ROUTE_MAX_SHARDS || n > h->max_batch) { h->err = "bad shard count / batch size"; return GCRA_INTERNAL; }
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    if (n == 0) { CK(cudaMemsetAsync(d_counts, 0, n_shards * sizeof(u32), st)); return GCRA_OK; }
    uint32_t tiles = (uint32_t)((n + TILE_THREADS - 1) / TILE_THREADS);
    route_count_kernel<<<tiles, TILE_THREADS, 0, st>>>(d_req, (u32)n, n_shards, tiles, h->route_counts);
    route_scan_kernel<<<1, TILE_THREADS, 0, st>>>(h->route_counts, n_shards, tiles, d_counts);
    route_scatter_kernel<<<tiles, TILE_THREADS, 0, st>>>(d_req, (u32)n, n_shards, tiles, h->route_counts, d_out, d_src_index);
    h->launches += 3;
    CK(cudaGetLastError());
    return GCRA_OK;
}

int32_t gcra_route_unpermute(gcra_engine *h, uint64_t n, const gcra_result *d_res_routed, const uint32_t *d_src_index,
                             gcra_result *d_res, void *stream) {
    CK(cudaSetDevice(h->device));
    if (n == 0) return GCRA_OK;
    cudaStream_t st = stream ? (cudaStream_t)stream : h->stream;
    route_unpermute_kernel<<<(uint32_t)((n + TILE_THREADS - 1) / TILE_THREADS), TILE_THREADS, 0, st>>>(
        d_res_routed, d_src_index, (u32)n, d_res);
    h->launches++;
    CK(cudaGetLastError());
    return GCRA_OK;
}

}  // extern "C"

#include "gcra_actor.inc"
#include "gcra_resp.inc"
