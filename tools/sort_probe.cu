// sort_probe.cu -- times the engine's stable slot sort against the three-kernel LSD sort it replaced and against
// cub::DeviceRadixSort, on keys shaped like bench.py's: (slot << 32 | index), 2^20 keys, slot = the low 25 bits of
// the engine's hash of the Zipf-1.0 key ids of one tick (tests/traces.py config2, written by
// tools/sort_probe_keys.py).  The 8 MB of keys stay in L2 between repetitions, as they do in the pipeline.
//
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o sort_probe tools/sort_probe.cu
//   python tools/sort_probe_keys.py keys.bin && ./sort_probe keys.bin
//
// Prints one JSON line: microseconds per sort (CUDA events over >= 200 repetitions) of each sort, whether every
// result equals a host stable sort, and the engine sort at the residue sizes of the index-order pipeline (device
// count, launched for 2^20 keys).
#include <cuda_runtime.h>
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "../throttlecrab_b200/csrc/gcra_kernels.cuh"

using namespace gcra;

#define CK(x)                                                                                       \
    do {                                                                                            \
        cudaError_t e_ = (x);                                                                       \
        if (e_ != cudaSuccess) { fprintf(stderr, "%s:%d %s\n", __FILE__, __LINE__, cudaGetErrorString(e_)); exit(1); } \
    } while (0)

// ---- the three-kernel LSD sort the engine used before (per pass: histogram, one CTA per digit row scan, scatter)
namespace old_sort {
constexpr int ITEMS = 4, TILE = TILE_THREADS * ITEMS;

__global__ void __launch_bounds__(TILE_THREADS) hist_kernel(const u64 *in, u32 n, u32 shift, u32 bits, u32 *hist) {
    __shared__ u32 h[SORT_MAX_DIGITS];
    const u32 num_tiles = (n + TILE - 1) / TILE, nd = 1u << bits, mask = nd - 1;
    for (u32 tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        for (u32 d = threadIdx.x; d < nd; d += TILE_THREADS) h[d] = 0;
        __syncthreads();
        for (int k = 0; k < ITEMS; k++) {
            u32 i = tile * TILE + k * TILE_THREADS + threadIdx.x;
            if (i < n) atomicAdd(&h[(u32)(in[i] >> shift) & mask], 1u);
        }
        __syncthreads();
        for (u32 d = threadIdx.x; d < nd; d += TILE_THREADS) hist[(size_t)d * num_tiles + tile] = h[d];
        __syncthreads();
    }
}

__global__ void __launch_bounds__(TILE_THREADS) rowscan_kernel(u32 *hist, u32 n, u32 *tot) {
    __shared__ u32 part[TILE_THREADS / 32];
    const u32 num_tiles = (n + TILE - 1) / TILE;
    u32 *row = hist + (size_t)blockIdx.x * num_tiles;
    const u32 per = (num_tiles + TILE_THREADS - 1) / TILE_THREADS;
    const u32 lo = min(threadIdx.x * per, num_tiles), hi = min(lo + per, num_tiles);
    u32 s = 0;
    for (u32 i = lo; i < hi; i++) s += row[i];
    u32 total;
    u32 acc = block_exclusive_scan(s, part, &total);
    for (u32 i = lo; i < hi; i++) { u32 v = row[i]; row[i] = acc; acc += v; }
    if (threadIdx.x == 0) tot[blockIdx.x] = total;
}

__global__ void __launch_bounds__(TILE_THREADS)
scatter_kernel(const u64 *in, u64 *outk, u32 n, u32 shift, u32 bits, const u32 *hist, const u32 *tot) {
    constexpr int NW = TILE_THREADS / 32;
    __shared__ u32 cnt[NW][SORT_MAX_DIGITS], gbase[SORT_MAX_DIGITS], part[NW];
    const u32 num_tiles = (n + TILE - 1) / TILE;
    if (blockIdx.x >= num_tiles) return;
    const u32 nd = 1u << bits, mask = nd - 1, w = threadIdx.x >> 5, lane = threadIdx.x & 31, lt = (1u << lane) - 1;
    const u32 d0 = 2 * threadIdx.x, d1 = d0 + 1;
    const u32 t0 = d0 < nd ? tot[d0] : 0, t1 = d1 < nd ? tot[d1] : 0;
    u32 total;
    const u32 ex = block_exclusive_scan(t0 + t1, part, &total);
    for (u32 tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        for (u32 d = threadIdx.x; d < nd; d += TILE_THREADS)
            for (int x = 0; x < NW; x++) cnt[x][d] = 0;
        if (d0 < nd) gbase[d0] = ex + hist[(size_t)d0 * num_tiles + tile];
        if (d1 < nd) gbase[d1] = ex + t0 + hist[(size_t)d1 * num_tiles + tile];
        __syncthreads();
        const u32 base = tile * TILE + w * (32 * ITEMS);
        u64 key[ITEMS];
        u32 dig[ITEMS], rank[ITEMS];
        for (int k = 0; k < ITEMS; k++) {
            u32 i = base + k * 32 + lane;
            bool valid = i < n;
            key[k] = valid ? in[i] : 0;
            dig[k] = (u32)(key[k] >> shift) & mask;
            u32 peers = __match_any_sync(0xffffffffu, valid ? dig[k] : (0x80000000u | lane));
            u32 before = valid ? cnt[w][dig[k]] : 0;
            rank[k] = before + __popc(peers & lt);
            __syncwarp();
            if (valid && (peers & lt) == 0) cnt[w][dig[k]] = before + __popc(peers);
            __syncwarp();
        }
        __syncthreads();
        for (u32 d = threadIdx.x; d < nd; d += TILE_THREADS) {
            u32 acc = 0;
            for (int x = 0; x < NW; x++) { u32 v = cnt[x][d]; cnt[x][d] = acc; acc += v; }
        }
        __syncthreads();
        for (int k = 0; k < ITEMS; k++) {
            u32 i = base + k * 32 + lane;
            if (i < n) outk[gbase[dig[k]] + cnt[w][dig[k]] + rank[k]] = key[k];
        }
        __syncthreads();
    }
}
}  // namespace old_sort

struct Bufs {
    u64 *a, *b;
    u32 *hist, *tot;                  // old sort
    u64 *status;                      // one-sweep sort
    u32 *dtot, *ticket, *n_dev;
    u32 tickets = 0, seq = 0, parity = 0;
};

static const u32 BITS = 25;
static const u32 PASSES = (BITS + SORT_MAX_BITS - 1) / SORT_MAX_BITS;

static u64 *run_old(Bufs &B, u32 n) {
    const u32 tiles = (n + old_sort::TILE - 1) / old_sort::TILE;
    u64 *src = B.a, *dst = B.b;
    u32 shift = 32;
    for (u32 p = 0; p < PASSES; p++) {
        const u32 pb = sort_pass_bits(BITS, PASSES, p);
        old_sort::hist_kernel<<<tiles, TILE_THREADS>>>(src, n, shift, pb, B.hist);
        old_sort::rowscan_kernel<<<1u << pb, TILE_THREADS>>>(B.hist, n, B.tot);
        old_sort::scatter_kernel<<<tiles, TILE_THREADS>>>(src, dst, n, shift, pb, B.hist, B.tot);
        std::swap(src, dst);
        shift += pb;
    }
    return src;
}

// the engine's launch sequence (gcra_b200.cu enqueue_sort); n_dev != null: device count, launched for n_max keys
static u64 *run_onesweep(Bufs &B, u32 n_max, const u32 *n_dev) {
    const u32 tiles = (n_max + SORT_TILE - 1) / SORT_TILE;
    u32 *tot = B.dtot + B.parity * SORT_MAX_PASSES * SORT_MAX_DIGITS;
    u32 *clear = B.dtot + (B.parity ^ 1) * SORT_MAX_PASSES * SORT_MAX_DIGITS;
    B.parity ^= 1;
    const u32 hgrid = std::min<u32>((n_max + SORT_HIST_KEYS - 1) / SORT_HIST_KEYS, 4 * 148);
    sort_digits_hist_kernel<<<hgrid, TILE_THREADS>>>(B.a, n_max, n_dev, BITS, PASSES, tot, clear);
    u64 *src = B.a, *dst = B.b;
    u32 shift = 32;
    for (u32 p = 0; p < PASSES; p++) {
        const u32 pb = sort_pass_bits(BITS, PASSES, p);
        sort_onesweep_kernel<<<tiles, TILE_THREADS>>>(src, dst, n_max, n_dev, shift, pb, tot + p * SORT_MAX_DIGITS,
                                                      B.status, B.ticket, B.tickets, ++B.seq);
        B.tickets += tiles;
        std::swap(src, dst);
        shift += pb;
    }
    return src;
}

// keys: (slot << 32 | index); the sort is stable on the slot, so the expected result is a stable sort by slot
static bool check(const std::vector<u64> &keys, u32 n, const u64 *d_sorted) {
    std::vector<u64> want(keys.begin(), keys.begin() + n), got(n);
    std::stable_sort(want.begin(), want.end(), [](u64 x, u64 y) { return (x >> 32) < (y >> 32); });
    if (n) CK(cudaMemcpy(got.data(), d_sorted, (size_t)n * 8, cudaMemcpyDeviceToHost));
    return want == got;
}

template <typename F>
static double time_us(F f, int reps) {
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    for (int i = 0; i < 10; i++) f();
    CK(cudaEventRecord(e0));
    for (int i = 0; i < reps; i++) f();
    CK(cudaEventRecord(e1));
    CK(cudaEventSynchronize(e1));
    float ms = 0;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    CK(cudaGetLastError());
    return 1e3 * ms / reps;
}

int main(int argc, char **argv) {
    if (argc < 2) { fprintf(stderr, "usage: %s KEYS_FILE (raw little-endian u64 key hashes)\n", argv[0]); return 2; }
    FILE *f = fopen(argv[1], "rb");
    if (!f) { perror(argv[1]); return 2; }
    std::vector<u64> hashes;
    u64 x;
    while (fread(&x, 8, 1, f) == 1) hashes.push_back(x);
    fclose(f);
    const u32 N = (u32)hashes.size();
    std::vector<u64> keys(N);
    for (u32 i = 0; i < N; i++) keys[i] = ((hashes[i] & ((1ULL << BITS) - 1)) << 32) | i;
    const int REPS = 200;

    Bufs B{};
    const u32 tiles_max = (N + SORT_TILE - 1) / SORT_TILE;
    CK(cudaMalloc(&B.a, (size_t)N * 8));
    CK(cudaMalloc(&B.b, (size_t)N * 8));
    CK(cudaMalloc(&B.hist, (size_t)SORT_MAX_DIGITS * ((N + old_sort::TILE - 1) / old_sort::TILE) * 4));
    CK(cudaMalloc(&B.tot, SORT_MAX_DIGITS * 4));
    CK(cudaMalloc(&B.status, (size_t)SORT_MAX_DIGITS * tiles_max * 8));
    CK(cudaMemset(B.status, 0, (size_t)SORT_MAX_DIGITS * tiles_max * 8));
    CK(cudaMalloc(&B.dtot, (2 * SORT_MAX_PASSES * SORT_MAX_DIGITS + 1) * 4));
    CK(cudaMemset(B.dtot, 0, (2 * SORT_MAX_PASSES * SORT_MAX_DIGITS + 1) * 4));
    B.ticket = B.dtot + 2 * SORT_MAX_PASSES * SORT_MAX_DIGITS;
    CK(cudaMalloc(&B.n_dev, 4));
    u64 *c_out = nullptr;
    void *c_tmp = nullptr;
    size_t c_bytes = 0;
    CK(cudaMalloc(&c_out, (size_t)N * 8));
    CK(cub::DeviceRadixSort::SortKeys(nullptr, c_bytes, B.a, c_out, (int)N, 32, 32 + BITS));
    CK(cudaMalloc(&c_tmp, c_bytes));

    // every sort reads B.a (the unsorted keys) and leaves it alone: the passes ping-pong A -> B -> A -> B, and
    // the keys are copied back in before each check
    auto load = [&](u32 n) { CK(cudaMemcpy(B.a, keys.data(), (size_t)n * 8, cudaMemcpyHostToDevice)); };
    load(N);
    const bool ok_old = check(keys, N, run_old(B, N));
    load(N);
    const bool ok_new = check(keys, N, run_onesweep(B, N, nullptr));
    load(N);
    CK(cub::DeviceRadixSort::SortKeys(c_tmp, c_bytes, B.a, c_out, (int)N, 32, 32 + BITS));
    const bool ok_cub = check(keys, N, c_out);

    // timing: an odd pass count leaves the result in B.b, and B.a then holds an intermediate permutation of the
    // same keys -- the work per sort does not depend on the order, so the repetitions sort whatever B.a holds
    const double us_old = time_us([&] { run_old(B, N); }, REPS);
    const double us_new = time_us([&] { run_onesweep(B, N, nullptr); }, REPS);
    const double us_cub = time_us([&] { cub::DeviceRadixSort::SortKeys(c_tmp, c_bytes, B.a, c_out, (int)N, 32, 32 + BITS); }, REPS);

    // residue sizes: device count, launched for N keys like the index-order pipeline's tail
    const u32 sizes[] = {0, 1, (u32)SORT_TILE - 1, (u32)SORT_TILE, (u32)SORT_TILE + 1, 290000};
    printf("{\"probe\": \"sort\", \"keys\": %u, \"slot_bits\": %u, \"passes\": %u, \"reps\": %d, "
           "\"keys_l2_resident\": true, \"us_per_sort\": {\"three_kernel_lsd\": %.2f, \"onesweep\": %.2f, \"cub_sortkeys\": %.2f}, "
           "\"launches\": {\"three_kernel_lsd\": %u, \"onesweep\": %u}, \"correct\": {\"three_kernel_lsd\": %s, \"onesweep\": %s, \"cub_sortkeys\": %s}, "
           "\"residue_device_count\": [",
           N, BITS, PASSES, REPS, us_old, us_new, us_cub, 3 * PASSES, 1 + PASSES, ok_old ? "true" : "false",
           ok_new ? "true" : "false", ok_cub ? "true" : "false");
    for (size_t s = 0; s < sizeof(sizes) / sizeof(sizes[0]); s++) {
        const u32 n = std::min(sizes[s], N);
        CK(cudaMemcpy(B.n_dev, &n, 4, cudaMemcpyHostToDevice));
        load(N);
        const bool ok = check(keys, n, run_onesweep(B, N, B.n_dev));
        const double us = time_us([&] { run_onesweep(B, N, B.n_dev); }, REPS);
        printf("%s{\"n\": %u, \"us\": %.2f, \"correct\": %s}", s ? ", " : "", n, us, ok ? "true" : "false");
    }
    printf("]}\n");
    return 0;
}
