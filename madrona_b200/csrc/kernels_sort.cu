// kernels_sort.cu -- hot system 1: stable radix sort / compaction of an
// archetype table (all worlds' rows) + fused multi-column permutation.
//
// Semantics follow the reference GPU sort (src/mw/device/sort_archetype.cpp
// :977-1551, SURVEY.md 9.3): key = first 4 bytes of the sort column compared on
// the low 8*P bits, stable LSD; for WorldID sorts rows with key -1 (destroyed)
// sort last and are truncated, worldOffsets/worldCounts are rebuilt (empty
// worlds: offset = numRows, count = 0), entity slots are re-pointed, and the
// whole thing is skipped when !needsSort.
//
// Mechanism is new (the reference expands one sort into ~40 megakernel nodes
// with a device-wide barrier between each and moves every column twice with
// per-element memcpy):
//   1 histogram kernel  (all passes' digit histograms in one read of the keys)
//   P onesweep kernels  (TMA-staged tiles, decoupled look-back that reads 8
//                        predecessors per step, ticketed persistent tiles,
//                        warp match-any ranking -> stable)
//   1 rearrange kernel  (ALL columns in one launch as ticketed (column, chunk)
//                        items in column-major order, each column read once and
//                        written once into its twin buffer; the table's column
//                        pointers are flipped on the device, so no copy-back;
//                        also entity remap + offsets/counts + scratch reset)
// => P+2 launches per sort.  Exported columns must keep their address, so
// they (only) get one extra copy-back launch.
#include "engine.hpp"
#include <cstdio>

namespace mb2 {

constexpr int kSortThreads = 256;
constexpr int kSortWarps = kSortThreads / 32;
#ifndef MB2_SORT_ITEMS
#define MB2_SORT_ITEMS 8
#endif
constexpr int kItemsPerThread = MB2_SORT_ITEMS;
constexpr int kTileItems = kSortThreads * kItemsPerThread;   // 2048
constexpr int kMaxPasses = 4;

struct SortCtrl {
    int32_t tickets[kMaxPasses];
    int32_t numDeleted;
    int32_t blocksDone;
    int32_t didSort;
    int32_t copyBlocksDone;
    int32_t moveTicket;               // rearrange work-item ticket
};

struct SortScratch {
    uint32_t *keys[2] = {};
    int32_t *idx[2] = {};
    int32_t *bins = nullptr;        // [kMaxPasses][256]
    uint32_t *lookback = nullptr;   // [tile][kMaxPasses][256] (layout independent of the table size)
    VMRange keyRanges[2], idxRanges[2], lookbackRange;
    SortCtrl *ctrl = nullptr;
    void **altColumns = nullptr;    // device [kMaxArchetypes][kMaxColumns]
    uint8_t exportedMask[kMaxArchetypes][kMaxColumns] = {};
    bool hasExported[kMaxArchetypes] = {};
    int32_t maxTiles = 0;
    int32_t maxCapacity = 0;
};

struct SortParams {
    EngineState *state;
    uint32_t archetype;
    int32_t keyCol;
    int32_t numPasses;
    int32_t worldSort;
    uint32_t *keys[2];
    int32_t *idx[2];
    int32_t *bins;
    uint32_t *lookback;
    SortCtrl *ctrl;
    void **alt;       // this archetype's row of altColumns
    int32_t maxTiles;
    int32_t hasExported;
};

// ---- TMA (bulk async copy) staging of contiguous tiles: global -> shared memory by the
// copy engine, completion through an mbarrier transaction count.  One elected thread
// issues, everybody waits on the barrier phase.
__device__ __forceinline__ uint32_t smemAddr(const void *p)
{
    return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ void mbarInit(unsigned long long *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smemAddr(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbarExpectTx(unsigned long long *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smemAddr(bar)), "r"(bytes)
                 : "memory");
}

__device__ __forceinline__ void mbarWait(unsigned long long *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@!p bra WAIT_LOOP;\n"
        "}\n" :: "r"(smemAddr(bar)), "r"(parity) : "memory");
}

// global -> shared, bytes a multiple of 16, both addresses 16-byte aligned
__device__ __forceinline__ void tmaLoad1D(void *dst_smem, const void *src_gmem, uint32_t bytes,
                                          unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smemAddr(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smemAddr(bar)) : "memory");
}

// generic-proxy writes to shared memory must be ordered before the async proxy reuses it
__device__ __forceinline__ void fenceProxyAsync()
{
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

__device__ __forceinline__ bool sortActive(const SortParams &p, const TableDesc &t)
{
    // WorldID sorts are skipped for clean tables (sort_archetype.cpp:988-997);
    // custom-key sorts always run.
    return !p.worldSort || t.needsSort != 0;
}

__device__ __forceinline__ uint32_t loadKey(const TableDesc &t, int32_t col, int32_t row)
{
    const char *base = (const char *)t.columns[col];
    return *(const uint32_t *)(base + (size_t)row * t.columnBytes[col]);
}

// ---- kernel 1: digit histograms for every pass + deleted-row count -----------
__global__ void __launch_bounds__(kSortThreads)
sortHistogramKernel(SortParams p)
{
    const TableDesc &t = p.state->tables[p.archetype];
    if (!sortActive(p, t)) return;
    const int32_t n = t.numRows;

    __shared__ uint32_t hist[kMaxPasses][256];
    __shared__ uint32_t deleted;
    for (int i = threadIdx.x; i < kMaxPasses * 256; i += blockDim.x) (&hist[0][0])[i] = 0;
    if (threadIdx.x == 0) deleted = 0;
    __syncthreads();

    uint32_t my_deleted = 0;
    for (int32_t row = blockIdx.x * blockDim.x + threadIdx.x; row < n;
         row += gridDim.x * blockDim.x) {
        uint32_t key = loadKey(t, p.keyCol, row);
        if (key == 0xFFFFFFFFu) my_deleted++;
        for (int pass = 0; pass < p.numPasses; pass++) {
            atomicAdd(&hist[pass][(key >> (8 * pass)) & 0xffu], 1u);
        }
    }
    if (my_deleted) atomicAdd(&deleted, my_deleted);
    __syncthreads();

    for (int i = threadIdx.x; i < p.numPasses * 256; i += blockDim.x) {
        uint32_t v = (&hist[0][0])[i];
        if (v) atomicAdd(&p.bins[i], (int32_t)v);
    }
    if (threadIdx.x == 0 && deleted && p.worldSort) atomicAdd(&p.ctrl->numDeleted, (int32_t)deleted);
}

// ---- kernels 2..P+1: one onesweep pass -------------------------------------------
constexpr uint32_t kFlagAggregate = 1u << 30;
constexpr uint32_t kFlagInclusive = 2u << 30;
constexpr uint32_t kValueMask = (1u << 30) - 1u;
#ifndef MB2_SORT_LOOK_WINDOW
#define MB2_SORT_LOOK_WINDOW 8
#endif
constexpr int kLookWindow = MB2_SORT_LOOK_WINDOW;
// ticketed tiles: any grid size is deadlock free; more resident blocks hide the
// ranking / look-back latency of each tile
// (B200, 3.1M rows: 2 -> 0.659, 3 -> 0.615, 4 -> 0.598, 6 -> 0.599 ms)
#ifndef MB2_SWEEP_BLOCKS_PER_SM
#define MB2_SWEEP_BLOCKS_PER_SM 4
#endif

__global__ void __launch_bounds__(kSortThreads, 4)
sortOnesweepKernel(SortParams p, int pass)
{
    const TableDesc &t = p.state->tables[p.archetype];
    if (!sortActive(p, t)) return;
    const int32_t n = t.numRows;
    const int32_t num_tiles = (n + kTileItems - 1) / kTileItems;
    const bool last_pass = pass == p.numPasses - 1;

    // Side job of the last pass of a world sort: defaults for empty worlds
    // (offset = new numRows, count = 0; sort_archetype.cpp:1269-1337).
    if (last_pass && p.worldSort) {
        const int32_t new_n = n - p.ctrl->numDeleted;
        const int32_t W = (int32_t)p.state->numWorlds;
        for (int32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < W;
             w += gridDim.x * blockDim.x) {
            t.worldOffsets[w] = new_n;
            t.worldCounts[w] = 0;
        }
    }

    const uint32_t *keys_in = p.keys[(pass + 1) & 1];
    const int32_t *idx_in = p.idx[(pass + 1) & 1];
    uint32_t *keys_out = p.keys[pass & 1];
    int32_t *idx_out = p.idx[pass & 1];
    uint32_t *lookback = p.lookback + (size_t)pass * 256;
    constexpr size_t kTileStride = (size_t)kMaxPasses * 256;
    const int shift = 8 * pass;

    __shared__ uint32_t warp_hist[kSortWarps][256];
    __shared__ uint32_t digit_base[256];
    __shared__ uint32_t scan_tmp[kSortWarps];
    __shared__ uint32_t tile_digit_start[256];
    __shared__ __align__(128) uint32_t stage_keys[kTileItems];
    __shared__ __align__(128) int32_t stage_idx[kTileItems];
    __shared__ __align__(8) unsigned long long tile_bar;
    __shared__ int32_t tile_s;
    if (threadIdx.x == 0) mbarInit(&tile_bar, 1);
    uint32_t tile_phase = 0;
    // the (key, index) tile of a pass is contiguous: whole tiles are staged by TMA;
    // pass 0 reads the key column itself (contiguous when it is 4 bytes wide)
    const bool key_col_dense = t.columnBytes[p.keyCol] == 4;

    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;

    // exclusive scan of this pass's global digit histogram (256 bins)
    uint32_t bin_excl;
    {
        uint32_t v = (uint32_t)p.bins[pass * 256 + threadIdx.x];
        uint32_t incl = v;
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += up;
        }
        if (lane == 31) scan_tmp[warp] = incl;
        __syncthreads();
        uint32_t warp_off = 0;
        for (int w = 0; w < warp; w++) warp_off += scan_tmp[w];
        bin_excl = warp_off + incl - v;
        __syncthreads();
    }

    while (true) {
        if (threadIdx.x == 0) tile_s = atomicAdd(&p.ctrl->tickets[pass], 1);
        for (int i = threadIdx.x; i < kSortWarps * 256; i += blockDim.x) (&warp_hist[0][0])[i] = 0;
        __syncthreads();
        const int32_t tile = tile_s;
        if (tile >= num_tiles) break;

        // -- load + stable rank inside the warp's 256-item strip
        uint32_t key[kItemsPerThread];
        int32_t idx[kItemsPerThread];
        uint32_t rank[kItemsPerThread];
        const int32_t strip = tile * kTileItems + warp * (32 * kItemsPerThread);
        const bool whole_tile = (tile + 1) * kTileItems <= n;
        const bool staged = whole_tile && (pass > 0 || key_col_dense);
        if (staged) {
            if (threadIdx.x == 0) {
                fenceProxyAsync();      // the previous tile's digit-order staging wrote these buffers
                const uint32_t bytes = kTileItems * 4;
                mbarExpectTx(&tile_bar, pass == 0 ? bytes : 2 * bytes);
                if (pass == 0) {
                    tmaLoad1D(stage_keys, (const uint32_t *)t.columns[p.keyCol] + (size_t)tile * kTileItems, bytes,
                              &tile_bar);
                } else {
                    tmaLoad1D(stage_keys, keys_in + (size_t)tile * kTileItems, bytes, &tile_bar);
                    tmaLoad1D(stage_idx, idx_in + (size_t)tile * kTileItems, bytes, &tile_bar);
                }
            }
            mbarWait(&tile_bar, tile_phase);
            tile_phase ^= 1u;
        }
        // (a) load the items and match digits across the warp: kItemsPerThread independent
        //     match.any operations in flight instead of one between each pair of shared-memory
        //     updates of (b)
        uint32_t peers_of[kItemsPerThread];
#pragma unroll
        for (int r = 0; r < kItemsPerThread; r++) {
            const int32_t i = strip + r * 32 + lane;
            const bool valid = i < n;
            uint32_t k = 0;
            int32_t src = i;
            if (staged) {
                const int local = warp * (32 * kItemsPerThread) + r * 32 + lane;
                k = stage_keys[local];
                if (pass > 0) src = stage_idx[local];
            } else if (valid) {
                if (pass == 0) {
                    k = loadKey(t, p.keyCol, i);
                } else {
                    k = keys_in[i];
                    src = idx_in[i];
                }
            }
            key[r] = k;
            idx[r] = src;
            const uint32_t digit = (k >> shift) & 0xffu;
            const uint32_t match_val = valid ? digit : (0x100u + (uint32_t)lane);
            peers_of[r] = __match_any_sync(0xffffffffu, match_val);
        }
        // (b) stable ranks: the warp's running digit counts live in shared memory
#pragma unroll
        for (int r = 0; r < kItemsPerThread; r++) {
            const bool valid = strip + r * 32 + lane < n;
            const uint32_t digit = (key[r] >> shift) & 0xffu;
            const uint32_t peers = peers_of[r];
            const uint32_t before = __popc(peers & ((1u << lane) - 1u));
            uint32_t base = 0;
            if (valid) base = warp_hist[warp][digit];
            __syncwarp();
            if (valid && before == 0) warp_hist[warp][digit] = base + __popc(peers);
            __syncwarp();
            rank[r] = valid ? base + before : 0xFFFFFFFFu;
        }
        __syncthreads();

        // -- per digit (thread d): offsets of each warp inside the tile, tile total
        const int d = threadIdx.x;
        uint32_t tile_count = 0;
#pragma unroll
        for (int w = 0; w < kSortWarps; w++) {
            uint32_t c = warp_hist[w][d];
            warp_hist[w][d] = tile_count;
            tile_count += c;
        }

        // -- decoupled look-back across tiles for digit d
        volatile uint32_t *lb = lookback;
        uint32_t excl = 0;
        if (tile == 0) {
            lb[d] = kFlagInclusive | tile_count;
        } else {
            lb[(size_t)tile * kTileStride + d] = kFlagAggregate | tile_count;
            __threadfence();
            // windowed look-back: kLookWindow predecessors are fetched with independent loads and
            // consumed in order, so the serial chain of L2 round trips is 1/kLookWindow as long
            // (with every block starting at once, tile k otherwise walks ~k/2 predecessors one
            // dependent load at a time)
            int32_t look = tile - 1;
            bool done = false;
            while (!done) {
                uint32_t v[kLookWindow];
#pragma unroll
                for (int j = 0; j < kLookWindow; j++) {
                    const int32_t tl = look - j;
                    v[j] = tl >= 0 ? lb[(size_t)tl * kTileStride + d] : 0u;
                }
                bool stop = false;
                int consumed = 0;
#pragma unroll
                for (int j = 0; j < kLookWindow; j++) {
                    const uint32_t flag = v[j] >> 30;
                    if (!stop) {
                        if (flag == 0) {
                            stop = true;                 // predecessor not published yet: retry from it
                        } else {
                            excl += v[j] & kValueMask;
                            consumed++;
                            if (flag == 2u) { done = true; stop = true; }
                        }
                    }
                }
                look -= consumed;
            }
            lb[(size_t)tile * kTileStride + d] = kFlagInclusive | (excl + tile_count);
        }
        // -- the tile's own digit offsets (exclusive scan of tile_count over the 256 digits)
        {
            uint32_t incl = tile_count;
            for (int o = 1; o < 32; o <<= 1) {
                uint32_t up = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += up;
            }
            if (lane == 31) scan_tmp[warp] = incl;
            __syncthreads();
            uint32_t warp_off = 0;
            for (int w = 0; w < warp; w++) warp_off += scan_tmp[w];
            const uint32_t tile_excl = warp_off + incl - tile_count;
            tile_digit_start[d] = tile_excl;
            // global position of the tile's FIRST element of digit d, minus its slot in the tile
            digit_base[d] = bin_excl + excl - tile_excl;
        }
        __syncthreads();

        // -- stage the tile in digit order in shared memory ...
#pragma unroll
        for (int r = 0; r < kItemsPerThread; r++) {
            if (rank[r] == 0xFFFFFFFFu) continue;
            const uint32_t digit = (key[r] >> shift) & 0xffu;
            const uint32_t slot = tile_digit_start[digit] + warp_hist[warp][digit] + rank[r];
            stage_keys[slot] = key[r];
            stage_idx[slot] = idx[r];
        }
        __syncthreads();

        // -- ... and write it out slot by slot: runs of equal digits land on
        //    consecutive addresses, so the scatter is coalesced per run
        const int32_t tile_items = min(kTileItems, n - tile * kTileItems);
        for (int32_t slot = threadIdx.x; slot < tile_items; slot += kSortThreads) {
            const uint32_t k = stage_keys[slot];
            const uint32_t pos = digit_base[(k >> shift) & 0xffu] + (uint32_t)slot;
            keys_out[pos] = k;
            idx_out[pos] = stage_idx[slot];
        }
        __syncthreads();
    }
}

// ---- kernel P+2: fused multi-column permutation ------------------------------------
// Work items = (column, chunk of kRearrangeTile consecutive OUTPUT rows), handed out through
// one ticket counter in COLUMN-MAJOR order: at any moment all blocks gather from the same
// column, so the randomly accessed source column (N x 4..16 bytes) stays L2 resident and
// every 32-byte sector is fetched from DRAM once, not once per element.  The chunk's slice
// of the permutation is staged in shared memory by one TMA bulk copy; each column is moved
// in its widest aligned unit (16/8/4/1 bytes) with coalesced stores, four independent
// gathers in flight per thread.
//
// The same kernel re-points entity slots, derives worldOffsets/worldCounts from the sorted
// keys and wipes the look-back scratch; the last block flips the column pointers and
// publishes the new row count.
constexpr int kRearrangeTile = 2048;
// (B200, sortcheck: 4 -> 0.459, 8 -> 0.458 ms/step, profiles/r2b_ab_table.txt)
#ifndef MB2_REARRANGE_BLOCKS_PER_SM
#define MB2_REARRANGE_BLOCKS_PER_SM 8
#endif

template <typename UnitT>
__device__ __forceinline__ void gatherTile(const void *src_v, void *dst_v, const int32_t *perm_s,
                                           int32_t tile_row0, int32_t rows, uint32_t units_per_row)
{
    const UnitT *__restrict__ src = (const UnitT *)src_v;
    UnitT *__restrict__ dst = (UnitT *)dst_v + (size_t)tile_row0 * units_per_row;
    const uint32_t total = (uint32_t)rows * units_per_row;
    const uint32_t B = blockDim.x;
    uint32_t i = threadIdx.x;
    if (units_per_row == 1) {
        for (; i + 3 * B < total; i += 4 * B) {
            const UnitT a = src[perm_s[i]], b = src[perm_s[i + B]];
            const UnitT c = src[perm_s[i + 2 * B]], d = src[perm_s[i + 3 * B]];
            dst[i] = a; dst[i + B] = b; dst[i + 2 * B] = c; dst[i + 3 * B] = d;
        }
        for (; i < total; i += B) dst[i] = src[perm_s[i]];
    } else if ((units_per_row & (units_per_row - 1)) == 0) {
        const int sh = __ffs(units_per_row) - 1;
        const uint32_t mask = units_per_row - 1;
        auto at = [&](uint32_t k) { return src[((size_t)perm_s[k >> sh] << sh) + (k & mask)]; };
        for (; i + 3 * B < total; i += 4 * B) {
            const UnitT a = at(i), b = at(i + B), c = at(i + 2 * B), d = at(i + 3 * B);
            dst[i] = a; dst[i + B] = b; dst[i + 2 * B] = c; dst[i + 3 * B] = d;
        }
        for (; i < total; i += B) dst[i] = at(i);
    } else {
        for (; i < total; i += B) {
            const uint32_t r = i / units_per_row;
            dst[i] = src[(size_t)perm_s[r] * units_per_row + (i - r * units_per_row)];
        }
    }
}

__global__ void __launch_bounds__(256)
sortRearrangeKernel(SortParams p)
{
    TableDesc &t = p.state->tables[p.archetype];
    if (!sortActive(p, t)) return;
    const int32_t n = t.numRows;
    const int32_t new_n = p.worldSort ? n - p.ctrl->numDeleted : n;
    const int last = (p.numPasses - 1) & 1;
    const int32_t *perm = p.idx[last];
    const uint32_t *sorted_keys = p.keys[last];
    const int32_t num_cols = t.numColumns;

    __shared__ __align__(128) int32_t perm_s[kRearrangeTile];
    __shared__ __align__(8) unsigned long long perm_bar;
    __shared__ int32_t item_s;
    if (threadIdx.x == 0) mbarInit(&perm_bar, 1);
    uint32_t perm_phase = 0;

    const int64_t gtid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t gstride = (int64_t)gridDim.x * blockDim.x;
    // scratch of the finished radix passes: wiped here, spread over all blocks
    {
        const int64_t tiles = (n + kTileItems - 1) / kTileItems;
        for (int64_t i = gtid; i < tiles * kMaxPasses * 256; i += gstride) p.lookback[i] = 0;
        for (int64_t i = gtid; i < p.numPasses * 256; i += gstride) p.bins[i] = 0;
    }
    // world boundaries from the sorted keys
    if (p.worldSort) {
        for (int64_t r64 = gtid; r64 < new_n; r64 += gstride) {
            const int32_t r = (int32_t)r64;
            const uint32_t k = sorted_keys[r];
            if (r == 0 || sorted_keys[r - 1] != k) {
                int32_t end = r + 1;
                while (end < new_n && sorted_keys[end] == k) end++;
                t.worldOffsets[k] = r;
                t.worldCounts[k] = end - r;
            }
        }
    }

    // ---- column moves: ticketed (column, chunk) items in column-major order
    const int32_t chunks = (new_n + kRearrangeTile - 1) / kRearrangeTile;
    const int64_t num_items = (int64_t)chunks * num_cols;
    int32_t staged_chunk = -1;      // which slice of the permutation perm_s holds
    while (true) {
        __syncthreads();            // the previous item is done with perm_s / item_s
        if (threadIdx.x == 0) item_s = atomicAdd(&p.ctrl->moveTicket, 1);
        __syncthreads();
        const int64_t item = item_s;
        if (item >= num_items) break;
        const int32_t col = (int32_t)(item / chunks);
        const int32_t chunk = (int32_t)(item - (int64_t)col * chunks);
        const int32_t row0 = chunk * kRearrangeTile;
        const int32_t rows = min(kRearrangeTile, new_n - row0);
        const uint32_t bytes = t.columnBytes[col];

        if (staged_chunk != chunk) {
            if (rows == kRearrangeTile) {
                // the chunk's slice of the permutation: one bulk copy
                if (threadIdx.x == 0) {
                    fenceProxyAsync();
                    mbarExpectTx(&perm_bar, kRearrangeTile * 4);
                    tmaLoad1D(perm_s, perm + row0, kRearrangeTile * 4, &perm_bar);
                }
                mbarWait(&perm_bar, perm_phase);
                perm_phase ^= 1u;
            } else {
                for (int32_t i = threadIdx.x; i < rows; i += blockDim.x) perm_s[i] = perm[row0 + i];
                __syncthreads();
            }
            staged_chunk = chunk;
        }

        const void *src = t.columns[col];
        void *dst = p.alt[col];
        if (col == 0) {
            // Entity column: move + re-point the entity slot at the new row
            // (sort_archetype.cpp:1357-1379)
            const unsigned long long *sp = (const unsigned long long *)src;
            unsigned long long *dp = (unsigned long long *)dst;
            EntitySlot *slots = p.state->entitySlots;
            for (int32_t i = threadIdx.x; i < rows; i += blockDim.x) {
                const unsigned long long e = sp[perm_s[i]];
                dp[row0 + i] = e;
                const uint32_t gen = (uint32_t)(e & 0xFFFFFFFFull);
                const int32_t id = (int32_t)(uint32_t)(e >> 32);
                if (id >= 0 && gen != 0xFFFFFFFFu && id < p.state->entityCapacity &&
                        slots[id].gen == gen && slots[id].a == (int32_t)p.archetype) {
                    slots[id].b = row0 + i;
                }
            }
        } else if ((bytes & 15u) == 0) {
            gatherTile<uint4>(src, dst, perm_s, row0, rows, bytes >> 4);
        } else if ((bytes & 7u) == 0) {
            gatherTile<uint2>(src, dst, perm_s, row0, rows, bytes >> 3);
        } else if ((bytes & 3u) == 0) {
            gatherTile<uint32_t>(src, dst, perm_s, row0, rows, bytes >> 2);
        } else if ((bytes & 1u) == 0) {
            gatherTile<unsigned short>(src, dst, perm_s, row0, rows, bytes >> 1);
        } else {
            gatherTile<unsigned char>(src, dst, perm_s, row0, rows, bytes);
        }
    }

    // ---- last block out: flip column buffers, publish the new row count
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t done = atomicAdd(&p.ctrl->blocksDone, 1);
        is_last = done == (int32_t)gridDim.x - 1;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();

    for (int c = threadIdx.x; c < num_cols; c += blockDim.x) {
        void *old_main = t.columns[c];
        t.columns[c] = p.alt[c];
        p.alt[c] = old_main;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        t.numRows = new_n;
        if ((uint32_t)n > t.highWater) t.highWater = (uint32_t)n;
        // a custom-key sort leaves the table out of world order
        // (sort_archetype.cpp:1003-1007)
        t.needsSort = p.worldSort ? 0u : 1u;
        for (int i = 0; i < kMaxPasses; i++) p.ctrl->tickets[i] = 0;
        p.ctrl->numDeleted = 0;
        p.ctrl->blocksDone = 0;
        p.ctrl->moveTicket = 0;
        p.ctrl->didSort = p.hasExported;
    }
}

// Exported columns must keep their address: after the flip their data sits in
// the twin buffer, so copy it back and flip those pointers again.
__global__ void __launch_bounds__(256)
sortCopyBackKernel(SortParams p, unsigned long long exported_mask)
{
    TableDesc &t = p.state->tables[p.archetype];
    if (!p.ctrl->didSort) return;
    const int32_t n = t.numRows;
    const int32_t col = blockIdx.y;
    if (col < t.numColumns && ((exported_mask >> col) & 1ull)) {
        // after the flip: t.columns[col] = twin (holds data), p.alt[col] = exported address
        // (columns are 256-byte aligned with 256 bytes of slack: whole 16-byte units)
        const uint4 *src = (const uint4 *)t.columns[col];
        uint4 *dst = (uint4 *)p.alt[col];
        const int64_t units = ((int64_t)n * t.columnBytes[col] + 15) / 16;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < units;
             i += (int64_t)gridDim.x * blockDim.x) {
            dst[i] = src[i];
        }
    }
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        int32_t done = atomicAdd(&p.ctrl->copyBlocksDone, 1);
        is_last = done == (int32_t)(gridDim.x * gridDim.y) - 1;
    }
    __syncthreads();
    if (!is_last) return;
    __threadfence();
    for (int c = threadIdx.x; c < t.numColumns; c += blockDim.x) {
        if ((exported_mask >> c) & 1ull) {
            void *twin = t.columns[c];
            t.columns[c] = p.alt[c];
            p.alt[c] = twin;
        }
    }
    if (threadIdx.x == 0) {
        p.ctrl->copyBlocksDone = 0;
        p.ctrl->didSort = 0;
    }
}

// ---- host side -----------------------------------------------------------------------

bool sortScratchCreate(Executor *ex, std::string *err)
{
    EngineState &S = *ex->hState;
    SortScratch *sc = new SortScratch();
    ex->sortScratch = sc;

    int32_t max_cap = 256;
    for (uint32_t a = 0; a < S.numArchetypes; a++) {
        if (S.archetypes[a].registered && !S.tables[a].isSingleton)
            max_cap = std::max(max_cap, S.tables[a].capacity);
    }

    // key / index / look-back scratch: address ranges big enough for any table, memory
    // mapped for the largest table that exists (sortScratchEnsure maps more)
    const size_t max_rows = 0x7fffff00ull;
    bool ok = true;
    for (int i = 0; i < 2 && ok; i++) {
        ok = vmReserve(ex->gpu, &sc->keyRanges[i], max_rows * 4, 4096, err) &&
             vmReserve(ex->gpu, &sc->idxRanges[i], max_rows * 4, 4096, err);
        sc->keys[i] = (uint32_t *)sc->keyRanges[i].base;
        sc->idx[i] = (int32_t *)sc->idxRanges[i].base;
    }
    ok = ok && vmReserve(ex->gpu, &sc->lookbackRange, (max_rows / kTileItems + 2) * kMaxPasses * 256 * 4, 4096, err);
    sc->lookback = (uint32_t *)sc->lookbackRange.base;
    if (!ok || !sortScratchEnsure(ex, max_cap, err)) return false;
    ok = ok && devAlloc(ex, (void **)&sc->bins, sizeof(int32_t) * kMaxPasses * 256);
    ok = ok && devAlloc(ex, (void **)&sc->ctrl, sizeof(SortCtrl));
    ok = ok && devAlloc(ex, (void **)&sc->altColumns, sizeof(void *) * kMaxArchetypes * kMaxColumns);
    if (!ok) {
        *err = "sort scratch allocation failed";
        return false;
    }

    for (uint32_t s = 0; s < S.numExported && s < (uint32_t)kMaxExports; s++) {
        const ExportInfo &e = S.exports[s];
        if (!e.used) continue;
        int col = S.columnLookup[e.archetype][e.component];
        sc->exportedMask[e.archetype][col] = 1;
        sc->hasExported[e.archetype] = true;
    }

    // twin buffer for every column of every sortable table
    std::vector<void *> alts((size_t)kMaxArchetypes * kMaxColumns, nullptr);
    for (uint32_t a = 0; a < S.numArchetypes; a++) {
        if (!S.archetypes[a].registered || S.tables[a].isSingleton) continue;
        const TableDesc &t = S.tables[a];
        const bool growable = !ex->columnRanges[a].empty();
        if (growable) ex->twinRanges[a].resize(t.numColumns);
        for (int32_t c = 0; c < t.numColumns; c++) {
            void *p = nullptr;
            if (growable) {
                // same address-range size as the column itself
                if (!vmReserve(ex->gpu, &ex->twinRanges[a][c], ex->columnRanges[a][c].reserved,
                               (size_t)t.columnBytes[c] * t.capacity + 256, err)) return false;
                p = ex->twinRanges[a][c].base;
            } else if (!devAlloc(ex, &p, (size_t)t.columnBytes[c] * t.capacity + 256)) {
                *err = "sort twin buffer allocation failed";
                return false;
            }
            alts[(size_t)a * kMaxColumns + c] = p;
        }
    }
    cudaMemcpyAsync(sc->altColumns, alts.data(), sizeof(void *) * alts.size(),
                    cudaMemcpyHostToDevice, ex->stream);
    cudaStreamSynchronize(ex->stream);
    return true;
}

bool sortScratchEnsure(Executor *ex, int32_t max_rows, std::string *err)
{
    SortScratch *sc = ex->sortScratch;
    if (max_rows <= sc->maxCapacity) return true;
    const size_t tiles = (size_t)(max_rows + kTileItems - 1) / kTileItems + 1;
    for (int i = 0; i < 2; i++) {
        if (!vmGrow(ex->gpu, &sc->keyRanges[i], (size_t)max_rows * 4, err) ||
            !vmGrow(ex->gpu, &sc->idxRanges[i], (size_t)max_rows * 4, err)) return false;
    }
    if (!vmGrow(ex->gpu, &sc->lookbackRange, tiles * kMaxPasses * 256 * 4, err)) return false;
    sc->maxCapacity = max_rows;
    sc->maxTiles = (int32_t)tiles;
    return true;
}

void sortScratchDestroy(Executor *ex)
{
    SortScratch *sc = ex->sortScratch;
    if (sc) {
        for (int i = 0; i < 2; i++) {
            vmRelease(&sc->keyRanges[i]);
            vmRelease(&sc->idxRanges[i]);
        }
        vmRelease(&sc->lookbackRange);
    }
    delete sc;
    ex->sortScratch = nullptr;
}

static int worldSortPasses(uint32_t num_worlds)
{
    // every valid world ID must stay below the all-ones masked key of a
    // destroyed row: W < 2^(8P)
    int bits = 0;
    while ((num_worlds >> bits) != 0) bits++;
    int passes = (bits + 7) / 8;
    return passes < 1 ? 1 : passes;
}

int sortNumPasses(Executor *ex, int32_t col)
{
    return col == 1 ? worldSortPasses(ex->hState->numWorlds) : 4;
}

void launchSortArchetype(Executor *ex, uint32_t archetype, int32_t col, cudaStream_t s)
{
    EngineState &S = *ex->hState;
    SortScratch *sc = ex->sortScratch;
    const TableDesc &t = S.tables[archetype];
    if (t.isSingleton) return;

    SortParams p;
    p.state = ex->dState;
    p.archetype = archetype;
    p.keyCol = col;
    p.worldSort = col == 1 ? 1 : 0;
    p.numPasses = p.worldSort ? worldSortPasses(S.numWorlds) : 4;
    p.keys[0] = sc->keys[0];
    p.keys[1] = sc->keys[1];
    p.idx[0] = sc->idx[0];
    p.idx[1] = sc->idx[1];
    p.bins = sc->bins;
    p.lookback = sc->lookback;
    p.ctrl = sc->ctrl;
    p.alt = sc->altColumns + (size_t)archetype * kMaxColumns;
    p.maxTiles = sc->maxTiles;

    unsigned long long mask = 0;
    for (int c = 0; c < t.numColumns; c++) {
        if (sc->exportedMask[archetype][c]) mask |= 1ull << c;
    }
    p.hasExported = mask ? 1 : 0;

    const int tiles = (t.capacity + kTileItems - 1) / kTileItems;
    const int hist_grid = std::max(1, std::min(tiles, ex->numSMs * 4));
    const int sweep_grid = std::max(1, std::min(tiles, ex->numSMs * MB2_SWEEP_BLOCKS_PER_SM));
    sortHistogramKernel<<<hist_grid, kSortThreads, 0, s>>>(p);
    for (int pass = 0; pass < p.numPasses; pass++) {
        sortOnesweepKernel<<<sweep_grid, kSortThreads, 0, s>>>(p, pass);
    }
    const int rtiles = (t.capacity + kRearrangeTile - 1) / kRearrangeTile;
    const int rblocks = std::max(1, std::min(rtiles * std::max(1, t.numColumns / 2),
                                             ex->numSMs * MB2_REARRANGE_BLOCKS_PER_SM));
    sortRearrangeKernel<<<rblocks, 256, 0, s>>>(p);
    const int row_blocks = std::max(1, std::min((t.capacity + 255) / 256, ex->numSMs * 4));
    dim3 rgrid((unsigned)row_blocks, (unsigned)t.numColumns);

    if (mask) sortCopyBackKernel<<<rgrid, 256, 0, s>>>(p, mask);
}

}
