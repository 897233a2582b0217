// engine.cpp -- libmadrona_b200.so host side: the C ABI declared in
// include/madrona_b200.h.  Replaces the reference's MWCudaExecutor
// implementation (src/mw/cuda_exec.cpp, 2807 LoC: NVRTC+nvJitLink megakernel
// build, VM allocator thread, print thread, megakernel CUDA graph) with:
//   JIT (jit.cpp) -> load cubin -> device-side registerTypes -> host allocates
//   SoA tables -> two-pass deterministic world construction -> device-side
//   setupTasks -> one CUDA graph per launch graph with one kernel node per
//   TaskGraph node (stream capture).
// The product path is CUDA only: there is no CPU fallback anywhere in here.
#include "../../include/madrona_b200.h"
#include "engine.hpp"
#include "physics_host.hpp"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>

namespace mb2 {

static thread_local std::string g_last_error;

void setError(const std::string &msg)
{
    g_last_error = msg;
    if (getenv("MADRONA_B200_VERBOSE")) fprintf(stderr, "[madrona_b200] %s\n", msg.c_str());
}

#define MB2_CUDA(expr) do { \
    cudaError_t mb2_err_ = (expr); \
    if (mb2_err_ != cudaSuccess) { \
        setError(std::string(#expr) + ": " + cudaGetErrorString(mb2_err_)); \
        return false; \
    } } while (0)

bool devAlloc(Executor *ex, void **ptr, size_t bytes, bool zero)
{
    if (bytes == 0) bytes = 16;
    MB2_CUDA(cudaMalloc(ptr, bytes));
    ex->allocations.push_back(*ptr);
    if (zero) MB2_CUDA(cudaMemsetAsync(*ptr, 0, bytes, ex->stream));
    return true;
}

static bool pushState(Executor *ex)
{
    MB2_CUDA(cudaMemcpyAsync(ex->dState, ex->hState, sizeof(EngineState),
                             cudaMemcpyHostToDevice, ex->stream));
    MB2_CUDA(cudaStreamSynchronize(ex->stream));
    return true;
}

static bool pullState(Executor *ex)
{
    MB2_CUDA(cudaStreamSynchronize(ex->stream));
    MB2_CUDA(cudaMemcpy(ex->hState, ex->dState, sizeof(EngineState),
                        cudaMemcpyDeviceToHost));
    return true;
}

static std::string describeErrors(uint32_t flags, uint32_t archetype)
{
    std::string s;
    if (flags & ErrTableOverflow) s += "table overflow (archetype " + std::to_string(archetype) +
        "; raise MADRONA_B200_ROWS_PER_WORLD) ";
    if (flags & ErrEntityOverflow) s += "entity store overflow ";
    if (flags & ErrTmpOverflow) s += "tmp allocator overflow (raise MADRONA_B200_TMP_BYTES) ";
    if (flags & ErrPersistOverflow) s += "persistent arena overflow (raise MADRONA_B200_PERSIST_BYTES) ";
    if (flags & ErrTooManyNodes) s += "too many taskgraph nodes ";
    if (flags & ErrRegistry) s += "ECS registration error (unregistered component, too many types, bad export slot) ";
    if (flags & ErrPhysicsOverflow) s += "physics buffer overflow ";
    return s;
}

static bool checkDeviceErrors(Executor *ex, const char *phase)
{
    uint32_t st[2];
    MB2_CUDA(cudaMemcpy(st, &ex->dState->errorFlags, sizeof(st), cudaMemcpyDeviceToHost));
    if (st[0] != 0) {
        setError(std::string(phase) + ": " + describeErrors(st[0], st[1]));
        return false;
    }
    return true;
}

static bool launch1(Executor *ex, cudaKernel_t k, unsigned grid, unsigned block)
{
    void *args[1] = { nullptr };
    MB2_CUDA(cudaLaunchKernel((const void *)k, dim3(grid), dim3(block), args, 0, ex->stream));
    MB2_CUDA(cudaStreamSynchronize(ex->stream));
    return true;
}

uint64_t envU64(const char *name, uint64_t dflt)
{
    const char *v = getenv(name);
    if (!v || !*v) return dflt;
    return strtoull(v, nullptr, 10);
}

// ---- table allocation after registerTypes ---------------------------------

static bool allocateTables(Executor *ex)
{
    EngineState &S = *ex->hState;
    const uint32_t W = S.numWorlds;

    memset(S.columnLookup, 0xff, sizeof(S.columnLookup));

    uint64_t total_entity_rows = 0;
    for (uint32_t a = 0; a < S.numArchetypes; a++) {
        const ArchetypeInfo &info = S.archetypes[a];
        TableDesc &t = S.tables[a];
        memset(&t, 0, sizeof(t));
        if (!info.registered) continue;

        uint64_t cap;
        if (info.isSingleton) cap = W;
        else if (info.maxPerWorld > 0) cap = (uint64_t)W * (uint64_t)info.maxPerWorld;
        else cap = (uint64_t)W * ex->rowsPerWorldHint;
        if (cap > 0x7fffff00ull) {
            setError("table too large");
            return false;
        }
        cap = (cap + 255) & ~255ull;

        t.numColumns = (int32_t)info.numUserComponents + 2;
        t.capacity = (int32_t)cap;
        t.maxPerWorld = info.maxPerWorld;
        t.isSingleton = info.isSingleton;
        t.numRows = info.isSingleton ? (int32_t)W : 0;

        // dynamic archetypes live in growable address ranges (up to 64x the initial
        // capacity, the row index stays a positive int32); fixed ones are W x max rows for good
        const bool growable = ex->tableGrowth && !info.isSingleton && info.maxPerWorld == 0;
        const uint64_t reserve_rows = std::min<uint64_t>(cap * 64, 0x7fffff00ull);
        if (growable) ex->columnRanges[a].resize(t.numColumns);
        for (int32_t c = 0; c < t.numColumns; c++) {
            uint32_t cid = c == 0 ? 0u : (c == 1 ? 1u : info.componentIDs[c - 2]);
            if (cid >= S.numComponents) {
                setError("archetype " + std::to_string(a) + " uses an unregistered component");
                return false;
            }
            uint32_t bytes = S.components[cid].numBytes;
            t.columnBytes[c] = bytes;
            if (growable) {
                std::string verr;
                if (!vmReserve(ex->gpu, &ex->columnRanges[a][c], (size_t)bytes * reserve_rows + 256,
                               (size_t)bytes * cap + 256, &verr)) {
                    setError(verr);
                    return false;
                }
                t.columns[c] = ex->columnRanges[a][c].base;
            } else if (!devAlloc(ex, &t.columns[c], (size_t)bytes * cap + 256)) {
                return false;
            }
            S.columnLookup[a][cid] = (i16)c;
        }
        if (!devAlloc(ex, (void **)&t.worldOffsets, sizeof(int32_t) * W)) return false;
        if (!devAlloc(ex, (void **)&t.worldCounts, sizeof(int32_t) * W)) return false;
        if (!info.isSingleton) total_entity_rows += cap;
    }

    // exports: pointer == base of the live column (reference:
    // src/mw/device/include/madrona/state.inl:522-532)
    for (uint32_t s = 0; s < S.numExported && s < (uint32_t)kMaxExports; s++) {
        const ExportInfo &e = S.exports[s];
        if (!e.used) continue;
        if (e.archetype >= S.numArchetypes || e.component >= S.numComponents ||
                S.columnLookup[e.archetype][e.component] < 0) {
            setError("export slot " + std::to_string(s) + " names a component its archetype lacks");
            return false;
        }
        int col = S.columnLookup[e.archetype][e.component];
        ex->exported[s] = S.tables[e.archetype].columns[col];
        ex->exportArchetype[s] = e.archetype;
        ex->exportRowBytes[s] = S.tables[e.archetype].columnBytes[col];
    }

    // entity store: singleton rows take the first IDs in registration order,
    // exactly as the CPU backend's init_state_cache_ hands them out
    // (include/madrona/state.inl:163-179).
    uint64_t singleton_ids = (uint64_t)S.numSingletons * W;
    uint64_t init_blocks = (singleton_ids + kIDsPerCache - 1) / kIDsPerCache;
    uint64_t ent_cap = init_blocks * kIDsPerCache + total_entity_rows +
        (uint64_t)W * kIDsPerCache * 2;
    ent_cap = (ent_cap + kIDsPerCache - 1) / kIDsPerCache * kIDsPerCache;
    if (ent_cap > 0x7fffff00ull) {
        setError("entity store too large");
        return false;
    }
    S.entityCapacity = (int32_t)ent_cap;
    S.initExpandBlocks = (int32_t)init_blocks;
    S.numEntitySlots = (int32_t)(init_blocks * kIDsPerCache);
    S.freeHead = ((u64)0 << 32) | (u32)kIDSentinel;
    if (ex->tableGrowth) {
        std::string verr;
        if (!vmReserve(ex->gpu, &ex->entityRange, sizeof(EntitySlot) * 0x7fffff00ull, sizeof(EntitySlot) * ent_cap,
                       &verr)) {
            setError(verr);
            return false;
        }
        S.entitySlots = (EntitySlot *)ex->entityRange.base;
    } else if (!devAlloc(ex, (void **)&S.entitySlots, sizeof(EntitySlot) * ent_cap)) {
        return false;
    }
    if (!devAlloc(ex, (void **)&S.idCaches, sizeof(IDCache) * W)) return false;

    S.tmpCapacity = envU64("MADRONA_B200_TMP_BYTES", 256ull << 20);
    S.persistCapacity = envU64("MADRONA_B200_PERSIST_BYTES", (64ull << 20) + (uint64_t)W * (24ull << 10));
    if (!devAlloc(ex, (void **)&S.tmpArena, S.tmpCapacity, false)) return false;
    if (!devAlloc(ex, (void **)&S.persistArena, S.persistCapacity)) return false;
    S.tmpOffset = 0;
    S.persistOffset = 0;
    return true;
}

}   // namespace mb2 (reopened below)

namespace mb2 {

bool growTable(Executor *ex, uint32_t a, int64_t new_cap, std::string *err)
{
    EngineState &S = *ex->hState;
    TableDesc &t = S.tables[a];
    if (ex->columnRanges[a].empty()) {
        *err = "archetype " + std::to_string(a) + " has a fixed size";
        return false;
    }
    new_cap = (new_cap + 255) & ~255ll;
    if (new_cap <= t.capacity) return true;
    if (new_cap > 0x7fffff00ll) {
        *err = "table too large";
        return false;
    }
    const int64_t added = new_cap - t.capacity;
    for (int32_t c = 0; c < t.numColumns; c++) {
        const size_t bytes = (size_t)t.columnBytes[c] * (size_t)new_cap + 256;
        if (!vmGrow(ex->gpu, &ex->columnRanges[a][c], bytes, err)) return false;
        if (!ex->twinRanges[a].empty() && !vmGrow(ex->gpu, &ex->twinRanges[a][c], bytes, err)) return false;
    }
    if (ex->sortScratch && !sortScratchEnsure(ex, (int32_t)new_cap, err)) return false;
    // one entity slot per possible row
    const int64_t new_ent = std::min<int64_t>((int64_t)S.entityCapacity + added, 0x7fffff00ll);
    if (!vmGrow(ex->gpu, &ex->entityRange, sizeof(EntitySlot) * (size_t)new_ent, err)) return false;
    S.entityCapacity = (int32_t)new_ent;
    t.capacity = (int32_t)new_cap;
    cudaMemcpy(&ex->dState->tables[a].capacity, &t.capacity, sizeof(int32_t), cudaMemcpyHostToDevice);
    cudaMemcpy(&ex->dState->entityCapacity, &S.entityCapacity, sizeof(int32_t), cudaMemcpyHostToDevice);
    if (getenv("MADRONA_B200_VERBOSE")) {
        fprintf(stderr, "[madrona_b200] archetype %u grown to %ld rows\n", a, (long)new_cap);
    }
    return true;
}

// Between steps: a dynamic table whose row count peaked above half its capacity during
// the last graph gets twice the room (so that one step can at most double a table
// without overflowing -- the worst case of a full reset before compaction).
static bool growTablesFromStatus(Executor *ex)
{
    if (!ex->tableGrowth) return true;
    EngineState &S = *ex->hState;
    for (uint32_t a = 0; a < S.numArchetypes && a < (uint32_t)kMaxArchetypes; a++) {
        if (ex->columnRanges[a].empty()) continue;
        const int64_t peak = ex->hStatus[2 + a];
        int64_t cap = S.tables[a].capacity;
        if (peak * 2 <= cap) continue;
        while (cap < peak * 2) cap *= 2;
        std::string err;
        if (!growTable(ex, a, cap, &err)) {
            setError("table growth: " + err);
            return false;
        }
    }
    return true;
}

static bool resetForInitPass(Executor *ex, uint32_t pass, const std::vector<int32_t> &expand_base,
                             uint64_t persist_mark)
{
    EngineState &S = *ex->hState;
    const uint32_t W = S.numWorlds;
    for (uint32_t a = 0; a < S.numArchetypes; a++) {
        TableDesc &t = S.tables[a];
        if (!S.archetypes[a].registered) continue;
        if (t.isSingleton) {
            t.numRows = (int32_t)W;
            for (int32_t c = 2; c < t.numColumns; c++) {
                MB2_CUDA(cudaMemsetAsync(t.columns[c], 0, (size_t)t.columnBytes[c] * t.capacity, ex->stream));
            }
        } else {
            t.numRows = 0;
        }
        t.needsSort = 0;
        t.highWater = 0;
    }
    MB2_CUDA(cudaMemsetAsync(S.entitySlots, 0, sizeof(EntitySlot) * (size_t)S.entityCapacity, ex->stream));
    std::vector<IDCache> caches(W);
    for (uint32_t w = 0; w < W; w++) {
        IDCache &c = caches[w];
        memset(&c, 0, sizeof(c));
        c.freeHead = kIDSentinel;
        c.overflowHead = kIDSentinel;
        c.expandBase = expand_base.empty() ? 0 : expand_base[w];
    }
    MB2_CUDA(cudaMemcpyAsync(S.idCaches, caches.data(), sizeof(IDCache) * W,
                             cudaMemcpyHostToDevice, ex->stream));
    MB2_CUDA(cudaMemsetAsync(S.worldData, 0, (size_t)S.worldDataStride * W, ex->stream));
    S.numEntitySlots = S.initExpandBlocks * kIDsPerCache;
    S.freeHead = ((u64)0 << 32) | (u32)kIDSentinel;
    S.tmpOffset = 0;
    S.persistOffset = persist_mark;
    S.errorFlags = 0;
    S.initPass = pass;
    if (!pushState(ex)) return false;
    launchFillSingletons(ex, ex->stream);
    MB2_CUDA(cudaStreamSynchronize(ex->stream));
    return true;
}

static bool createExecutor(Executor *ex, const mb2_state_config *sc,
                           const mb2_compile_config *cc,
                           const mb2_render_config *rc)
{
    if (sc->num_worlds == 0) {
        setError("numWorlds must be > 0");
        return false;
    }
    if (sc->num_taskgraphs > (uint32_t)kMaxTaskGraphs) {
        setError("too many taskgraphs");
        return false;
    }
    if (sc->num_exported_buffers > (uint32_t)kMaxExports) {
        setError("too many exported buffers");
        return false;
    }

    MB2_CUDA(cudaSetDevice(ex->gpu));
    cudaDeviceProp prop;
    MB2_CUDA(cudaGetDeviceProperties(&prop, ex->gpu));
    ex->numSMs = prop.multiProcessorCount;
    if (prop.major < 10) {
        setError("madrona_b200 requires an sm_100a device (found sm_" +
                 std::to_string(prop.major) + std::to_string(prop.minor) + ")");
        return false;
    }
    // a blocking stream, like the reference's cu::makeStream() (plain
    // cudaStreamCreate): work the caller queued on the legacy default stream --
    // torch's `actions.copy_(...)` -- is ordered before the step graph
    MB2_CUDA(cudaStreamCreate(&ex->stream));
    ex->rowsPerWorldHint = envU64("MADRONA_B200_ROWS_PER_WORLD", 128);
    ex->tableGrowth = envU64("MADRONA_B200_TABLE_GROWTH", 1) != 0;

    // ---- JIT the simulator
    std::vector<std::string> sources, flags;
    for (uint32_t i = 0; i < cc->num_user_sources; i++) sources.push_back(cc->user_sources[i]);
    for (uint32_t i = 0; i < cc->num_user_compile_flags; i++) flags.push_back(cc->user_compile_flags[i]);
    std::string err;
    if (!jitCompile(sources, flags, (int)cc->opt_mode, &ex->jit, &err)) {
        setError(err);
        return false;
    }
    MB2_CUDA(cudaLibraryLoadData(&ex->lib, ex->jit.cubin.data(), nullptr, nullptr, 0,
                                 nullptr, nullptr, 0));
    if (cudaLibraryGetKernel(&ex->initECS, ex->lib, "mb2_entry_init_ecs") != cudaSuccess ||
        cudaLibraryGetKernel(&ex->initWorlds, ex->lib, "mb2_entry_init_worlds") != cudaSuccess ||
        cudaLibraryGetKernel(&ex->initTasks, ex->lib, "mb2_entry_init_tasks") != cudaSuccess) {
        cudaGetLastError();
        setError("simulator module lacks MADRONA_BUILD_MWGPU_ENTRY(...) entry points");
        return false;
    }
    for (size_t i = 0; i < ex->jit.nodeKernels.size(); i++) {
        cudaKernel_t k;
        MB2_CUDA(cudaLibraryGetKernel(&k, ex->lib, ex->jit.nodeKernels[i].c_str()));
        void *meta = nullptr;
        size_t meta_bytes = 0;
        MB2_CUDA(cudaLibraryGetGlobal(&meta, &meta_bytes, ex->lib, ex->jit.nodeMetas[i].c_str()));
        ex->nodeKernels.push_back(k);
        ex->nodeMetaAddrs.push_back((uint64_t)(uintptr_t)meta);
    }

    // ---- engine state block
    ex->hState = (EngineState *)calloc(1, sizeof(EngineState));
    if (!devAlloc(ex, (void **)&ex->dState, sizeof(EngineState))) return false;
    MB2_CUDA(cudaMallocHost((void **)&ex->hStatus, sizeof(uint32_t) * kStatusWords));
    memset(ex->hStatus, 0, sizeof(uint32_t) * kStatusWords);

    EngineState &S = *ex->hState;
    S.numWorlds = sc->num_worlds;
    S.numTaskGraphs = sc->num_taskgraphs;
    S.numExported = sc->num_exported_buffers;
    if (!devAlloc(ex, &S.userConfig, std::max(sc->num_user_config_bytes, 16u))) return false;
    if (sc->num_user_config_bytes)
        MB2_CUDA(cudaMemcpy(S.userConfig, sc->user_config_ptr, sc->num_user_config_bytes,
                            cudaMemcpyHostToDevice));
    S.worldInitBytes = sc->num_world_init_bytes;
    size_t init_bytes = (size_t)sc->num_world_init_bytes * sc->num_worlds;
    if (!devAlloc(ex, &S.worldInits, std::max(init_bytes, (size_t)16))) return false;
    if (init_bytes)
        MB2_CUDA(cudaMemcpy(S.worldInits, sc->world_init_ptr, init_bytes, cudaMemcpyHostToDevice));

    // engine-owned systems get their device blocks before registerTypes so the
    // simulator's calls into PhysicsSystem / RenderingSystem can record into them
    if (!physicsHostCreate(ex, &err) || !renderHostCreate(ex, rc, &err)) {
        setError(err);
        return false;
    }
    if (!pushState(ex)) return false;

    void *state_sym = nullptr;
    size_t state_sym_bytes = 0;
    MB2_CUDA(cudaLibraryGetGlobal(&state_sym, &state_sym_bytes, ex->lib, "mb2_engine_state"));
    MB2_CUDA(cudaMemcpy(state_sym, &ex->dState, sizeof(void *), cudaMemcpyHostToDevice));

    // ---- phase 1: registerTypes on the device (1 thread)
    if (!launch1(ex, ex->initECS, 1, 1)) return false;
    if (!pullState(ex)) return false;
    if (!checkDeviceErrors(ex, "registerTypes")) return false;

    // ---- phase 2: storage.  numWorldDataBytes == 0 means "use sizeof(WorldT) as
    // the device compiler sees it" (the only size that matters here).
    {
        uint32_t bytes = sc->num_world_data_bytes ? sc->num_world_data_bytes : S.worldDataNeeded;
        if (bytes < S.worldDataNeeded) {
            setError("StateConfig::numWorldDataBytes (" + std::to_string(bytes) +
                     ") is smaller than the simulator's per-world data type (" +
                     std::to_string(S.worldDataNeeded) + ")");
            return false;
        }
        uint32_t align = std::max({ sc->world_data_alignment, S.worldDataAlignNeeded, 16u });
        S.worldDataStride = (bytes + align - 1) / align * align;
        if (!devAlloc(ex, (void **)&S.worldData, (size_t)S.worldDataStride * S.numWorlds)) return false;
    }
    if (!allocateTables(ex)) return false;
    if (!sortScratchCreate(ex, &err)) {
        setError(err);
        return false;
    }
    if (!physicsHostAfterRegistry(ex, rc, &err) || !renderHostAfterRegistry(ex, &err)) {
        setError(err);
        return false;
    }
    const uint64_t persist_mark = ex->hState->persistOffset;

    // ---- phase 3: world constructors, two passes (see mb2_state.h IDCache)
    const unsigned wblocks = (S.numWorlds + 127) / 128;
    for (int attempt = 0;; attempt++) {
        if (!resetForInitPass(ex, 0, {}, persist_mark)) return false;
        if (!launch1(ex, ex->initWorlds, wblocks, 128)) return false;
        // a dynamic table too small for the worlds' initial population: double it and
        // construct again (the dry run exists to be repeated)
        uint32_t st[2] = { 0, 0 };
        MB2_CUDA(cudaMemcpy(st, &ex->dState->errorFlags, sizeof(st), cudaMemcpyDeviceToHost));
        if (st[0] == (uint32_t)ErrTableOverflow && ex->tableGrowth && attempt < 12 &&
                st[1] < S.numArchetypes && !ex->columnRanges[st[1]].empty()) {
            std::string gerr;
            if (!growTable(ex, st[1], (int64_t)S.tables[st[1]].capacity * 2, &gerr)) {
                setError("world construction: " + gerr);
                return false;
            }
            continue;
        }
        if (!checkDeviceErrors(ex, "world construction (dry run)")) return false;
        break;
    }

    std::vector<IDCache> caches(S.numWorlds);
    MB2_CUDA(cudaMemcpy(caches.data(), S.idCaches, sizeof(IDCache) * S.numWorlds,
                        cudaMemcpyDeviceToHost));
    std::vector<int32_t> expand_base(S.numWorlds);
    int64_t next_block = S.initExpandBlocks;
    for (uint32_t w = 0; w < S.numWorlds; w++) {
        expand_base[w] = (int32_t)next_block;
        next_block += caches[w].numExpands;
    }
    if (next_block * kIDsPerCache > S.entityCapacity) {
        setError("entity store too small for world construction");
        return false;
    }
    if (!resetForInitPass(ex, 1, expand_base, persist_mark)) return false;
    if (!launch1(ex, ex->initWorlds, wblocks, 128)) return false;
    if (!checkDeviceErrors(ex, "world construction")) return false;
    if (!pullState(ex)) return false;
    S.numEntitySlots = (int32_t)(next_block * kIDsPerCache);
    S.initPass = 2;
    if (!pushState(ex)) return false;

    // ---- phase 4: setupTasks on the device (1 thread)
    if (!launch1(ex, ex->initTasks, 1, 1)) return false;
    if (!pullState(ex)) return false;
    if (!checkDeviceErrors(ex, "setupTasks")) return false;

    // resolve ParallelFor records to kernels
    for (uint32_t n = 0; n < S.numNodes; n++) {
        NodeRecord &r = S.nodes[n];
        if (r.kind != NodeUserParallelFor) continue;
        uint64_t addr = ((uint64_t)r.component << 32) | r.kernelID;
        size_t k = 0;
        for (; k < ex->nodeMetaAddrs.size(); k++) {
            if (ex->nodeMetaAddrs[k] == addr) break;
        }
        if (k == ex->nodeMetaAddrs.size()) {
            setError("taskgraph node " + std::to_string(n) + " has no kernel in the module");
            return false;
        }
        r.kernelID = (uint32_t)k;
    }
    MB2_CUDA(cudaMemcpy(ex->dState->nodes, S.nodes, sizeof(NodeRecord) * S.numNodes,
                        cudaMemcpyHostToDevice));

    // ---- phase 5: bring every table into world order so exported columns are
    // world-major from step 0 (the CPU backend's layout, src/core/state.cpp:576-619)
    for (uint32_t a = 0; a < S.numArchetypes; a++) {
        if (!S.archetypes[a].registered || S.tables[a].isSingleton) continue;
        launchSortArchetype(ex, a, 1, ex->stream);
    }
    MB2_CUDA(cudaStreamSynchronize(ex->stream));
    MB2_CUDA(cudaGetLastError());
    if (!checkDeviceErrors(ex, "initial sort")) return false;
    return true;
}

static void destroyExecutor(Executor *ex)
{
    if (!ex) return;
    cudaSetDevice(ex->gpu);
    if (ex->stream) cudaStreamSynchronize(ex->stream);
    physicsHostDestroy(ex);
    renderHostDestroy(ex);
    sortScratchDestroy(ex);
    for (int a = 0; a < kMaxArchetypes; a++) {
        for (VMRange &r : ex->columnRanges[a]) vmRelease(&r);
        for (VMRange &r : ex->twinRanges[a]) vmRelease(&r);
    }
    vmRelease(&ex->entityRange);
    for (void *p : ex->allocations) cudaFree(p);
    if (ex->hStatus) cudaFreeHost(ex->hStatus);
    if (ex->lib) cudaLibraryUnload(ex->lib);
    if (ex->stream) cudaStreamDestroy(ex->stream);
    free(ex->hState);
    delete ex;
}

// ---- launch graphs -----------------------------------------------------------

static bool enqueueNode(Executor *ex, uint32_t node_idx, cudaStream_t s)
{
    EngineState &S = *ex->hState;
    const NodeRecord &r = S.nodes[node_idx];
    switch (r.kind) {
    case NodeUserParallelFor: {
        const TableDesc &t = S.tables[r.archetype];
        uint64_t threads = (uint64_t)t.capacity * std::max(r.userTag, 1u);
        uint64_t blocks = (threads + 255) / 256;
        uint64_t max_blocks = (uint64_t)ex->numSMs * 8;
        unsigned grid = (unsigned)std::max<uint64_t>(1, std::min(blocks, max_blocks));
        const NodeRecord *drec = &ex->dState->nodes[node_idx];
        void *args[1] = { (void *)&drec };
        MB2_CUDA(cudaLaunchKernel((const void *)ex->nodeKernels[r.kernelID], dim3(grid), dim3(256), args, 0, s));
        return true;
    }
    case NodeSortArchetype:
    case NodeCompactArchetype: {
        int32_t col = 1;
        if (r.kind == NodeSortArchetype) {
            if (r.component >= S.numComponents || S.columnLookup[r.archetype][r.component] < 0) {
                setError("SortArchetypeNode: archetype lacks the sort component");
                return false;
            }
            col = S.columnLookup[r.archetype][r.component];
        }
        launchSortArchetype(ex, r.archetype, col, s);
        return true;
    }
    case NodeClearTmp:
        launchClearTmp(ex, r.archetype, s);
        return true;
    case NodeResetTmpAlloc:
        if (r.userTag == 0xFFFFFFFFu) return true;   // placeholder for an empty query
        launchResetTmpAlloc(ex, s);
        return true;
    case NodeRecycleEntities:
        // IDs are recycled at destroy time through the per-world caches
        // (state.hpp releaseEntityLocked); nothing left to do here.
        return true;
    case NodeRenderPrepare: {
        std::string err;
        if (!renderEnqueuePrepare(ex, s, &err)) {
            setError(err);
            return false;
        }
        return true;
    }
    default:
        if (r.kind >= NodePhysBroadphaseUpdate) {
            std::string err;
            if (!physicsEnqueueNode(ex, r, s, &err)) {
                setError(err);
                return false;
            }
            return true;
        }
        setError("unknown taskgraph node kind " + std::to_string(r.kind));
        return false;
    }
}

static LaunchGraph *buildGraph(Executor *ex, const uint32_t *ids, uint32_t n)
{
    EngineState &S = *ex->hState;
    cudaSetDevice(ex->gpu);
    LaunchGraph *g = new LaunchGraph();
    g->owner = ex;

    physicsBeforeGraphCapture(ex);

    // ---- units of work: one TaskGraph node each, except that a run of consecutive
    // physics nodes is one (internally ordered) unit.  Units keep the simulator's
    // dependency lists (reference: TaskGraphBuilder::build, src/core/taskgraph.cpp:
    // 53-117 -- a dependency can only name an earlier node, so registration order
    // is a topological order); units that do not depend on each other are captured
    // on different streams and become parallel branches of the CUDA graph.
    struct Unit {
        uint32_t first, last;
        bool usesSortScratch;
        std::vector<int> deps;      // unit indices
        int stream = -1;
        cudaEvent_t done = nullptr;
    };
    std::vector<Unit> units;
    std::vector<int> unit_of_node(S.numNodes, -1);
    bool ok = true;
    for (uint32_t i = 0; i < n && ok; i++) {
        if (ids[i] >= S.numTaskGraphs) {
            setError("taskgraph id out of range");
            ok = false;
            break;
        }
        const size_t first_unit_of_graph = units.size();
        for (uint32_t node = 0; node < S.numNodes; node++) {
            if (S.nodes[node].taskgraph != ids[i]) continue;
            auto is_phys = [&](uint32_t k) {
                return S.nodes[k].kind >= NodePhysBroadphaseUpdate && S.nodes[k].kind < NodeRenderPrepare;
            };
            Unit u;
            u.first = u.last = node;
            if (is_phys(node)) {
                while (u.last + 1 < S.numNodes && S.nodes[u.last + 1].taskgraph == ids[i] && is_phys(u.last + 1)) {
                    u.last++;
                }
            }
            u.usesSortScratch = false;
            for (uint32_t k = u.first; k <= u.last; k++) {
                const uint32_t kind = S.nodes[k].kind;
                if (kind == NodeSortArchetype || kind == NodeCompactArchetype || kind == NodePhysFindCandidates ||
                        kind == NodeRenderPrepare) {
                    u.usesSortScratch = true;     // one scratch block serves every sort: keep them in line
                }
                unit_of_node[k] = (int)units.size();
            }
            for (uint32_t k = u.first; k <= u.last; k++) {
                const NodeRecord &r = S.nodes[k];
                for (uint32_t d = 0; d < r.numDeps && d < (uint32_t)kMaxNodeDeps; d++) {
                    const uint32_t dep_node = r.deps[d];
                    if (dep_node >= S.numNodes || unit_of_node[dep_node] < 0) continue;
                    const int du = unit_of_node[dep_node];
                    if (du == (int)units.size() || du < (int)first_unit_of_graph) continue;
                    if (std::find(u.deps.begin(), u.deps.end(), du) == u.deps.end()) u.deps.push_back(du);
                }
            }
            if (u.usesSortScratch) {
                for (int k = (int)units.size() - 1; k >= (int)first_unit_of_graph; k--) {
                    if (units[k].usesSortScratch) {
                        if (std::find(u.deps.begin(), u.deps.end(), k) == u.deps.end()) u.deps.push_back(k);
                        break;
                    }
                }
            }
            // task graphs of one launch graph run one after the other
            if (u.deps.empty() && first_unit_of_graph > 0) {
                for (size_t k = 0; k < first_unit_of_graph; k++) u.deps.push_back((int)k);
            }
            node = u.last;
            units.push_back(std::move(u));
        }
    }
    const bool branches = envU64("MADRONA_B200_GRAPH_BRANCHES", 1) != 0;

    cudaError_t e = cudaStreamBeginCapture(ex->stream, cudaStreamCaptureModeThreadLocal);
    if (e != cudaSuccess) {
        setError(std::string("cudaStreamBeginCapture: ") + cudaGetErrorString(e));
        delete g;
        return nullptr;
    }
    // stream 0 = the capture origin; side streams join the capture through events
    std::vector<cudaStream_t> streams { ex->stream };
    std::vector<int> tail { -1 };              // last unit placed on each stream
    cudaEvent_t origin_start = nullptr;
    cudaEventCreateWithFlags(&origin_start, cudaEventDisableTiming);
    cudaEventRecord(origin_start, ex->stream);
    std::vector<cudaEvent_t> events { origin_start };

    for (size_t ui = 0; ui < units.size() && ok; ui++) {
        Unit &u = units[ui];
        int chosen = -1;
        if (!branches) {
            chosen = 0;
        } else {
            // continue on the stream of a dependency that is still that stream's tail
            for (int d : u.deps) {
                if (tail[units[d].stream] == d) {
                    chosen = units[d].stream;
                    break;
                }
            }
            if (chosen < 0 && tail[0] == -1) chosen = 0;
            if (chosen < 0) {
                // a free side stream (its tail is an ancestor everybody already waited for) or a new one
                cudaStream_t ns = nullptr;
                if (cudaStreamCreateWithFlags(&ns, cudaStreamNonBlocking) != cudaSuccess) {
                    chosen = 0;
                } else {
                    streams.push_back(ns);
                    tail.push_back(-1);
                    chosen = (int)streams.size() - 1;
                    cudaStreamWaitEvent(ns, origin_start, 0);
                }
            }
        }
        u.stream = chosen;
        cudaStream_t cs = streams[chosen];
        for (int d : u.deps) {
            if (units[d].stream != chosen || !branches) {
                if (units[d].stream != chosen) cudaStreamWaitEvent(cs, units[d].done, 0);
            }
        }
        if (u.last > u.first) {
            std::string perr;
            ok = physicsEnqueueNodes(ex, &S.nodes[u.first], u.last - u.first + 1, cs, &perr);
            if (!ok) setError(perr);
        } else {
            ok = enqueueNode(ex, u.first, cs);
        }
        cudaEventCreateWithFlags(&u.done, cudaEventDisableTiming);
        cudaEventRecord(u.done, cs);
        events.push_back(u.done);
        tail[chosen] = (int)ui;
    }
    // join every side stream back into the origin
    for (size_t si = 1; si < streams.size(); si++) {
        if (tail[si] >= 0) cudaStreamWaitEvent(ex->stream, units[tail[si]].done, 0);
    }
    if (ok) launchStatusCopy(ex, ex->stream);
    e = cudaStreamEndCapture(ex->stream, &g->graph);
    for (cudaEvent_t ev : events) cudaEventDestroy(ev);
    for (size_t si = 1; si < streams.size(); si++) cudaStreamDestroy(streams[si]);
    g->numBranches = (int64_t)streams.size();
    if (!ok || e != cudaSuccess) {
        if (ok) setError(std::string("cudaStreamEndCapture: ") + cudaGetErrorString(e));
        if (g->graph) cudaGraphDestroy(g->graph);
        delete g;
        return nullptr;
    }
    size_t num_nodes = 0;
    cudaGraphGetNodes(g->graph, nullptr, &num_nodes);
    std::vector<cudaGraphNode_t> nodes(num_nodes);
    if (num_nodes) cudaGraphGetNodes(g->graph, nodes.data(), &num_nodes);
    for (cudaGraphNode_t nd : nodes) {
        cudaGraphNodeType ty;
        if (cudaGraphNodeGetType(nd, &ty) == cudaSuccess && ty == cudaGraphNodeTypeKernel)
            g->numKernels++;
    }
    e = cudaGraphInstantiate(&g->exec, g->graph, 0);
    if (e != cudaSuccess) {
        setError(std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e));
        cudaGraphDestroy(g->graph);
        delete g;
        return nullptr;
    }
    return g;
}

// ---- per-node profiling ------------------------------------------------------

struct NodeProfile {
    double ms = 0;
    double bytes = 0;
    double rows = 0;
    int64_t launches = 0;
    int64_t samples = 0;
};

static int64_t profileNodes(Executor *ex, const uint32_t *ids, uint32_t n, uint32_t reps,
                            std::string *out)
{
    EngineState &S = *ex->hState;
    cudaSetDevice(ex->gpu);
    std::vector<uint32_t> order;
    for (uint32_t i = 0; i < n; i++) {
        if (ids[i] >= S.numTaskGraphs) {
            setError("taskgraph id out of range");
            return -1;
        }
        for (uint32_t node = 0; node < S.numNodes; node++) {
            if (S.nodes[node].taskgraph == ids[i]) order.push_back(node);
        }
    }
    std::vector<NodeProfile> prof(order.size());
    std::vector<cudaEvent_t> ev(order.size() + 1), ev_start(order.size());
    for (auto &e : ev) cudaEventCreate(&e);
    for (auto &e : ev_start) cudaEventCreate(&e);
    // released on every exit path
    struct EventGuard {
        std::vector<cudaEvent_t> &a, &b;
        ~EventGuard() {
            for (auto &e : a) if (e) { cudaEventDestroy(e); e = nullptr; }
            for (auto &e : b) if (e) { cudaEventDestroy(e); e = nullptr; }
        }
    } guard { ev, ev_start };
    std::vector<TableDesc> tables(S.numArchetypes);
    // same pre-capture refresh as buildLaunchGraph (sphere narrowphase selection)
    physicsBeforeGraphCapture(ex);

    for (uint32_t rep = 0; rep < reps + 1; rep++) {   // rep 0 = warm-up
        // snapshot row counts / dirty flags as they are at the start of the step
        cudaStreamSynchronize(ex->stream);
        cudaMemcpy(tables.data(), ex->dState->tables, sizeof(TableDesc) * S.numArchetypes,
                   cudaMemcpyDeviceToHost);
        cudaEventRecord(ev[0], ex->stream);
        for (size_t k = 0; k < order.size(); k++) {
            const NodeRecord &nr = S.nodes[order[k]];
            if (nr.kind == NodeSortArchetype || nr.kind == NodeCompactArchetype) {
                // whether this sort will actually run (and over how many rows) is only
                // known once the preceding nodes have executed: look now (the extra
                // sync sits between two event pairs, it is not timed)
                cudaStreamSynchronize(ex->stream);
                cudaMemcpy(&tables[nr.archetype], &ex->dState->tables[nr.archetype], sizeof(TableDesc),
                           cudaMemcpyDeviceToHost);
            }
            cudaEventRecord(ev_start[k], ex->stream);
            if (!enqueueNode(ex, order[k], ex->stream)) return -1;
            cudaEventRecord(ev[k + 1], ex->stream);
        }
        if (cudaStreamSynchronize(ex->stream) != cudaSuccess) {
            setError(std::string("profile step failed: ") + cudaGetErrorString(cudaGetLastError()));
            return -1;
        }
        if (rep == 0) continue;
        for (size_t k = 0; k < order.size(); k++) {
            float ms = 0;
            cudaEventElapsedTime(&ms, ev_start[k], ev[k + 1]);
            const NodeRecord &r = S.nodes[order[k]];
            NodeProfile &p = prof[k];
            p.ms += ms;
            p.samples++;
            const TableDesc &t = tables[r.archetype < S.numArchetypes ? r.archetype : 0];
            double rows = t.numRows, bytes = 0;
            if (r.kind == NodeUserParallelFor) {
                double per_row = 4;   // WorldID
                for (int c = 0; c < r.numCols; c++) per_row += t.columnBytes[r.cols[c]];
                bytes = rows * per_row;
            } else if (r.kind == NodeSortArchetype || r.kind == NodeCompactArchetype) {
                int col = r.kind == NodeSortArchetype ? S.columnLookup[r.archetype][r.component] : 1;
                bool active = col != 1 || t.needsSort;
                if (active) {
                    // SURVEY.md 8(d): 4 (histogram) + 16 P (key+idx in/out per pass) +
                    // 4 (idx read) + sum 2 b_c (payload once in, once out) + 8 (remap + offsets)
                    double per_row = 4 + 16.0 * sortNumPasses(ex, col) + 4 + 8;
                    for (int c = 0; c < t.numColumns; c++) {
                        if (c != col) per_row += 2.0 * t.columnBytes[c];
                    }
                    bytes = rows * per_row;
                } else {
                    rows = 0;
                }
            } else if (r.kind >= NodePhysBroadphaseUpdate) {
                const char *nm;
                int64_t prow = 0;
                bytes = (double)physicsNodeBytes(ex, r, &nm, &prow);
                rows = (double)prow;
            }
            p.bytes += bytes;
            p.rows += rows;
        }
    }

    static const char *kind_names[] = { "parallel_for", "sort_archetype", "compact_archetype",
                                        "clear_tmp", "reset_tmp_alloc", "recycle_entities" };
    std::string js = "[";
    for (size_t k = 0; k < order.size(); k++) {
        const NodeRecord &r = S.nodes[order[k]];
        const NodeProfile &p = prof[k];
        const char *kn = r.kind < 6 ? kind_names[r.kind] : "physics";
        if (r.kind >= NodePhysBroadphaseUpdate) {
            int64_t rows;
            physicsNodeBytes(ex, r, &kn, &rows);
        }
        std::string name = kn;
        if (r.kind == NodeUserParallelFor && r.kernelID < ex->jit.nodeKernels.size()) {
            // keep the mangled system name readable: take the part after "_Z" of the NTTP
            const std::string &m = ex->jit.nodeKernels[r.kernelID];
            size_t a = m.find("XadL_Z");
            if (a != std::string::npos) {
                size_t b = m.find("ERS", a);
                name += ":" + m.substr(a + 6, b == std::string::npos ? 32 : b - a - 6);
            }
        }
        double s = p.samples ? 1.0 / (double)p.samples : 0.0;
        char buf[512];
        snprintf(buf, sizeof(buf),
                 "%s{\"node\": %u, \"kind\": \"%s\", \"archetype\": %u, \"ms\": %.6f, "
                 "\"rows\": %.1f, \"bytes\": %.1f}",
                 k ? ", " : "", order[k], name.c_str(), r.archetype, p.ms * s, p.rows * s, p.bytes * s);
        js += buf;
    }
    js += "]";
    *out = js;
    return (int64_t)js.size();
}

}

using namespace mb2;

// driver entry points through the runtime (no link dependency on libcuda)
template <typename Fn>
static Fn driverFn(const char *name)
{
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint(name, &fn, cudaEnableDefault, &q) != cudaSuccess) return nullptr;
    return (Fn)fn;
}

extern "C" {

int64_t mb2_profile_nodes(mb2_executor *exec, const uint32_t *taskgraph_ids,
                          uint32_t num_taskgraphs, uint32_t reps,
                          char *json_out, uint64_t json_capacity)
{
    g_last_error.clear();
    std::string js;
    int64_t n = profileNodes((Executor *)exec, taskgraph_ids, num_taskgraphs, reps, &js);
    if (n < 0) return -1;
    if (json_out && json_capacity > 0) {
        size_t c = std::min<size_t>(js.size(), json_capacity - 1);
        memcpy(json_out, js.data(), c);
        json_out[c] = 0;
    }
    return n;
}


const char *mb2_last_error(void) { return g_last_error.c_str(); }

const char *mb2_version(void) { return "madrona_b200 0.1 (sm_100a)"; }

int mb2_init_cuda(int gpu_id)
{
    cudaError_t e = cudaSetDevice(gpu_id);
    if (e != cudaSuccess) {
        setError(std::string("cudaSetDevice: ") + cudaGetErrorString(e));
        return 1;
    }
    cudaFree(nullptr);
    return 0;
}

int mb2_init_cuda_ctx(int gpu_id, void **cu_context_out)
{
    if (mb2_init_cuda(gpu_id) != 0) return 1;
    if (cu_context_out) {
        *cu_context_out = nullptr;
        auto retain = driverFn<int (*)(void **, int)>("cuDevicePrimaryCtxRetain");
        auto dev_get = driverFn<int (*)(int *, int)>("cuDeviceGet");
        int dev = 0;
        if (!retain || !dev_get || dev_get(&dev, gpu_id) != 0 || retain(cu_context_out, dev) != 0) {
            setError("cuDevicePrimaryCtxRetain failed");
            return 1;
        }
    }
    return 0;
}

int mb2_device_of_context(void *cu_context)
{
    int cur = 0;
    cudaGetDevice(&cur);
    if (!cu_context) return cur;
    auto push = driverFn<int (*)(void *)>("cuCtxPushCurrent");
    auto pop = driverFn<int (*)(void **)>("cuCtxPopCurrent");
    auto get_dev = driverFn<int (*)(int *)>("cuCtxGetDevice");
    if (!push || !pop || !get_dev || push(cu_context) != 0) return cur;
    int dev = cur;
    get_dev(&dev);
    void *old = nullptr;
    pop(&old);
    return dev;
}

mb2_executor *mb2_executor_create(const mb2_state_config *state_cfg,
                                  const mb2_compile_config *compile_cfg,
                                  int gpu_id, const mb2_render_config *render_cfg)
{
    g_last_error.clear();
    if (!state_cfg || !compile_cfg) {
        setError("null config");
        return nullptr;
    }
    Executor *ex = new Executor();
    ex->gpu = gpu_id;
    if (!createExecutor(ex, state_cfg, compile_cfg, render_cfg)) {
        std::string keep = g_last_error;
        destroyExecutor(ex);
        g_last_error = keep;
        return nullptr;
    }
    return (mb2_executor *)ex;
}

void mb2_executor_destroy(mb2_executor *exec) { destroyExecutor((Executor *)exec); }

// stat_name is part of the reference's signature; this executor keeps no per-graph statistics
mb2_launch_graph *mb2_build_launch_graph(mb2_executor *exec, const uint32_t *taskgraph_ids,
                                         uint32_t num_taskgraphs, const char * /*stat_name*/)
{
    g_last_error.clear();
    return (mb2_launch_graph *)buildGraph((Executor *)exec, taskgraph_ids, num_taskgraphs);
}

mb2_launch_graph *mb2_build_launch_graph_all(mb2_executor *exec)
{
    Executor *ex = (Executor *)exec;
    std::vector<uint32_t> ids(ex->hState->numTaskGraphs);
    for (uint32_t i = 0; i < ids.size(); i++) ids[i] = i;
    return mb2_build_launch_graph(exec, ids.data(), (uint32_t)ids.size(), "all");
}

mb2_launch_graph *mb2_build_render_graph(mb2_executor *exec)
{
    g_last_error.clear();
    Executor *ex = (Executor *)exec;
    std::string err;
    LaunchGraph *g = physicsBuildRenderGraph(ex, &err);
    if (!g) setError(err);
    return (mb2_launch_graph *)g;
}

void mb2_launch_graph_destroy(mb2_launch_graph *graph)
{
    LaunchGraph *g = (LaunchGraph *)graph;
    if (!g) return;
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->graph) cudaGraphDestroy(g->graph);
    delete g;
}

int mb2_run_async(mb2_executor *exec, mb2_launch_graph *graph, void *cuda_stream)
{
    Executor *ex = (Executor *)exec;
    LaunchGraph *g = (LaunchGraph *)graph;
    if (!ex || !g) {
        setError("null executor or launch graph");
        return 1;
    }
    // an idle executor can act on the status its last graph published (table growth)
    if ((cudaStream_t)cuda_stream != ex->stream && ex->tableGrowth &&
            cudaStreamQuery((cudaStream_t)cuda_stream) == cudaSuccess && cudaStreamQuery(ex->stream) == cudaSuccess) {
        if (ex->hStatus[0] == 0 && !growTablesFromStatus(ex)) return 1;
    }
    cudaError_t e = cudaGraphLaunch(g->exec, (cudaStream_t)cuda_stream);
    if (e != cudaSuccess) {
        setError(std::string("cudaGraphLaunch: ") + cudaGetErrorString(e));
        return 1;
    }
    return 0;
}

int mb2_run(mb2_executor *exec, mb2_launch_graph *graph)
{
    Executor *ex = (Executor *)exec;
    if (mb2_run_async(exec, graph, ex ? ex->stream : nullptr) != 0) return 1;
    cudaError_t e = cudaStreamSynchronize(ex->stream);
    if (e != cudaSuccess) {
        setError(std::string("step failed: ") + cudaGetErrorString(e));
        return 1;
    }
    if (ex->hStatus[0] != 0) {
        setError("step failed: " + describeErrors(ex->hStatus[0], ex->hStatus[1]));
        return 2;
    }
    if (!growTablesFromStatus(ex)) return 1;
    return 0;
}

void *mb2_get_exported(const mb2_executor *exec, int64_t slot)
{
    const Executor *ex = (const Executor *)exec;
    if (!ex || slot < 0 || slot >= kMaxExports) return nullptr;
    return ex->exported[slot];
}

int64_t mb2_get_exported_num_rows(mb2_executor *exec, int64_t slot)
{
    Executor *ex = (Executor *)exec;
    if (!ex || slot < 0 || slot >= kMaxExports || !ex->exported[slot]) return -1;
    int32_t n = 0;
    cudaStreamSynchronize(ex->stream);
    cudaMemcpy(&n, &ex->dState->tables[ex->exportArchetype[slot]].numRows, sizeof(n),
               cudaMemcpyDeviceToHost);
    return n;
}

int64_t mb2_get_exported_row_bytes(const mb2_executor *exec, int64_t slot)
{
    const Executor *ex = (const Executor *)exec;
    if (!ex || slot < 0 || slot >= kMaxExports || !ex->exported[slot]) return -1;
    return ex->exportRowBytes[slot];
}

int64_t mb2_launch_graph_num_kernels(const mb2_launch_graph *graph)
{
    return graph ? ((const LaunchGraph *)graph)->numKernels : -1;
}

void *mb2_render_debug_hits(mb2_executor *exec)
{
    return exec ? renderDebugHitBuffer((Executor *)exec) : nullptr;
}

void *mb2_render_debug_buffer(mb2_executor *exec, int which, int64_t *max_instances_per_world)
{
    int64_t stride = 0;
    void *p = exec ? renderDebugBuffer((Executor *)exec, which, &stride) : nullptr;
    if (max_instances_per_world) *max_instances_per_world = stride;
    return p;
}

int64_t mb2_launch_graph_num_branches(const mb2_launch_graph *graph)
{
    return graph ? ((const LaunchGraph *)graph)->numBranches : -1;
}

void *mb2_executor_stream(mb2_executor *exec)
{
    return exec ? (void *)((Executor *)exec)->stream : nullptr;
}

int mb2_jit_precompile(const mb2_compile_config *cc)
{
    g_last_error.clear();
    std::vector<std::string> sources, flags;
    for (uint32_t i = 0; i < cc->num_user_sources; i++) sources.push_back(cc->user_sources[i]);
    for (uint32_t i = 0; i < cc->num_user_compile_flags; i++) flags.push_back(cc->user_compile_flags[i]);
    JitModule m;
    std::string err;
    if (!jitCompile(sources, flags, (int)cc->opt_mode, &m, &err)) {
        setError(err);
        return 1;
    }
    return 0;
}

}
