// engine.hpp -- host-side executor state behind the C ABI (include/madrona_b200.h).
#pragma once

#include <cuda_runtime.h>
#include <cstdint>
#include <string>
#include <vector>

#include "mb2_state.h"
#include "jit.hpp"
#include "vm_alloc.hpp"

namespace mb2 {

struct SortScratch;   // kernels_sort.cu
struct PhysicsHost;   // kernels_physics.cu
struct RenderHost;    // kernels_render.cu

struct Executor {
    int gpu = 0;
    int numSMs = 148;
    cudaStream_t stream = nullptr;

    JitModule jit;
    cudaLibrary_t lib = nullptr;
    cudaKernel_t initECS = nullptr, initWorlds = nullptr, initTasks = nullptr;
    std::vector<cudaKernel_t> nodeKernels;
    std::vector<uint64_t> nodeMetaAddrs;

    EngineState *dState = nullptr;     // device
    EngineState *hState = nullptr;     // host mirror (registry, nodes, table descs)
    uint32_t *hStatus = nullptr;       // pinned: [0] errorFlags, [1] errorArchetype

    std::vector<void *> allocations;   // cudaMalloc'd blocks owned by the executor
    void *exported[kMaxExports] = {};
    uint32_t exportArchetype[kMaxExports] = {};
    uint32_t exportRowBytes[kMaxExports] = {};

    SortScratch *sortScratch = nullptr;
    PhysicsHost *physics = nullptr;
    RenderHost *render = nullptr;

    uint64_t rowsPerWorldHint = 64;

    // ---- growable storage (vm_alloc.hpp): dynamic archetypes' columns and their sort
    // twins, the sort's key / index / look-back scratch and the entity store keep their
    // base address and get more physical memory between steps
    bool tableGrowth = true;                                   // MADRONA_B200_TABLE_GROWTH
    std::vector<VMRange> columnRanges[kMaxArchetypes];         // [archetype][column]; empty: fixed table
    std::vector<VMRange> twinRanges[kMaxArchetypes];
    VMRange entityRange;
};

// status block published by the last kernel of every launch graph (pinned host memory)
constexpr int kStatusWords = 2 + kMaxArchetypes;   // errorFlags, errorArchetype, peak rows per table

struct LaunchGraph {
    Executor *owner = nullptr;
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    int64_t numKernels = 0;
    int64_t numBranches = 1;   // capture streams used (parallel branches of independent nodes)
};

void setError(const std::string &msg);

// unsigned environment variable, `dflt` when unset or empty
uint64_t envU64(const char *name, uint64_t dflt);

// cudaMalloc'd block owned by the executor (freed with it), zeroed on ex->stream unless
// `zero` is false; a zero-byte request gets 16 bytes.  On failure: setError and false.
bool devAlloc(Executor *ex, void **ptr, size_t bytes, bool zero = true);

// ---- ahead-of-time engine kernels (kernels_core.cu / kernels_sort.cu) -----
void launchClearTmp(Executor *ex, uint32_t archetype, cudaStream_t s);
void launchResetTmpAlloc(Executor *ex, cudaStream_t s);
void launchStatusCopy(Executor *ex, cudaStream_t s);
void launchFillSingletons(Executor *ex, cudaStream_t s);

bool sortScratchCreate(Executor *ex, std::string *err);
void sortScratchDestroy(Executor *ex);
// Stable sort of `archetype` by the low bits of column `col`; col==1 (WorldID)
// additionally drops rows with key -1 and rebuilds worldOffsets/worldCounts.
void launchSortArchetype(Executor *ex, uint32_t archetype, int32_t col, cudaStream_t s);
int sortNumPasses(Executor *ex, int32_t col);
// the sort's key / index / look-back scratch must cover the largest table
bool sortScratchEnsure(Executor *ex, int32_t max_rows, std::string *err);
// grow a dynamic table to new_capacity rows (columns, twins, entity store, sort scratch)
bool growTable(Executor *ex, uint32_t archetype, int64_t new_capacity, std::string *err);

}
