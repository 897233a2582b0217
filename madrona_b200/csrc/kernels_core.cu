// kernels_core.cu -- small engine-owned TaskGraph nodes (reference:
// src/mw/device/taskgraph_utils.cpp:176-223 ClearTmpNodeBase / ResetTmpAllocNode)
// and executor bookkeeping kernels.
#include "engine.hpp"

namespace mb2 {

// ClearTmpNode: drop every row of a temporary archetype (numRows.exchange(0)
// in the reference) and zero its per-world counts.
__global__ void clearTmpKernel(EngineState *S, uint32_t archetype)
{
    TableDesc &t = S->tables[archetype];
    const int32_t W = (int32_t)S->numWorlds;
    for (int32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < W; w += gridDim.x * blockDim.x) {
        t.worldCounts[w] = 0;
        t.worldOffsets[w] = 0;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if ((uint32_t)t.numRows > t.highWater) t.highWater = (uint32_t)t.numRows;
        t.numRows = 0;
        t.needsSort = 0;
    }
}

__global__ void resetTmpAllocKernel(EngineState *S)
{
    S->tmpOffset = 0;
}

// Last node of every launch graph: publish error flags to pinned host memory.
__global__ void statusCopyKernel(EngineState *S, uint32_t *host_status)
{
    host_status[0] = S->errorFlags;
    host_status[1] = S->errorArchetype;
    // peak row count of every table during this graph (the host grows tables between steps)
    for (uint32_t a = threadIdx.x; a < S->numArchetypes; a += blockDim.x) {
        TableDesc &t = S->tables[a];
        const uint32_t rows = (uint32_t)max(t.numRows, 0);
        host_status[2 + a] = rows > t.highWater ? rows : t.highWater;
        t.highWater = rows;
    }
}

// Singleton archetypes: one row per world, row == world, created at
// registration time by the reference (include/madrona/state.inl:163-179);
// entity IDs follow the CPU backend's init cache: order * W + world.
__global__ void fillSingletonsKernel(EngineState *S)
{
    const int32_t W = (int32_t)S->numWorlds;
    for (uint32_t a = 0; a < S->numArchetypes; a++) {
        const ArchetypeInfo &info = S->archetypes[a];
        if (!info.registered || !info.isSingleton) continue;
        TableDesc &t = S->tables[a];
        for (int32_t w = blockIdx.x * blockDim.x + threadIdx.x; w < W; w += gridDim.x * blockDim.x) {
            int32_t id = (int32_t)info.singletonOrder * W + w;
            ((int32_t *)t.columns[0])[2 * w] = 0;        // gen
            ((int32_t *)t.columns[0])[2 * w + 1] = id;
            ((int32_t *)t.columns[1])[w] = w;
            t.worldOffsets[w] = w;
            t.worldCounts[w] = 1;
            S->entitySlots[id].a = (int32_t)a;
            S->entitySlots[id].b = w;
            S->entitySlots[id].gen = 0;
        }
    }
}

void launchClearTmp(Executor *ex, uint32_t archetype, cudaStream_t s)
{
    int grid = (int)std::min<uint32_t>((ex->hState->numWorlds + 255) / 256, (uint32_t)ex->numSMs * 2);
    clearTmpKernel<<<std::max(grid, 1), 256, 0, s>>>(ex->dState, archetype);
}

void launchResetTmpAlloc(Executor *ex, cudaStream_t s)
{
    resetTmpAllocKernel<<<1, 1, 0, s>>>(ex->dState);
}

void launchStatusCopy(Executor *ex, cudaStream_t s)
{
    statusCopyKernel<<<1, 32, 0, s>>>(ex->dState, ex->hStatus);
}

void launchFillSingletons(Executor *ex, cudaStream_t s)
{
    int grid = (int)std::min<uint32_t>((ex->hState->numWorlds + 255) / 256, (uint32_t)ex->numSMs * 2);
    fillSingletonsKernel<<<std::max(grid, 1), 256, 0, s>>>(ex->dState);
}

}
