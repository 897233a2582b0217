// mb2_state.h -- device-resident engine state shared by three compilers:
//   * g++       (host side of libmadrona_b200.so, engine.cpp)
//   * nvcc      (ahead-of-time engine kernels: sort / physics / render, *.cu)
//   * NVRTC     (the simulator's own sources + madrona_b200/device/madrona/*.hpp)
// It therefore uses only fixed-width builtin types and no std headers.
//
// Data model (replaces the reference's StateManager / Table / TaskGraph device
// structures: src/mw/device/include/madrona/state.hpp:235-256, table.hpp:18-40,
// src/mw/device/taskgraph.cpp): one global SoA table per archetype holding the
// rows of *all* worlds, rows grouped by world after a world sort, plus
// worldOffsets/worldCounts.  Column 0 = Entity, column 1 = WorldID, user
// components from 2 in registration order (reference: src/mw/device/state.cpp
// :269-341).  There is no megakernel: every TaskGraph node is a NodeRecord that
// the host turns into one (or a few) kernel nodes of a CUDA graph.
#pragma once

namespace mb2 {

typedef unsigned char u8;
typedef unsigned short u16;
typedef unsigned int u32;
typedef int i32;
typedef short i16;
typedef unsigned long long u64;
typedef long long i64;

constexpr int kMaxColumns = 48;        // per archetype, including Entity + WorldID
constexpr int kMaxArchetypes = 96;
constexpr int kMaxComponents = 320;
constexpr int kMaxBundles = 48;
constexpr int kMaxBundleComponents = 32;
constexpr int kMaxExports = 64;
constexpr int kMaxNodes = 1024;
constexpr int kMaxNodeCols = 16;
constexpr int kMaxNodeDeps = 8;
constexpr int kMaxTaskGraphs = 8;
constexpr int kIDsPerCache = 64;       // reference: include/madrona/impl/id_map.hpp:132
constexpr i32 kIDSentinel = (i32)0xFFFFFFFF;
constexpr u32 kBundleMask = 0x80000000u;  // reference: include/madrona/state.hpp:401
constexpr u32 kUnassignedType = 0xFFFFFFFFu;

struct ComponentInfo {
    u32 numBytes;
    u32 alignment;
};

// Filled on the device by ECSRegistry::registerArchetype (1 thread), read by
// the host to size and allocate the table.
struct ArchetypeInfo {
    u32 registered;
    u32 numUserComponents;               // after bundle flattening
    u32 componentIDs[kMaxColumns];       // user components only (col = i + 2)
    u32 flags;
    i32 maxPerWorld;                     // 0 => dynamic
    u32 isSingleton;
    u32 singletonOrder;                  // n-th registerSingleton call
};

struct BundleInfo {
    u32 registered;
    u32 numComponents;
    u32 componentIDs[kMaxBundleComponents];
};

struct ExportInfo {
    u32 used;
    u32 archetype;
    u32 component;
    u32 pad;
};

struct alignas(16) TableDesc {
    void *columns[kMaxColumns];
    u32 columnBytes[kMaxColumns];
    i32 numColumns;
    i32 numRows;          // live rows (append with atomicAdd)
    i32 capacity;         // rows backed by memory
    i32 maxPerWorld;
    i32 *worldOffsets;    // [numWorlds]
    i32 *worldCounts;     // [numWorlds]
    u32 needsSort;
    u32 isSingleton;
    u32 highWater;        // max numRows ever seen (host growth heuristic)
    u32 pad;
};

// 12-byte entity slot.  While live: {archetype,row}; while free: the IDMap
// FreeNode {subNext, globalNext} (reference: include/madrona/impl/id_map.hpp
// :37-48 -- the same union trick, so the CPU oracle's ID sequence can be
// reproduced exactly).
struct EntitySlot {
    i32 a;    // Loc.archetype | FreeNode.subNext
    i32 b;    // Loc.row       | FreeNode.globalNext
    u32 gen;
};

// Per-world entity-ID cache == IDMap::Cache (id_map.hpp:23-35) + a spin lock
// because several rows of one world may create entities concurrently here.
struct IDCache {
    i32 freeHead;
    i32 numFree;
    i32 overflowHead;
    i32 numOverflow;
    i32 lock;
    i32 numExpands;       // 64-ID blocks this world took from expand() (init dry run)
    i32 expandBase;       // first block index assigned to this world (init pass 2)
    i32 pad;
};

enum NodeKind : u32 {
    NodeUserParallelFor = 0,
    NodeSortArchetype = 1,
    NodeCompactArchetype = 2,
    NodeClearTmp = 3,
    NodeResetTmpAlloc = 4,
    NodeRecycleEntities = 5,
    // engine-owned systems (ahead-of-time kernels)
    NodePhysBroadphaseUpdate = 16,   // leaf AABB update + refit
    NodePhysBVHRebuild = 17,
    NodePhysFindCandidates = 18,
    NodePhysSubstepBegin = 19,
    NodePhysNarrowphase = 20,
    NodePhysSolvePositions = 21,
    NodePhysSetVelocities = 22,
    NodePhysSolveVelocities = 23,
    NodePhysClearContacts = 24,
    NodePhysClearCandidates = 25,
    NodePhysTGSVelocities = 26,    // tgs::integrateVelocities (src/physics/tgs.cpp:92-142)
    NodePhysTGSPositions = 27,     // tgs::integratePositions (tgs.cpp:171-195)
    NodeRenderPrepare = 32,
};

struct NodeRecord {
    u32 kind;
    u32 taskgraph;
    u32 kernelID;          // index into the JIT module's node-kernel list (user nodes)
    u32 archetype;
    u32 component;         // sort key component
    i32 numCols;
    i32 cols[kMaxNodeCols];
    u32 numDeps;
    u32 deps[kMaxNodeDeps];
    u32 userTag;
};

struct PhysicsState;   // physics_state.h
struct RenderState;

struct EngineState {
    // ---- config
    u32 numWorlds;
    u32 numTaskGraphs;
    u32 numExported;
    u32 worldDataStride;
    char *worldData;
    void *userConfig;
    void *worldInits;
    u32 worldInitBytes;
    u32 initPass;          // 0 = dry run (count ID blocks), 1 = real
    u32 worldDataNeeded;   // sizeof(WorldT), reported by the device entry
    u32 worldDataAlignNeeded;

    // ---- registry (written by device-side registerTypes, 1 thread)
    u32 numComponents;
    u32 numArchetypes;
    u32 numBundles;
    u32 numSingletons;
    ComponentInfo components[kMaxComponents];
    ArchetypeInfo archetypes[kMaxArchetypes];
    BundleInfo bundles[kMaxBundles];
    ExportInfo exports[kMaxExports];

    // ---- storage (allocated by the host after registerTypes)
    TableDesc tables[kMaxArchetypes];
    i16 columnLookup[kMaxArchetypes][kMaxComponents];   // -1 => absent

    // ---- entities
    EntitySlot *entitySlots;
    i32 entityCapacity;
    i32 numEntitySlots;              // expand() bump pointer
    u64 freeHead;                    // {gen:32 | head:32}, global free list
    IDCache *idCaches;               // [numWorlds]
    i32 initExpandBlocks;            // blocks consumed before world ctors (singletons)

    // ---- allocators
    char *tmpArena;
    u64 tmpCapacity;
    u64 tmpOffset;
    char *persistArena;
    u64 persistCapacity;
    u64 persistOffset;

    // ---- task graphs (written by device-side setupTasks, 1 thread)
    u32 numNodes;
    u32 curTaskGraph;
    NodeRecord nodes[kMaxNodes];

    // ---- status
    u32 errorFlags;
    u32 errorArchetype;

    // ---- engine-owned systems
    PhysicsState *physics;
    RenderState *render;
};

enum ErrorFlags : u32 {
    ErrTableOverflow = 1u << 0,
    ErrEntityOverflow = 1u << 1,
    ErrTmpOverflow = 1u << 2,
    ErrPersistOverflow = 1u << 3,
    ErrTooManyNodes = 1u << 4,
    ErrRegistry = 1u << 5,
    ErrPhysicsOverflow = 1u << 6,
};

}
