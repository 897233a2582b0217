// kernels_physics.cu -- hot system 2: rigid-body physics for every world of the
// batch, as ahead-of-time sm_100a kernels over the ECS SoA columns.
//
// WHAT is computed follows the reference's CPU backend so results can be
// compared number for number (SURVEY.md 9.5-9.7):
//   broadphase  src/physics/broadphase.cpp:47-285 (top-down 4-wide midpoint
//               build, only on reset), :440-485 (leaf boxes grown by motion),
//               :550-647 (grow-only refit), :930-993 (pair emission order)
//   narrowphase src/physics/narrowphase.cpp:151-223, 339-365, 464-567, 617-652,
//               659-768, 771-1138, 1214-1514, 1682-1899 (scalar SAT path --
//               the warp-cooperative variant is dead code there, SURVEY F4)
//   XPBD        src/physics/xpbd.cpp:100-185, 454-550, 607-718, 720-779,
//               916-1052
// HOW it runs is new:
//   * candidates and contacts are flat per-world segments written in the CPU
//     backend's iteration order by warp-per-world kernels (count -> warp scan ->
//     emit; ballot-compaction for contacts).  The reference GPU backend
//     appends them with global atomics in racy order and then needs a full
//     radix sort of the Contact and Joint archetypes every substep; here order
//     is deterministic by construction and those ~8 sorts disappear.
//   * every kernel reads the component columns straight from the table
//     descriptors (coalesced AoS-in-SoA rows), no per-row Context / hash lookup.
//   * IEEE arithmetic (--fmad=false) and the reference's operation order, so
//     floats track the CPU oracle.
#include "physics_host.hpp"
#include "physics_state.h"

#include <madrona/math.hpp>
#include <madrona/gjk.hpp>

#include <cfloat>
#include <algorithm>

namespace mb2 {

using madrona::math::Vector3;
using madrona::math::Vector4;
using madrona::math::Quat;
using madrona::math::Diag3x3;
using madrona::math::Mat3x3;
using madrona::math::AABB;
using madrona::math::cross;
using madrona::math::dot;
using madrona::geo::HalfEdge;
using madrona::geo::HalfEdgeMesh;
using madrona::geo::Plane;
using madrona::phys::CollisionPrimitive;
using madrona::phys::JointConstraint;
using madrona::phys::ObjectManager;
using madrona::phys::PhysicsSystemState;
using madrona::phys::ResponseType;
using madrona::phys::RigidBodyMetadata;
using madrona::phys::Velocity;
using madrona::phys::xpbd::PreSolvePositional;
using madrona::phys::xpbd::PreSolveVelocity;
using madrona::phys::xpbd::SubstepPrevState;

constexpr int kPhysWarps = 2;     // worlds (warps) per block of the per-world physics kernels

struct PhysicsHost {
    PhysicsState *dPhys = nullptr;
    PhysicsState hPhys;
    bool active = false;
    bool spheres = false;     // some registered object has a sphere primitive (read before graph capture)
};

// ---- small device helpers ------------------------------------------------------------

__device__ __forceinline__ const BodyArchetype *bodyOf(const PhysicsState &P, u32 arch)
{
    if (arch >= (u32)kMaxArchetypes) return nullptr;
    const int idx = P.bodyIndex[arch];
    return idx < 0 ? nullptr : &P.bodies[idx];
}

template <typename T>
__device__ __forceinline__ T &bodyCol(const EngineState &S, const BodyArchetype &b, int pc, i32 row)
{
    return ((T *)S.tables[b.archetype].columns[b.cols[pc]])[row];
}

// Column base pointers of every (rigid-body archetype, physics component), staged in shared
// memory by each per-world / per-candidate kernel before its first access (fillColCache).
// A component access by (archetype id, row) is then one shared-memory lookup and one global
// load; through PhysicsState::bodyIndex -> bodies[].cols -> tables[].columns it was a chain
// of three dependent global loads before the data (ncu, position solve: 37 % of the stall
// samples sat on that chain).  Sorts flip column pointers only between kernels.
struct ColCache {
    void *ptr[kMaxBodyArchetypes][PCCount];
    signed char bodyIndex[kMaxArchetypes];
};
__shared__ ColCache g_cols;

__device__ __forceinline__ void fillColCache(const EngineState &S, const PhysicsState &P)
{
    const int n = (int)P.numBodyArchetypes * (int)PCCount;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int bi = i / (int)PCCount, pc = i - bi * (int)PCCount;
        const BodyArchetype &b = P.bodies[bi];
        const i32 col = b.cols[pc];
        g_cols.ptr[bi][pc] = col >= 0 ? S.tables[b.archetype].columns[col] : nullptr;
    }
    for (int i = threadIdx.x; i < kMaxArchetypes; i += blockDim.x) g_cols.bodyIndex[i] = P.bodyIndex[i];
    __syncthreads();
}

__device__ __forceinline__ bool isBodyArchetype(u32 arch)
{
    return arch < (u32)kMaxArchetypes && g_cols.bodyIndex[arch] >= 0;
}

template <typename T>
__device__ __forceinline__ T &locCol(const EngineState &, const PhysicsState &, u32 arch, i32 row, int pc)
{
    return ((T *)g_cols.ptr[g_cols.bodyIndex[arch]][pc])[row];
}

__device__ __forceinline__ WorldBVH &worldBVH(const EngineState &S, const PhysicsState &P, i32 w)
{
    return ((WorldBVH *)S.tables[P.bvhArchetype].columns[2])[w];
}

__device__ __forceinline__ const PhysicsSystemState &worldParams(const EngineState &S, const PhysicsState &P, i32 w)
{
    return ((const PhysicsSystemState *)S.tables[P.paramsArchetype].columns[2])[w];
}

__device__ __forceinline__ const ObjectManager &worldObjects(const EngineState &S, const PhysicsState &P, i32 w)
{
    return **(const ObjectManager *const *)((const char *)S.tables[P.objectDataArchetype].columns[2] +
                                            (size_t)w * 8);
}

__device__ __forceinline__ Vector3 mulDiag(Vector3 d, Vector3 v)
{
    return Vector3 { d.x * v.x, d.y * v.y, d.z * v.z };
}

// Wide accesses for the 16 / 24 / 40-byte row types (columns are 256-byte
// aligned, BVH arrays 128-byte aligned): one request per 8 or 16 bytes instead
// of one per float -- the row kernels are LSU-queue bound otherwise.
__device__ __forceinline__ Quat loadQuat(const Quat *p)
{
    const float4 v = *reinterpret_cast<const float4 *>(p);
    return Quat { v.x, v.y, v.z, v.w };
}

__device__ __forceinline__ void storeQuat(Quat *p, Quat q)
{
    *reinterpret_cast<float4 *>(p) = make_float4(q.w, q.x, q.y, q.z);
}

template <typename T>
__device__ __forceinline__ T loadPairs(const T *p)
{
    static_assert(sizeof(T) % 8 == 0, "");
    union { T t; float2 v[sizeof(T) / 8]; } u;
#pragma unroll
    for (int i = 0; i < (int)(sizeof(T) / 8); i++) u.v[i] = reinterpret_cast<const float2 *>(p)[i];
    return u.t;
}

template <typename T>
__device__ __forceinline__ void storePairs(T *p, const T &value)
{
    static_assert(sizeof(T) % 8 == 0, "");
    union U { T t; float2 v[sizeof(T) / 8]; __device__ U() {} } u;
    u.t = value;
#pragma unroll
    for (int i = 0; i < (int)(sizeof(T) / 8); i++) reinterpret_cast<float2 *>(p)[i] = u.v[i];
}

// Float min / max as ONE native integer atomic (no CAS loop, no return value needed): for
// value >= 0 the signed-int order of the bit patterns is the float order (every negative float
// is a negative int), for value < 0 the unsigned order is the reversed float order.
__device__ __forceinline__ void atomicMinFloat(float *addr, float value)
{
    if (value >= 0.f) atomicMin((int *)addr, __float_as_int(value));
    else atomicMax((unsigned int *)addr, __float_as_uint(value));
}

__device__ __forceinline__ void atomicMaxFloat(float *addr, float value)
{
    if (value >= 0.f) atomicMax((int *)addr, __float_as_int(value));
    else atomicMin((unsigned int *)addr, __float_as_uint(value));
}

// =============================================================================================
// Broadphase
// =============================================================================================

// Leaf box = object box under TRS, stretched along the motion of the next
// step: per axis delta = velExpansion * v, min += delta - a if negative,
// max += delta + a if positive (broadphase.cpp:440-464).
__device__ __forceinline__ AABB growByMotion(AABB box, Vector3 v, float vel_k, float accel_k)
{
    for (int i = 0; i < 3; i++) {
        float delta = vel_k * v[i];
        float lo = delta - accel_k;
        float hi = delta + accel_k;
        if (lo < 0.f) box.pMin[i] += lo;
        if (hi > 0.f) box.pMax[i] += hi;
    }
    return box;
}

__device__ __forceinline__ void rowUpdateLeaf(const EngineState &S, const PhysicsState &P, const BodyArchetype &b, const i32 row, const i32 w)
{
    {
        WorldBVH &bvh = worldBVH(S, P, w);
        const ObjectManager &objs = *bvh.objMgr;

        const i32 leaf = bodyCol<i32>(S, b, PCLeafID, row);
        const Vector3 pos = bodyCol<Vector3>(S, b, PCPosition, row);
        const Quat rot = loadQuat(&bodyCol<Quat>(S, b, PCRotation, row));
        const Diag3x3 scale = bodyCol<Diag3x3>(S, b, PCScale, row);
        const i32 obj = bodyCol<i32>(S, b, PCObjectID, row);
        const Vector3 lin_vel = bodyCol<Velocity>(S, b, PCVelocity, row).linear;

        AABB world_box = objs.rigidBodyAABBs[obj].applyTRS(pos, rot, scale);
        AABB grown = growByMotion(world_box, lin_vel, bvh.velExpansion, bvh.accelExpansion);

        storePairs(&bvh.leafAABBs[leaf], grown);
        LeafTransform lt { pos, rot, { scale.d0, scale.d1, scale.d2 } };
        storePairs(&bvh.leafTransforms[leaf], lt);
        bvh.sortedLeaves[leaf] = leaf;
    }
}

// ---- top-down build, one thread per world, only when the world asked for it -----------

__device__ __forceinline__ Vector3 leafCenter(const WorldBVH &bvh, i32 slot)
{
    const AABB b = bvh.leafAABBs[bvh.sortedLeaves[slot]];
    return (b.pMin + b.pMax) / 2.f;
}

// Partition sortedLeaves[base, base+n) around the midpoint of the centroid
// range on its widest axis; returns the size of the left part (n/2 when the
// partition degenerates).
__device__ i32 midpointPartition(WorldBVH &bvh, i32 base, i32 n)
{
    Vector3 cmin { FLT_MAX, FLT_MAX, FLT_MAX };
    Vector3 cmax { -FLT_MAX, -FLT_MAX, -FLT_MAX };
    for (i32 i = 0; i < n; i++) {
        Vector3 c = leafCenter(bvh, base + i);
        cmin = Vector3::min(cmin, c);
        cmax = Vector3::max(cmax, c);
    }
    Vector3 extent = cmax - cmin;
    int axis;
    if (extent.x > extent.y && extent.x > extent.z) axis = 0;
    else if (extent.y > extent.x && extent.y > extent.z) axis = 1;
    else axis = 2;

    const float split = 0.5f * (cmin[axis] + cmax[axis]);
    i32 lo = 0, hi = n;
    while (lo < hi) {
        while (lo < hi && leafCenter(bvh, base + lo)[axis] < split) ++lo;
        while (lo < hi && leafCenter(bvh, base + hi - 1)[axis] >= split) --hi;
        if (lo < hi) {
            i32 tmp = bvh.sortedLeaves[base + lo];
            bvh.sortedLeaves[base + lo] = bvh.sortedLeaves[base + hi - 1];
            bvh.sortedLeaves[base + hi - 1] = tmp;
            ++lo;
            --hi;
        }
    }
    return (lo > 0 && lo < n) ? lo : n / 2;
}

__device__ void rebuildWorldBVH(WorldBVH &bvh)
{
    const i32 num_leaves = bvh.numLeaves;
    i32 third = (num_leaves - 1 + 2) / 3;
    bvh.numNodes = (third > 1 ? third : 1) + num_leaves;

    struct Pending {
        i32 node;     // -1 until the entry got its node
        i32 parent;
        i32 offset;
        i32 count;
    };
    Pending stack[64];
    stack[0] = Pending { -1, -1, 0, num_leaves };
    i32 depth = 1;
    i32 next_node = 0;

    while (depth > 0) {
        Pending &top = stack[depth - 1];
        i32 node_id;
        if (top.count <= 4) {
            // leaf-level node: up to four leaves, in sorted order
            node_id = next_node++;
            BVHNode &node = bvh.nodes[node_id];
            node.parentID = top.parent;
            for (int i = 0; i < 4; i++) {
                if (i < top.count) {
                    i32 leaf = bvh.sortedLeaves[top.offset + i];
                    const AABB box = bvh.leafAABBs[leaf];
                    bvh.leafParents[leaf] = ((u32)node_id << 2) | (u32)i;
                    node.children[i] = (i32)(0x80000000u | (u32)leaf);
                    node.minX[i] = box.pMin.x; node.minY[i] = box.pMin.y; node.minZ[i] = box.pMin.z;
                    node.maxX[i] = box.pMax.x; node.maxY[i] = box.pMax.y; node.maxZ[i] = box.pMax.z;
                } else {
                    node.children[i] = -1;
                    node.minX[i] = FLT_MAX; node.minY[i] = FLT_MAX; node.minZ[i] = FLT_MAX;
                    node.maxX[i] = -FLT_MAX; node.maxY[i] = -FLT_MAX; node.maxZ[i] = -FLT_MAX;
                }
            }
        } else if (top.node == -1) {
            // first visit of an inner entry: take a node, split the range into
            // quarters (half, then each half again) and descend left to right
            node_id = next_node++;
            top.node = node_id;
            BVHNode &node = bvh.nodes[node_id];
            for (int i = 0; i < 4; i++) node.children[i] = -1;
            node.parentID = top.parent;

            const i32 offset = top.offset, count = top.count;
            const i32 half = midpointPartition(bvh, offset, count);
            const i32 n_left = half, n_right = count - half;
            const i32 q1 = midpointPartition(bvh, offset, n_left);
            const i32 q3 = midpointPartition(bvh, offset + half, n_right);

            stack[depth++] = Pending { -1, node_id, offset + n_left + q3, n_right - q3 };
            stack[depth++] = Pending { -1, node_id, offset + n_left, q3 };
            stack[depth++] = Pending { -1, node_id, offset + q1, n_left - q1 };
            stack[depth++] = Pending { -1, node_id, offset, q1 };
            continue;
        } else {
            node_id = top.node;   // children done
        }

        depth -= 1;
        BVHNode &node = bvh.nodes[node_id];
        if (node.parentID == -1) continue;

        AABB merged = AABB::invalid();
        for (int i = 0; i < 4; i++) {
            if (node.children[i] == -1) break;
            merged = AABB::merge(merged, AABB { { node.minX[i], node.minY[i], node.minZ[i] },
                                                { node.maxX[i], node.maxY[i], node.maxZ[i] } });
        }
        BVHNode &parent = bvh.nodes[node.parentID];
        int slot = 0;
        while (parent.children[slot] != -1) slot++;
        parent.children[slot] = node_id;
        parent.minX[slot] = merged.pMin.x; parent.minY[slot] = merged.pMin.y; parent.minZ[slot] = merged.pMin.z;
        parent.maxX[slot] = merged.pMax.x; parent.maxY[slot] = merged.pMax.y; parent.maxZ[slot] = merged.pMax.z;
    }

    // report order of an un-pruned traversal (include/madrona/broadphase.inl:21-59)
    i32 order_n = 0;
    i32 walk[64];
    walk[0] = 0;
    i32 walk_n = 1;
    while (walk_n > 0) {
        const BVHNode &node = bvh.nodes[walk[--walk_n]];
        for (int i = 0; i < 4; i++) {
            const i32 child = node.children[i];
            if (child == -1) continue;
            if (child & 0x80000000) {
                if (order_n < bvh.numAllocatedLeaves) bvh.traversalOrder[order_n++] = child & 0x7fffffff;
            } else if (walk_n < 64) {
                walk[walk_n++] = child;
            }
        }
    }
    bvh.numTraversal = order_n;
    for (i32 k = 0; k < order_n; k++) {
        const i32 leaf = bvh.traversalOrder[k];
        bvh.leafOrderPos[leaf] = k;
        const u32 packed = bvh.leafParents[leaf];
        const BVHNode &node = bvh.nodes[packed >> 2];
        const int sub = (int)(packed & 3u);
        bvh.orderedBoxes[2 * k] = PVec4 { node.minX[sub], node.minY[sub], node.minZ[sub], node.maxX[sub] };
        bvh.orderedBoxes[2 * k + 1] = PVec4 { node.maxY[sub], node.maxZ[sub], __int_as_float(leaf), 0.f };
    }
}

__device__ void refitLeaf(WorldBVH &bvh, i32 leaf);

// Rebuild (rare: after a reset) followed by the refit of every leaf of the
// world, which the fused update+refit kernel skipped for this world.
__device__ __forceinline__ void phaseRebuild(const EngineState &S, const PhysicsState &P, const i32 w, const int lane)
{
    if (lane != 0) return;
    WorldBVH &bvh = worldBVH(S, P, w);
    if (!bvh.forceRebuild) return;
    bvh.forceRebuild = 0;
    rebuildWorldBVH(bvh);
    for (u32 bi = 0; bi < P.numBodyArchetypes; bi++) {
        const BodyArchetype &b = P.bodies[bi];
        const TableDesc &t = S.tables[b.archetype];
        const i32 first_row = t.worldOffsets[w];
        const i32 num_rows = t.worldCounts[w];
        for (i32 row = first_row; row < first_row + num_rows; row++) {
            if (((const i32 *)t.columns[1])[row] != w) continue;
            refitLeaf(bvh, bodyCol<i32>(S, b, PCLeafID, row));
        }
    }
}

// Grow-only refit: push the leaf's box into its slot, then keep growing
// ancestors while something actually grew (broadphase.cpp:550-647).
__device__ void refitLeaf(WorldBVH &bvh, i32 leaf)
{
    const AABB box = bvh.leafAABBs[leaf];
    const u32 packed = bvh.leafParents[leaf];
    i32 node_idx = (i32)(packed >> 2);
    const int sub = (int)(packed & 3u);
    BVHNode &leaf_node = bvh.nodes[node_idx];
    {
        bool grew = false;
        float prev;
        prev = leaf_node.minX[sub]; if (box.pMin.x < prev) { leaf_node.minX[sub] = box.pMin.x; grew = true; }
        prev = leaf_node.minY[sub]; if (box.pMin.y < prev) { leaf_node.minY[sub] = box.pMin.y; grew = true; }
        prev = leaf_node.minZ[sub]; if (box.pMin.z < prev) { leaf_node.minZ[sub] = box.pMin.z; grew = true; }
        prev = leaf_node.maxX[sub]; if (box.pMax.x > prev) { leaf_node.maxX[sub] = box.pMax.x; grew = true; }
        prev = leaf_node.maxY[sub]; if (box.pMax.y > prev) { leaf_node.maxY[sub] = box.pMax.y; grew = true; }
        prev = leaf_node.maxZ[sub]; if (box.pMax.z > prev) { leaf_node.maxZ[sub] = box.pMax.z; grew = true; }
        if (!grew) return;
        // keep the flat list in step with the slot box (only this leaf's thread writes either)
        const i32 k = bvh.leafOrderPos[leaf];
        float4 *flat = reinterpret_cast<float4 *>(bvh.orderedBoxes);
        flat[2 * k] = make_float4(leaf_node.minX[sub], leaf_node.minY[sub], leaf_node.minZ[sub], leaf_node.maxX[sub]);
        flat[2 * k + 1] = make_float4(leaf_node.maxY[sub], leaf_node.maxZ[sub], __int_as_float(leaf), 0.f);
    }
    i32 child = node_idx;
    node_idx = leaf_node.parentID;
    while (node_idx != -1) {
        BVHNode &node = bvh.nodes[node_idx];
        int slot = -1;
        for (int j = 0; j < 4; j++) {
            if (node.children[j] == child) { slot = j; break; }
        }
        if (slot < 0) return;
        // the six bounds are fetched together (L2: other SMs grow them with atomics), the
        // components that this leaf extends are pushed with fire-and-forget atomics; a bound
        // that a concurrent leaf has grown past ours meanwhile only costs a redundant climb
        const float o0 = __ldcg(&node.minX[slot]), o1 = __ldcg(&node.minY[slot]), o2 = __ldcg(&node.minZ[slot]);
        const float o3 = __ldcg(&node.maxX[slot]), o4 = __ldcg(&node.maxY[slot]), o5 = __ldcg(&node.maxZ[slot]);
        bool grew = false;
        if (box.pMin.x < o0) { atomicMinFloat(&node.minX[slot], box.pMin.x); grew = true; }
        if (box.pMin.y < o1) { atomicMinFloat(&node.minY[slot], box.pMin.y); grew = true; }
        if (box.pMin.z < o2) { atomicMinFloat(&node.minZ[slot], box.pMin.z); grew = true; }
        if (box.pMax.x > o3) { atomicMaxFloat(&node.maxX[slot], box.pMax.x); grew = true; }
        if (box.pMax.y > o4) { atomicMaxFloat(&node.maxY[slot], box.pMax.y); grew = true; }
        if (box.pMax.z > o5) { atomicMaxFloat(&node.maxZ[slot], box.pMax.z); grew = true; }
        if (!grew) break;
        child = node_idx;
        node_idx = node.parentID;
    }
}

__device__ __forceinline__ void rowRefit(const EngineState &S, const PhysicsState &P, const BodyArchetype &b, const i32 row, const i32 w)
{
    refitLeaf(worldBVH(S, P, w), bodyCol<i32>(S, b, PCLeafID, row));
}

// A body takes part in contact ordering unless writing it back is a no-op:
// static (inverse mass / inertia forced to 0, so x is unchanged) AND its
// rotation is a bitwise fixpoint of normalize() (so q is unchanged).  Decided
// once per step by the candidate search (a fixpoint stays one: the solvers
// write back normalize(q) == q; treating a body that BECAME a fixpoint during
// the step as still mutable only adds ordering edges, never removes one).
__device__ __forceinline__ bool rotationIsNormalizeFixpoint(Quat q)
{
    const Quat n = q.normalize();
    return n.w == q.w && n.x == q.x && n.y == q.y && n.z == q.z;
}

constexpr u32 kUnknownSlot = 0x7fffu;

// ---- candidate pairs: one warp per world, CPU iteration order -----------------------------

struct PairVisitor {
    const EngineState &S;
    const PhysicsState &P;
    const ObjectManager &objs;
    i32 selfID;
    bool selfStatic;
    u32 selfPrims;
};

// Visit every (a, b) pair the leaf box of body `a` produces, in traversal
// order: children 0..3 of a node in order, inner nodes pushed and popped LIFO
// (include/madrona/broadphase.inl:21-59); keep only e_a.id < e_b.id and drop
// static-static (broadphase.cpp:930-993).
template <typename Fn>
__device__ __forceinline__ void forEachPartner(const WorldBVH &bvh, const PairVisitor &v,
                                               const AABB &box, Fn &&fn)
{
    i32 stack[32];
    stack[0] = 0;
    int depth = 1;
    while (depth > 0) {
        const BVHNode &node = bvh.nodes[stack[--depth]];
        for (int i = 0; i < 4; i++) {
            const i32 child = node.children[i];
            if (child == -1) continue;
            AABB child_box { { node.minX[i], node.minY[i], node.minZ[i] },
                             { node.maxX[i], node.maxY[i], node.maxZ[i] } };
            if (!box.overlaps(child_box)) continue;
            if (child & 0x80000000) {
                const u64 packed = bvh.leafEntities[child & 0x7fffffff];
                const i32 other_id = (i32)(u32)(packed >> 32);
                const u32 other_gen = (u32)(packed & 0xFFFFFFFFull);
                if (!(v.selfID < other_id)) continue;
                const EntitySlot slot = v.S.entitySlots[other_id];
                if (slot.gen != other_gen) continue;
                const u32 b_arch = (u32)slot.a;
                const i32 b_row = slot.b;
                const BodyArchetype *bb = bodyOf(v.P, b_arch);
                if (!bb) continue;
                if (v.selfStatic &&
                    bodyCol<ResponseType>(v.S, *bb, PCResponseType, b_row) == ResponseType::Static) continue;
                const u32 b_prims = v.objs.rigidBodyPrimitiveCounts[bodyCol<i32>(v.S, *bb, PCObjectID, b_row)];
                fn(b_arch, b_row, b_prims);
            } else if (depth < 32) {
                stack[depth++] = child;
            }
        }
    }
}

constexpr int kMaxStagedLeaves = 128;          // bodies per world the candidate search handles
constexpr int kLeafMaskWords = kMaxStagedLeaves / 64;

struct __align__(16) StagedLeaf {
    float box[6];       // the leaf's slot in its parent node (grow-only since the last rebuild)
    i32 entityID;
    u32 arch;
    i32 row;
    u32 prims;          // 0 => stale entity / not a rigid body: never a partner
    u32 isStatic;
    u32 slotInfo;       // (world body slot << 1) | mutable  (Candidate::slots)
};

struct CandidateScratch {
    StagedLeaf leaves[kPhysWarps][kMaxStagedLeaves];
};

// Candidate pairs of one world, in the CPU backend's order (bodies: archetype
// ascending, then row; partners of a body: BVH report order).  The set a
// traversal reports for body a is { leaf b : slotBox(b) overlaps leafBox(a) }
// (ancestor boxes contain their leaves' slot boxes, so pruning removes nothing
// else) and its order is the tree's fixed report order, so the search is a
// uniform loop over the staged leaves instead of 32 divergent stack walks.
__device__ void phaseFindCandidates(EngineState &S, const PhysicsState &P, const i32 w, const int lane,
                                    const int warp, CandidateScratch &scratch)
{
    const WorldBVH &bvh = worldBVH(S, P, w);
    const ObjectManager &objs = *bvh.objMgr;
    Candidate *out = P.candidates + (size_t)w * P.maxCandidatesPerWorld;
    StagedLeaf *staged = scratch.leaves[warp];
    i32 running = 0;

    const i32 num_leaves = bvh.numTraversal;
    if (num_leaves > kMaxStagedLeaves) {
        if (lane == 0) {
            atomicOr(&S.errorFlags, (u32)ErrPhysicsOverflow);
            P.candCounts[w] = 0;
        }
        return;
    }
    // slot of a body inside its world's body list: archetypes ascending, rows in order
    auto bodySlotInfo = [&](u32 arch, i32 row, bool is_static) -> u32 {
        i32 slot_base = 0;
        i32 slot = -1;
        for (u32 bi = 0; bi < P.numBodyArchetypes; bi++) {
            const TableDesc &bt = S.tables[P.bodies[bi].archetype];
            if (P.bodies[bi].archetype == arch) {
                slot = slot_base + (row - bt.worldOffsets[w]);
                break;
            }
            slot_base += bt.worldCounts[w];
        }
        bool is_mutable = true;
        if (is_static) is_mutable = !rotationIsNormalizeFixpoint(locCol<Quat>(S, P, arch, row, PCRotation));
        const u32 s15 = (slot < 0 || slot >= (i32)kUnknownSlot) ? kUnknownSlot : (u32)slot;
        return (s15 << 1) | (is_mutable ? 1u : 0u);
    };
    // stage 1: lane k describes the k-th reported leaf
    for (i32 k = lane; k < num_leaves; k += 32) {
        const float4 b0 = reinterpret_cast<const float4 *>(bvh.orderedBoxes)[2 * k];
        const float4 b1 = reinterpret_cast<const float4 *>(bvh.orderedBoxes)[2 * k + 1];
        const i32 leaf = __float_as_int(b1.z);
        StagedLeaf sl;
        sl.box[0] = b0.x; sl.box[1] = b0.y; sl.box[2] = b0.z;
        sl.box[3] = b0.w; sl.box[4] = b1.x; sl.box[5] = b1.y;
        const u64 packed = bvh.leafEntities[leaf];
        sl.entityID = (i32)(u32)(packed >> 32);
        const u32 gen = (u32)(packed & 0xFFFFFFFFull);
        sl.arch = 0; sl.row = 0; sl.prims = 0; sl.isStatic = 0; sl.slotInfo = 0;
        if (sl.entityID >= 0 && sl.entityID < S.entityCapacity) {
            const EntitySlot es = S.entitySlots[sl.entityID];
            const BodyArchetype *bb = es.gen == gen ? bodyOf(P, (u32)es.a) : nullptr;
            if (bb) {
                sl.arch = (u32)es.a;
                sl.row = es.b;
                sl.isStatic = bodyCol<ResponseType>(S, *bb, PCResponseType, es.b) == ResponseType::Static ? 1u : 0u;
                sl.prims = objs.rigidBodyPrimitiveCounts[bodyCol<i32>(S, *bb, PCObjectID, es.b)];
                sl.slotInfo = bodySlotInfo(sl.arch, sl.row, sl.isStatic != 0);
                if (sl.arch > 0xffu || sl.prims > 0xffu) {
                    atomicOr(&S.errorFlags, (u32)ErrPhysicsOverflow);   // does not fit the packed candidate
                    sl.prims = 0;
                }
            }
        }
        staged[k] = sl;
    }
    __syncwarp();

    for (u32 bi = 0; bi < P.numBodyArchetypes; bi++) {
        const BodyArchetype &b = P.bodies[bi];
        const TableDesc &t = S.tables[b.archetype];
        const i32 first = t.worldOffsets[w];
        const i32 count = t.worldCounts[w];
        for (i32 base = 0; base < count; base += 32) {
            const i32 row = first + base + lane;
            const bool valid = base + lane < count && ((const i32 *)t.columns[1])[row] == w;

            i32 self_id = 0;
            bool self_static = false;
            u32 self_prims = 0;
            u32 self_info = 0;
            AABB box = AABB::invalid();
            if (valid) {
                const u64 packed = ((const u64 *)t.columns[0])[row];
                self_id = (i32)(u32)(packed >> 32);
                self_static = bodyCol<ResponseType>(S, b, PCResponseType, row) == ResponseType::Static;
                self_prims = objs.rigidBodyPrimitiveCounts[bodyCol<i32>(S, b, PCObjectID, row)];
                self_info = bodySlotInfo(b.archetype, row, self_static);
                if (b.archetype > 0xffu || self_prims > 0xffu) {
                    atomicOr(&S.errorFlags, (u32)ErrPhysicsOverflow);
                    self_prims = 0;
                }
                box = bvh.leafAABBs[bodyCol<i32>(S, b, PCLeafID, row)];
            }

            // stage 2: which staged leaves does this body pair with (bit k of word k / 64)
            unsigned long long partners[kLeafMaskWords];
#pragma unroll
            for (int wd = 0; wd < kLeafMaskWords; wd++) partners[wd] = 0;
            i32 mine = 0;
#pragma unroll
            for (int wd = 0; wd < kLeafMaskWords; wd++) {
                const i32 k_end = min(num_leaves, (wd + 1) * 64);
                for (i32 k = wd * 64; k < k_end; k++) {
                    const StagedLeaf &sl = staged[k];
                    const AABB other { { sl.box[0], sl.box[1], sl.box[2] }, { sl.box[3], sl.box[4], sl.box[5] } };
                    const bool pair = valid && sl.prims != 0 && box.overlaps(other) &&
                        self_id < sl.entityID && !(self_static && sl.isStatic);
                    if (pair) {
                        partners[wd] |= 1ull << (k - wd * 64);
                        mine += (i32)(self_prims * sl.prims);
                    }
                }
            }
            // exclusive scan across the warp = emission offsets in row order
            i32 incl = mine;
            for (int o = 1; o < 32; o <<= 1) {
                i32 up = __shfl_up_sync(0xffffffffu, incl, o);
                if (lane >= o) incl += up;
            }
            const i32 total = __shfl_sync(0xffffffffu, incl, 31);
            i32 at = running + incl - mine;
#pragma unroll
            for (int wd = 0; wd < kLeafMaskWords; wd++) {
                unsigned long long word = partners[wd];
                while (word) {
                    const int k = wd * 64 + __ffsll((long long)word) - 1;
                    word &= word - 1;
                    const StagedLeaf &sl = staged[k];
                    const u32 checks = self_prims * sl.prims;
                    for (u32 c = 0; c < checks; c++) {
                        if (at < P.maxCandidatesPerWorld) {
                            out[at] = Candidate { b.archetype | (sl.arch << 8) | ((c / sl.prims) << 16) |
                                                      ((c % sl.prims) << 24),
                                                  row, sl.row, self_info | (sl.slotInfo << 16) };
                        }
                        at++;
                    }
                }
            }
            running += total;
        }
    }
    if (lane == 0) {
        if (running > P.maxCandidatesPerWorld) {
            atomicOr(&S.errorFlags, (u32)ErrPhysicsOverflow);
            running = P.maxCandidatesPerWorld;
        }
        P.candCounts[w] = running;
    }
}

// =============================================================================================
// Integration (xpbd.cpp:100-185) and velocity update (xpbd.cpp:738-779)
// =============================================================================================

__device__ __forceinline__ void rowIntegrate(const EngineState &S, const PhysicsState &P, const BodyArchetype &b, const i32 row, const i32 w)
{
    {

        Vector3 x = bodyCol<Vector3>(S, b, PCPosition, row);
        Quat q = loadQuat(&bodyCol<Quat>(S, b, PCRotation, row));
        const Velocity vel = loadPairs(&bodyCol<Velocity>(S, b, PCVelocity, row));
        Vector3 v = vel.linear;
        Vector3 omega = vel.angular;
        const ResponseType resp = bodyCol<ResponseType>(S, b, PCResponseType, row);

        SubstepPrevState &prev = bodyCol<SubstepPrevState>(S, b, PCPrevState, row);
        PreSolvePositional &pre_pos = bodyCol<PreSolvePositional>(S, b, PCPreSolvePos, row);
        PreSolveVelocity &pre_vel = bodyCol<PreSolveVelocity>(S, b, PCPreSolveVel, row);

        prev.prevPosition = x;
        prev.prevRotation = q;
        if (resp == ResponseType::Static) {
            pre_pos.x = x;
            pre_pos.q = q;
            storePairs(&pre_vel, PreSolveVelocity { Vector3::zero(), Vector3::zero() });
            return;
        }

        const PhysicsSystemState &params = worldParams(S, P, w);
        const ObjectManager &objs = worldObjects(S, P, w);
        const RigidBodyMetadata &meta = objs.metadata[bodyCol<i32>(S, b, PCObjectID, row)];
        const float inv_m = meta.mass.invMass;
        const Vector3 inv_I = meta.mass.invInertiaTensor;
        const float h = params.h;
        const Vector3 g { params.g.x, params.g.y, params.g.z };
        const Vector3 ext_force = bodyCol<Vector3>(S, b, PCExtForce, row);
        const Vector3 ext_torque = bodyCol<Vector3>(S, b, PCExtTorque, row);

        if (resp == ResponseType::Dynamic) v += h * g;
        v += h * inv_m * ext_force;
        x += h * v;

        const Vector3 I { inv_I.x == 0 ? 0.0f : 1.0f / inv_I.x,
                          inv_I.y == 0 ? 0.0f : 1.0f / inv_I.y,
                          inv_I.z == 0 ? 0.0f : 1.0f / inv_I.z };
        const Quat to_local = q.inv();
        const Vector3 tau_local = to_local.rotateVec(ext_torque);
        Vector3 omega_local = to_local.rotateVec(omega);
        const Vector3 I_omega = mulDiag(I, omega_local);
        // Euler's equations in the body frame (gyroscopic term included)
        omega_local += h * mulDiag(inv_I, tau_local - cross(omega_local, I_omega));
        omega = q.rotateVec(omega_local);

        const Quat spin = Quat::fromAngularVec(0.5f * h * omega);
        q += spin * q;
        q = q.normalize();

        bodyCol<Vector3>(S, b, PCPosition, row) = x;
        storeQuat(&bodyCol<Quat>(S, b, PCRotation, row), q);
        pre_pos.x = x;
        pre_pos.q = q;
        storePairs(&pre_vel, PreSolveVelocity { v, omega });
    }
}

// ---- TGS (src/physics/tgs.cpp): the reference's solver skeleton integrates and nothing else
__device__ __forceinline__ void rowTGSVelocities(const EngineState &S, const PhysicsState &P, const BodyArchetype &b, const i32 row, const i32 w)
{
    const ResponseType resp = bodyCol<ResponseType>(S, b, PCResponseType, row);
    if (resp == ResponseType::Static) return;
    Velocity &vel_ref = bodyCol<Velocity>(S, b, PCVelocity, row);
    const Velocity vel = loadPairs(&vel_ref);
    Vector3 v = vel.linear;
    Vector3 omega = vel.angular;
    const Quat q = loadQuat(&bodyCol<Quat>(S, b, PCRotation, row));
    const PhysicsSystemState &params = worldParams(S, P, w);
    const ObjectManager &objs = worldObjects(S, P, w);
    const RigidBodyMetadata &meta = objs.metadata[bodyCol<i32>(S, b, PCObjectID, row)];
    const float inv_m = meta.mass.invMass;
    const Vector3 inv_I = meta.mass.invInertiaTensor;
    const float h = params.h;
    const Vector3 g { params.g.x, params.g.y, params.g.z };
    if (resp == ResponseType::Dynamic) v += h * g;
    v += h * inv_m * bodyCol<Vector3>(S, b, PCExtForce, row);
    const Vector3 I { inv_I.x == 0 ? 0.0f : 1.0f / inv_I.x,
                      inv_I.y == 0 ? 0.0f : 1.0f / inv_I.y,
                      inv_I.z == 0 ? 0.0f : 1.0f / inv_I.z };
    const Quat to_local = q.inv();
    const Vector3 tau_local = to_local.rotateVec(bodyCol<Vector3>(S, b, PCExtTorque, row));
    Vector3 omega_local = to_local.rotateVec(omega);
    // NB: the reference multiplies I by the WORLD-space omega here (tgs.cpp:133-134)
    omega_local += h * mulDiag(inv_I, tau_local - cross(omega_local, mulDiag(I, omega)));
    omega = q.rotateVec(omega_local);
    storePairs(&vel_ref, Velocity { v, omega });
}

__device__ __forceinline__ void rowTGSPositions(const EngineState &S, const PhysicsState &P, const BodyArchetype &b, const i32 row, const i32 w)
{
    const float h = worldParams(S, P, w).h;
    Vector3 x = bodyCol<Vector3>(S, b, PCPosition, row);
    Quat q = loadQuat(&bodyCol<Quat>(S, b, PCRotation, row));
    const Velocity vel = loadPairs(&bodyCol<Velocity>(S, b, PCVelocity, row));
    x += h * vel.linear;
    const Quat spin = Quat::fromAngularVec(0.5f * h * vel.angular);
    q += spin * q;
    q = q.normalize();
    bodyCol<Vector3>(S, b, PCPosition, row) = x;
    storeQuat(&bodyCol<Quat>(S, b, PCRotation, row), q);
}

__device__ __forceinline__ void rowSetVelocity(const EngineState &S, const PhysicsState &P, const BodyArchetype &b, const i32 row, const i32 w)
{
    {
        const float h = worldParams(S, P, w).h;
        const Vector3 x = bodyCol<Vector3>(S, b, PCPosition, row);
        const Quat q = loadQuat(&bodyCol<Quat>(S, b, PCRotation, row));
        const SubstepPrevState prev = bodyCol<SubstepPrevState>(S, b, PCPrevState, row);

        // bitwise-equal orientations mean exactly zero angular velocity
        Quat dq;
        if (q.w != prev.prevRotation.w || q.x != prev.prevRotation.x ||
            q.y != prev.prevRotation.y || q.z != prev.prevRotation.z) {
            dq = q * prev.prevRotation.inv();
        } else {
            dq = Quat { 1, 0, 0, 0 };
        }
        const Vector3 new_omega = 2.f / h * Vector3 { dq.x, dq.y, dq.z };

        Velocity out;
        out.linear = (x - prev.prevPosition) / h;
        out.angular = dq.w > 0.f ? new_omega : -new_omega;
        storePairs(&bodyCol<Velocity>(S, b, PCVelocity, row), out);
    }
}

// =============================================================================================
// Narrowphase (scalar SAT path of the reference)
// =============================================================================================

struct HullInWorld {
    const HalfEdgeMesh *mesh;
    Vector3 *verts;     // world space
    Plane *planes;      // world space
    u32 numVerts;
    u32 numFaces;
    Vector3 center;
};

// (placement: vertex = R S v + t, normal = normalize(R S^-1 n), plane offset through a
// transformed point of the plane, centre = vertex mean -- narrowphase.cpp:151-223;
// done by the lanes of the warp in hullHullCooperative, on the fly for hull-plane)
__device__ __forceinline__ float planeDistance(const Plane &pl, Vector3 p)
{
    return dot(p, pl.normal) - pl.d;
}

__device__ float hullSupportDistance(const Plane &pl, const HullInWorld &h)
{
    float lowest = FLT_MAX;
#pragma unroll 1
    for (u32 i = 0; i < h.numVerts; i++) {
        float along = dot(h.verts[i], pl.normal);
        if (along < lowest) lowest = along;
    }
    return lowest - pl.d;
}

struct FaceAxis {
    float separation;
    i32 face;
    Plane plane;
};

// faces of a against b: ascending, strictly greater wins, stop at the first
// positive separation (narrowphase.cpp:339-365)
__device__ FaceAxis bestFaceAxis(const HullInWorld &a, const HullInWorld &b)
{
    FaceAxis best { -FLT_MAX, -1, Plane { Vector3::zero(), 0.f } };
    for (u32 f = 0; f < a.numFaces; f++) {
        Plane pl = a.planes[f];
        float sep = hullSupportDistance(pl, b);
        if (sep > best.separation) {
            best.separation = sep;
            best.face = (i32)f;
            best.plane = pl;
            if (sep > 0) break;
        }
    }
    return best;
}

struct EdgeAxis {
    float separation;
    Vector3 normal;
    i32 edgeA;
    i32 edgeB;
};

__device__ __forceinline__ bool gaussMapArcsCross(Vector3 a, Vector3 b, Vector3 c, Vector3 d)
{
    Vector3 bxa = b.cross(a);
    Vector3 dxc = d.cross(c);
    float cba = c.dot(bxa);
    float dba = d.dot(bxa);
    float adc = a.dot(dxc);
    float bdc = b.dot(dxc);
    return cba * dba < 0.0f && adc * bdc < 0.0f && cba * bdc > 0.0f;
}

// edge pairs a-major over numHalfEdges/2 edges (half-edge 2k, twin 2k+1); only
// pairs forming a face of the Minkowski difference are measured
// (narrowphase.cpp:367-567)
__device__ EdgeAxis bestEdgeAxis(const HullInWorld &a, const HullInWorld &b)
{
    EdgeAxis best { -FLT_MAX, Vector3::zero(), 0, 0 };
    const u32 ea = a.mesh->numHalfEdges / 2, eb = b.mesh->numHalfEdges / 2;
    for (u32 ia = 0; ia < ea; ia++) {
        const u32 ha = ia * 2;
        const HalfEdge a0 = a.mesh->halfEdges[ha];
        const HalfEdge a1 = a.mesh->halfEdges[ha ^ 1u];
        const Vector3 an0 = a.planes[a0.face].normal;
        const Vector3 an1 = a.planes[a1.face].normal;
        for (u32 ib = 0; ib < eb; ib++) {
            const u32 hb = ib * 2;
            const HalfEdge b0 = b.mesh->halfEdges[hb];
            const HalfEdge b1 = b.mesh->halfEdges[hb ^ 1u];
            const Vector3 bn0 = b.planes[b0.face].normal;
            const Vector3 bn1 = b.planes[b1.face].normal;

            float sep = -FLT_MAX;
            Vector3 normal = Vector3::zero();
            if (gaussMapArcsCross(an0, an1, -bn0, -bn1)) {
                const Vector3 pa = a.verts[a0.rootVertex];
                const Vector3 qa = a.verts[a.mesh->halfEdges[a0.next].rootVertex];
                const Vector3 pb = b.verts[b0.rootVertex];
                const Vector3 qb = b.verts[b.mesh->halfEdges[b0.next].rootVertex];
                const Vector3 axis = (qa - pa).cross(qb - pb);
                const float len2 = axis.length2();
                if (len2 != 0) {
                    normal = axis * (1.f / sqrtf(len2));
                    if (normal.dot(pa - a.center) < 0.0f) normal = -normal;
                    sep = normal.dot(pb - pa);
                }
            }
            if (sep > best.separation) {
                best.separation = sep;
                best.normal = normal;
                best.edgeA = (i32)ha;
                best.edgeB = (i32)hb;
                if (sep > 0) return best;
            }
        }
    }
    return best;
}

// face most anti-parallel to the reference normal, first minimum wins
__device__ i32 mostOpposedFace(const HullInWorld &h, Vector3 ref_normal)
{
    float lowest = FLT_MAX;
    i32 face = -1;
#pragma unroll 1
    for (u32 f = 0; f < h.numFaces; f++) {
        float d = dot(h.planes[f].normal, ref_normal);
        if (d < lowest) {
            lowest = d;
            face = (i32)f;
        }
    }
    return face;
}

// Sutherland-Hodgman against one plane; "<= 0" is inside (narrowphase.cpp:617-652)
__device__ __noinline__ int clipAgainst(Vector3 *dst, const Plane &pl, const Vector3 *src, int n)
{
    int m = 0;
    Vector3 v1 = src[n - 1];
    float d1 = planeDistance(pl, v1);
#pragma unroll 1
    for (int i = 0; i < n; i++) {
        Vector3 v2 = src[i];
        float d2 = planeDistance(pl, v2);
        if (d1 <= 0.0f && d2 <= 0.0f) {
            dst[m++] = v2;
        } else if (d1 <= 0.0f && d2 > 0.0f) {
            dst[m++] = v1 + (v2 - v1) * (-d1 / pl.normal.dot(v2 - v1));
        } else if (d2 <= 0.0f && d1 > 0.0f) {
            dst[m++] = v1 + (v2 - v1) * (-d1 / pl.normal.dot(v2 - v1));
            dst[m++] = v2;
        }
        v1 = v2;
        d1 = d2;
    }
    return m;
}

struct ManifoldOut {
    Vector3 points[4];
    float depths[4];
    i32 count;
    Vector3 normal;
};

// <= 4 points pass through; otherwise keep A (first), B (farthest from A), C
// (largest |area| with AB), Q (most negative area outside ABC)
// (narrowphase.cpp:771-879).  World offset / frame are identity in the only
// live call sites.
__device__ __noinline__ ManifoldOut reduceManifoldLarge(Vector3 normal, const Vector3 *pts, const float *depths, int n)
{
    ManifoldOut m;
    m.normal = normal;
    for (int i = 0; i < 4; i++) {
        m.points[i] = Vector3::zero();
        m.depths[i] = 0.f;
    }
    if (n <= 4) {
        m.count = n;
        for (int i = 0; i < n; i++) {
            m.points[i] = pts[i];
            m.depths[i] = depths[i];
        }
        return m;
    }
    m.count = 4;
    m.points[0] = pts[0];
    m.depths[0] = depths[0];

    float far2 = 0.f;
#pragma unroll 1
    for (int i = 1; i < n; i++) {
        float d2 = m.points[0].distance2(pts[i]);
        if (d2 > far2) {
            far2 = d2;
            m.points[1] = pts[i];
            m.depths[1] = depths[i];
        }
    }
    Vector3 ba = m.points[1] - m.points[0];

    float best_area = 0.0f;
    // NB: the reference stores this sign in a bool, so "-1" never compares
    // equal and the winding flip below never fires; kept for parity.
    bool best_sign = false;
#pragma unroll 1
    for (int i = 1; i < n; i++) {
        Vector3 bc = pts[i] - m.points[1];
        float signed_area = normal.dot(cross(ba, bc));
        float area = copysignf(signed_area, 1.f);
        if (area > best_area) {
            best_area = area;
            best_sign = copysignf(1.f, signed_area) != 0.f;
            m.points[2] = pts[i];
            m.depths[2] = depths[i];
        }
    }
    if ((float)best_sign == -1.f) {
        ba = -ba;
        Vector3 tmp = m.points[0];
        m.points[0] = m.points[1];
        m.points[1] = tmp;
    }

    Vector3 cb = m.points[2] - m.points[1];
    Vector3 ac = m.points[0] - m.points[2];
    float most_neg = 0.f;
#pragma unroll 1
    for (int i = 1; i < n; i++) {
        Vector3 aq = m.points[0] - pts[i];
        Vector3 qc = pts[i] - m.points[2];
        float abq = normal.dot(cross(ba, aq));
        float bcq = normal.dot(cross(cb, qc));
        float caq = normal.dot(cross(aq, ac));
        float lowest = fminf(abq, fminf(bcq, caq));
        if (lowest < most_neg) {
            most_neg = lowest;
            m.points[3] = pts[i];
            m.depths[3] = depths[i];
        }
    }
    if (far2 == 0.f || best_area == 0.f || most_neg == 0.f) {
        m.count = 0;
        m.normal = Vector3::zero();
    }
    return m;
}

// the common case (a box face resting on something: <= 4 points) stays inline
__device__ __forceinline__ ManifoldOut reduceManifold(Vector3 normal, const Vector3 *pts, const float *depths, int n)
{
    if (n > 4) return reduceManifoldLarge(normal, pts, depths, n);
    ManifoldOut m;
    m.normal = normal;
    m.count = n;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        m.points[i] = i < n ? pts[i] : Vector3::zero();
        m.depths[i] = i < n ? depths[i] : 0.f;
    }
    return m;
}

constexpr int kClipCap = kMaxFaceVerts * 2 + 4;

__device__ ManifoldOut faceFaceManifold(const Plane &ref_plane, i32 ref_face, i32 inc_face,
                                        const HullInWorld &ref, const HullInWorld &inc,
                                        Vector3 *buf_a, Vector3 *buf_b)
{
    // incident polygon
    int n = 0;
    {
        u32 he = inc.mesh->faceBaseHalfEdges[inc_face];
        const u32 start = he;
        do {
            const HalfEdge cur = inc.mesh->halfEdges[he];
            he = cur.next;
            if (n < kClipCap) buf_a[n++] = inc.verts[cur.rootVertex];
        } while (he != start);
    }
    Vector3 *src = buf_a, *dst = buf_b;
    // clip against the side planes of the reference face (normal = edge x n_ref)
    {
        u32 he = ref.mesh->faceBaseHalfEdges[ref_face];
        const u32 start = he;
        Vector3 cur_pt = ref.verts[ref.mesh->halfEdges[he].rootVertex];
        do {
            he = ref.mesh->halfEdges[he].next;
            Vector3 next_pt = ref.verts[ref.mesh->halfEdges[he].rootVertex];
            Vector3 side_n = cross(next_pt - cur_pt, ref_plane.normal);
            Plane side { side_n, dot(side_n, cur_pt) };
            cur_pt = next_pt;
            n = n > 0 ? clipAgainst(dst, side, src, n) : 0;
            if (n > kClipCap) n = kClipCap;
            Vector3 *tmp = src;
            src = dst;
            dst = tmp;
        } while (he != start);
    }
    // keep what is at or below the reference plane, projected onto it
    float depths[kClipCap];
    int kept = 0;
#pragma unroll 1
    for (int i = 0; i < n; i++) {
        Vector3 p = src[i];
        float d = planeDistance(ref_plane, p);
        if (d <= 0.0f) {
            src[kept] = p - d * ref_plane.normal;
            depths[kept] = -d;
            kept++;
        }
    }
    return reduceManifold(ref_plane.normal, src, depths, kept);
}

// closest points of two segments, clamped (narrowphase.cpp:1037-1071); only the
// point on segment 1 is used by the caller
__device__ Vector3 closestOnFirstSegment(Vector3 p1, Vector3 q1, Vector3 p2, Vector3 q2)
{
    Vector3 v1 = q1 - p1;
    Vector3 v2 = q2 - p2;
    Vector3 v21 = p2 - p1;
    float d22 = v2.dot(v2);
    float d11 = v1.dot(v1);
    float d21 = v2.dot(v1);
    float d211 = v21.dot(v1);
    float d212 = v21.dot(v2);
    float denom = d21 * d21 - d22 * d11;
    float s;
    if (fabsf(denom) < 0.00001f) {
        s = 0.0f;
    } else {
        s = (d212 * d21 - d22 * d211) / denom;
    }
    s = fmaxf(fminf(s, 1.0f), 0.0f);
    return p1 + s * v1;
}

__device__ __forceinline__ void writeContact(Contact &c, u32 ref_arch, i32 ref_row, u32 alt_arch,
                                             i32 alt_row, const ManifoldOut &m)
{
    c.refArch = ref_arch; c.refRow = ref_row;
    c.altArch = alt_arch; c.altRow = alt_row;
    for (int i = 0; i < 4; i++) {
        c.points[i][0] = m.points[i].x;
        c.points[i][1] = m.points[i].y;
        c.points[i][2] = m.points[i].z;
        c.points[i][3] = m.depths[i];
    }
    c.numPoints = m.count;
    c.normal = m.normal;
    c.lambdaN = 0.f;
    c.level = 0;
}

__device__ __forceinline__ ManifoldOut singlePoint(Vector3 p, Vector3 n, float depth)
{
    ManifoldOut m;
    for (int i = 0; i < 4; i++) {
        m.points[i] = Vector3::zero();
        m.depths[i] = 0.f;
    }
    m.points[0] = p;
    m.depths[0] = depth;
    m.count = 1;
    m.normal = n;
    return m;
}

// ---- one candidate -> at most one contact (narrowphase.cpp:1682-1899 + 1516-1680) ------
//
// Stage A (every lane, its own candidate): order the pair by primitive type,
// fetch both transforms, primitive-AABB reject, and finish the cheap pair
// types (sphere-sphere, sphere-plane, hull-plane) on the spot.
// Stage B (whole warp, one hull-hull candidate at a time): both hulls are
// transformed into shared memory by all lanes, the 2 x F face queries and the
// E_a x E_b edge query are spread over the lanes, and the winner is picked with
// the reference's sequential rule (first strictly-greater separation in index
// order, stop at the first positive one) -- expressed as "lowest index among
// positives, else lowest index among maxima", which is order independent and
// therefore bit-identical.  Only the final clipping runs on the owning lane.

struct PairSetup {
    u32 aArch, bArch;
    i32 aRow, bRow;
    u32 aInfo, bInfo;  // (world body slot << 1) | mutable, see Candidate::slots
    const CollisionPrimitive *aPrim, *bPrim;
    Vector3 aPos, bPos;
    Quat aRot, bRot;
    Diag3x3 aScale, bScale;
    u32 test;          // 0 = rejected
};

template <bool REJECT>
__device__ __forceinline__ PairSetup setupPairImpl(const EngineState &S, const PhysicsState &P,
                                                   const ObjectManager &objs, const Candidate &cand)
{
    PairSetup ps;
    ps.aArch = cand.archPrim & 0xffu; ps.bArch = (cand.archPrim >> 8) & 0xffu;
    ps.aRow = cand.aRow; ps.bRow = cand.bRow;
    ps.aInfo = cand.slots & 0xffffu; ps.bInfo = cand.slots >> 16;
    u32 a_prim_idx = objs.rigidBodyPrimitiveOffsets[locCol<i32>(S, P, ps.aArch, ps.aRow, PCObjectID)] +
                     ((cand.archPrim >> 16) & 0xffu);
    u32 b_prim_idx = objs.rigidBodyPrimitiveOffsets[locCol<i32>(S, P, ps.bArch, ps.bRow, PCObjectID)] +
                     (cand.archPrim >> 24);
    ps.aPrim = &objs.collisionPrimitives[a_prim_idx];
    ps.bPrim = &objs.collisionPrimitives[b_prim_idx];
    u32 ta = (u32)ps.aPrim->type, tb = (u32)ps.bPrim->type;
    // order the pair by primitive type: sphere(1) < hull(2) < plane(4)
    if (ta > tb) {
        u32 tu;
        i32 ti;
        const CollisionPrimitive *tp;
        tu = ps.aArch; ps.aArch = ps.bArch; ps.bArch = tu;
        ti = ps.aRow; ps.aRow = ps.bRow; ps.bRow = ti;
        tu = ps.aInfo; ps.aInfo = ps.bInfo; ps.bInfo = tu;
        tp = ps.aPrim; ps.aPrim = ps.bPrim; ps.bPrim = tp;
        tu = a_prim_idx; a_prim_idx = b_prim_idx; b_prim_idx = tu;
        tu = ta; ta = tb; tb = tu;
    }
    ps.aPos = locCol<Vector3>(S, P, ps.aArch, ps.aRow, PCPosition);
    ps.bPos = locCol<Vector3>(S, P, ps.bArch, ps.bRow, PCPosition);
    ps.aRot = locCol<Quat>(S, P, ps.aArch, ps.aRow, PCRotation);
    ps.bRot = locCol<Quat>(S, P, ps.bArch, ps.bRow, PCRotation);
    ps.aScale = locCol<Diag3x3>(S, P, ps.aArch, ps.aRow, PCScale);
    ps.bScale = locCol<Diag3x3>(S, P, ps.bArch, ps.bRow, PCScale);

    if constexpr (REJECT) {
        AABB a_box = objs.primitiveAABBs[a_prim_idx].applyTRS(ps.aPos, ps.aRot, ps.aScale);
        AABB b_box = objs.primitiveAABBs[b_prim_idx].applyTRS(ps.bPos, ps.bRot, ps.bScale);
        ps.test = a_box.intersects(b_box) ? (ta | tb) : 0u;
    } else {
        ps.test = ta | tb;
    }
    return ps;
}

__device__ __forceinline__ PairSetup setupPair(const EngineState &S, const PhysicsState &P,
                                               const ObjectManager &objs, const Candidate &cand)
{
    return setupPairImpl<true>(S, P, objs, cand);
}

// sphere (a) - hull (b): GJK closest point of the hull to the sphere centre, SAT
// over the face planes when the centre is inside (narrowphase.cpp:1326-1402).
// Out of line and by value: rare in the box-world fixtures, inlining the GJK
// loop doubles the narrowphase kernel's code size, and handing it the caller's
// PairSetup / Contact by reference would push those into local memory for every
// pair type (measured: +5 % on the room step).
struct SphereHullResult {
    Vector3 point;
    Vector3 normal;
    float depth;
    i32 hit;          // 1 contact, 0 none, -1 hull too large for the staging array
};

__device__ __noinline__ SphereHullResult sphereHullContact(Vector3 a_pos, float radius, Vector3 b_pos,
                                                           Quat b_rot, Diag3x3 b_scale,
                                                           const HalfEdgeMesh *mesh)
{
    const HalfEdgeMesh &bm = *mesh;
    SphereHullResult res { Vector3::zero(), Vector3::zero(), 0.f, 0 };
    if (bm.numVertices > (u32)kMaxHullVerts) {
        res.hit = -1;
        return res;
    }
    // the hull relative to the sphere centre, so the query point is the origin
    const Vector3 hull_origin = b_pos - a_pos;
    const Mat3x3 rot = Mat3x3::fromQuat(b_rot);
    const Mat3x3 vert_m = rot * b_scale;
    const Mat3x3 norm_m = rot * b_scale.inv();
    Vector3 verts[kMaxHullVerts];
#pragma unroll 1
    for (u32 i = 0; i < bm.numVertices; i++) verts[i] = vert_m * bm.vertices[i] + hull_origin;

    Vector3 to_hull;
    const float dist2 = madrona::geo::hullVerticesClosestPointToOriginGJK(verts, bm.numVertices, 1e-10f,
                                                                         &to_hull);
    if (dist2 > radius * radius) return res;

    if (dist2 == 0.f) {
        // centre inside the hull: least-penetrated face (SAT over the face planes)
        float max_sep = -FLT_MAX;
        Vector3 sep_normal = Vector3::zero();
#pragma unroll 1
        for (u32 f = 0; f < bm.numFaces; f++) {
            const Plane local = bm.facePlanes[f];
            const Vector3 on_plane = vert_m * (local.normal * local.d) + hull_origin;
            const Vector3 n = (norm_m * local.normal).normalize();
            const float face_dist = -dot(n, on_plane);
            if (face_dist > max_sep) {
                max_sep = face_dist;
                sep_normal = n;
            }
        }
        if (max_sep > 0.f) return res;      // GJK and SAT disagree by rounding
        res.point = a_pos + sep_normal * radius;
        res.normal = sep_normal;
        res.depth = -max_sep;
    } else {
        const float to_hull_len = sqrtf(dist2);
        const Vector3 normal = to_hull / to_hull_len;
        res.point = a_pos + normal * radius;
        res.normal = -normal;
        res.depth = radius - to_hull_len;
    }
    res.hit = 1;
    return res;
}

// sphere-sphere (1), sphere-plane (5), hull-plane (6): finished by the lane itself
template <bool SPHERE_HULL>
__device__ bool narrowphaseSimple(EngineState &S, const PairSetup &ps, Contact &out)
{
    switch (ps.test) {
    case 1: {
        const float ra = ps.aScale.d0 * ps.aPrim->sphere.radius;
        const float rb = ps.bScale.d0 * ps.bPrim->sphere.radius;
        const Vector3 to_b = ps.bPos - ps.aPos;
        const float dist = to_b.length();
        if (dist > ra + rb) return false;
        const Vector3 n = dist > 0.f ? to_b / dist : madrona::math::up;
        // single-point contacts store (ref, alt) = (b, a)
        writeContact(out, ps.bArch, ps.bRow, ps.aArch, ps.aRow,
                     singlePoint(ps.aPos + ra * n, n, ra + rb - dist));
        return true;
    }
    case 5: {
        const float ra = ps.aScale.d0 * ps.aPrim->sphere.radius;
        const Vector3 n = ps.bRot.rotateVec(Vector3 { 0, 0, 1 });
        const float d = n.dot(ps.bPos);
        const float t = n.dot(ps.aPos) - d;
        const float pen = ra - t;
        if (pen < 0) return false;
        writeContact(out, ps.bArch, ps.bRow, ps.aArch, ps.aRow, singlePoint(ps.aPos - t * n, n, pen));
        return true;
    }
    case 6: {   // plane is b and the reference
        // The hull is never stored: every world-space vertex / face normal is
        // produced where it is consumed, with placeHull's per-element formulas
        // (vertex = R S v + t, normal = normalize(R S^-1 n)).
        const HalfEdgeMesh &am = ps.aPrim->hull.halfEdgeMesh;
        const Mat3x3 rot = Mat3x3::fromQuat(ps.aRot);
        const Mat3x3 vert_m = rot * ps.aScale;
        const Mat3x3 norm_m = rot * ps.aScale.inv();
        const Vector3 n = ps.bRot.rotateVec(Vector3 { 0, 0, 1 });
        const Plane plane { n, dot(n, ps.bPos) };

        float lowest = FLT_MAX;                       // hullSupportDistance
#pragma unroll 2
        for (u32 i = 0; i < am.numVertices; i++) {
            const Vector3 p = vert_m * am.vertices[i] + ps.aPos;
            const float along = dot(p, plane.normal);
            if (along < lowest) lowest = along;
        }
        if (lowest - plane.d > 0.0f) return false;

        float most = FLT_MAX;                         // mostOpposedFace
        i32 inc_face = -1;
#pragma unroll 2
        for (u32 f = 0; f < am.numFaces; f++) {
            const Vector3 face_n = (norm_m * am.facePlanes[f].normal).normalize();
            const float d = dot(face_n, plane.normal);
            if (d < most) {
                most = d;
                inc_face = (i32)f;
            }
        }

        Vector3 clip[kClipCap];                       // incident-face points at or below the plane
        float depths[kClipCap];
        int kept = 0;
        u32 he = am.faceBaseHalfEdges[inc_face];
        const u32 start = he;
        do {
            const HalfEdge cur = am.halfEdges[he];
            he = cur.next;
            const Vector3 p = vert_m * am.vertices[cur.rootVertex] + ps.aPos;
            const float d = planeDistance(plane, p);
            if (d <= 0.0f && kept < kClipCap) {
                clip[kept] = p - d * plane.normal;
                depths[kept] = -d;
                kept++;
            }
        } while (he != start);
        ManifoldOut m = reduceManifold(plane.normal, clip, depths, kept);
        if (m.count <= 0) return false;
        writeContact(out, ps.bArch, ps.bRow, ps.aArch, ps.aRow, m);
        return true;
    }
    case 3: {
        if constexpr (SPHERE_HULL) {
            const SphereHullResult r = sphereHullContact(ps.aPos, ps.aScale.d0 * ps.aPrim->sphere.radius,
                                                         ps.bPos, ps.bRot, ps.bScale, &ps.bPrim->hull.halfEdgeMesh);
            if (r.hit < 0) atomicOr(&S.errorFlags, (u32)ErrPhysicsOverflow);
            if (r.hit <= 0) return false;
            writeContact(out, ps.bArch, ps.bRow, ps.aArch, ps.aRow, singlePoint(r.point, r.normal, r.depth));
            return true;
        } else {
            // a sphere appeared after the launch graph was built without the
            // sphere-hull path: rebuild the launch graph
            atomicOr(&S.errorFlags, (u32)ErrPhysicsOverflow);
            return false;
        }
    }
    default:
        atomicOr(&S.errorFlags, (u32)ErrPhysicsOverflow);
        return false;
    }
}

struct HullScratch {
    Vector3 verts[2 * kMaxHullVerts];
    Plane planes[2 * kMaxHullFaces];
    Vector3 clipA[kClipCap];
    Vector3 clipB[kClipCap];
};

template <typename T>
__device__ __forceinline__ T warpBroadcast(T v, int src)
{
    static_assert(sizeof(T) % 4 == 0, "");
    union { T t; u32 w[sizeof(T) / 4]; } in, out;
    in.t = v;
#pragma unroll
    for (int i = 0; i < (int)(sizeof(T) / 4); i++) out.w[i] = __shfl_sync(0xffffffffu, in.w[i], src);
    return out.t;
}

// Hull - hull pairs are worked on by GROUPS of kGroupLanes lanes, kNarrowGroups
// pairs per warp at a time: a box has 6 faces and 8 vertices, so a whole warp on
// one pair leaves most lanes idle in the face queries and all but one in the
// clipping, and the pair's dependent load chains (primitive -> mesh -> vertex
// arrays) are not overlapped with anything.  Four pairs in flight give four
// independent chains per warp and keep 6 of 8 lanes busy in the face queries.
constexpr int kGroupLanes = 8;

// (separation, index) of the element the sequential scan would have kept.
struct Winner {
    float sep;
    i32 idx;
};

// Reduction over the lanes of one group (mask gm, xor distances stay inside the
// aligned group).  Input per lane: its own candidate (sep, idx) chosen by the
// same rule over the elements it looked at, or have = false.
// Rule == the scalar loop "keep strictly greater, stop at the first positive":
// lowest index among positives, else lowest index among maxima.
__device__ __forceinline__ Winner groupSequentialWinner(unsigned gm, float sep, i32 idx, bool have)
{
    const bool positive = have && sep > 0.f;
    if (__any_sync(gm, positive)) {
        i32 cand = positive ? idx : 0x7fffffff;
#pragma unroll
        for (int o = kGroupLanes / 2; o >= 1; o >>= 1) {
            const i32 other = __shfl_xor_sync(gm, cand, o);
            if (other < cand) cand = other;
        }
        const unsigned owner = __ballot_sync(gm, positive && idx == cand);
        const int src = __ffs(owner) - 1;
        return Winner { __shfl_sync(gm, sep, src), cand };
    }
    float s = have ? sep : -FLT_MAX;
    i32 k = have ? idx : 0x7fffffff;
#pragma unroll
    for (int o = kGroupLanes / 2; o >= 1; o >>= 1) {
        const float os = __shfl_xor_sync(gm, s, o);
        const i32 ok = __shfl_xor_sync(gm, k, o);
        if (os > s || (os == s && ok < k)) {
            s = os;
            k = ok;
        }
    }
    return Winner { s, k };
}

// faces of one hull against the other hull's vertices: lane `sub` measures faces
// sub, sub + 8, ... in ascending order with the scalar rule, then the group combines
__device__ __forceinline__ Winner groupFaceQuery(unsigned gm, int sub, const Plane *planes, u32 num_faces,
                                                 const HullInWorld &other)
{
    float best = -FLT_MAX;
    i32 best_face = 0x7fffffff;
    bool have = false;
    for (u32 f = (u32)sub; f < num_faces; f += kGroupLanes) {
        const float sep = hullSupportDistance(planes[f], other);
        if (!have || sep > best) {
            // first element, or strictly greater than what this lane kept so far
            best = sep;
            best_face = (i32)f;
            have = true;
            if (sep > 0.f) break;    // the scalar loop stops at the first positive
        }
    }
    return groupSequentialWinner(gm, best, best_face, have);
}

// Executed by the kGroupLanes lanes of one group for the hull - hull pair `ps`
// (every lane holds the same copy); lane sub 0 writes the contact (if any) to
// `out`.  Returns, on every lane of the group, whether a contact was made.
__device__ bool hullHullGroup(EngineState &S, const PairSetup &ps, HullScratch &scratch, const unsigned gm,
                              const int sub, Contact &out)
{
    const HalfEdgeMesh &am = ps.aPrim->hull.halfEdgeMesh;
    const HalfEdgeMesh &bm = ps.bPrim->hull.halfEdgeMesh;
    const u32 nva = am.numVertices, nvb = bm.numVertices, nfa = am.numFaces, nfb = bm.numFaces;
    if (nva > (u32)kMaxHullVerts || nvb > (u32)kMaxHullVerts ||
            nfa > (u32)kMaxHullFaces || nfb > (u32)kMaxHullFaces) {
        if (sub == 0) atomicOr(&S.errorFlags, (u32)ErrPhysicsOverflow);
        return false;
    }

    // -- both hulls into shared memory (vertex = R S v + t, plane via R S^-1)
    Vector3 *verts_a = scratch.verts, *verts_b = scratch.verts + kMaxHullVerts;
    Plane *planes_a = scratch.planes, *planes_b = scratch.planes + kMaxHullFaces;
    {
        const Mat3x3 rot_a = Mat3x3::fromQuat(ps.aRot), rot_b = Mat3x3::fromQuat(ps.bRot);
        const Mat3x3 vm_a = rot_a * ps.aScale, vm_b = rot_b * ps.bScale;
        const Mat3x3 nm_a = rot_a * ps.aScale.inv(), nm_b = rot_b * ps.bScale.inv();
        const Vector3 a_pos = ps.aPos, b_pos = ps.bPos;
#pragma unroll 1
        for (u32 i = (u32)sub; i < nva + nvb; i += kGroupLanes) {
            if (i < nva) verts_a[i] = vm_a * am.vertices[i] + a_pos;
            else verts_b[i - nva] = vm_b * bm.vertices[i - nva] + b_pos;
        }
#pragma unroll 1
        for (u32 i = (u32)sub; i < nfa + nfb; i += kGroupLanes) {
            const bool is_a = i < nfa;
            const Plane local = is_a ? am.facePlanes[i] : bm.facePlanes[i - nfa];
            const Mat3x3 &vm = is_a ? vm_a : vm_b;
            const Mat3x3 &nm = is_a ? nm_a : nm_b;
            const Vector3 on_plane = vm * (local.normal * local.d) + (is_a ? a_pos : b_pos);
            const Vector3 n = (nm * local.normal).normalize();
            (is_a ? planes_a[i] : planes_b[i - nfa]) = Plane { n, dot(n, on_plane) };
        }
    }
    __syncwarp(gm);
    // centres: vertex sums in index order (float addition is not associative)
    Vector3 center_a = Vector3::zero();
#pragma unroll 1
    for (u32 i = 0; i < nva; i++) center_a += verts_a[i];
    center_a /= (float)nva;

    HullInWorld a { &am, verts_a, planes_a, nva, nfa, center_a };
    HullInWorld b { &bm, verts_b, planes_b, nvb, nfb, Vector3::zero() };

    // -- face queries (A's faces vs B, then B's vs A)
    const Winner fa = groupFaceQuery(gm, sub, planes_a, nfa, b);
    if (fa.sep > 0.0f) return false;
    const Winner fb = groupFaceQuery(gm, sub, planes_b, nfb, a);
    if (fb.sep > 0.0f) return false;
    const float sep_a = fa.sep, sep_b = fb.sep;
    const i32 face_a = fa.idx, face_b = fb.idx;

    // -- edge query: pair p = ia * eb + ib, lanes take p = sub, sub + 8, ...
    const u32 ea = am.numHalfEdges / 2, eb = bm.numHalfEdges / 2;
    float e_sep = -FLT_MAX;
    i32 e_pair = 0x7fffffff;
    Vector3 e_normal = Vector3::zero();
#pragma unroll 1
    for (u32 p = (u32)sub; p < ea * eb; p += kGroupLanes) {
        const u32 ha = (p / eb) * 2, hb = (p % eb) * 2;
        const HalfEdge a0 = am.halfEdges[ha];
        const HalfEdge a1 = am.halfEdges[ha ^ 1u];
        const HalfEdge b0 = bm.halfEdges[hb];
        const HalfEdge b1 = bm.halfEdges[hb ^ 1u];
        float sep = -FLT_MAX;
        Vector3 normal = Vector3::zero();
        if (gaussMapArcsCross(planes_a[a0.face].normal, planes_a[a1.face].normal,
                              -planes_b[b0.face].normal, -planes_b[b1.face].normal)) {
            const Vector3 pa = verts_a[a0.rootVertex];
            const Vector3 qa = verts_a[am.halfEdges[a0.next].rootVertex];
            const Vector3 pb = verts_b[b0.rootVertex];
            const Vector3 qb = verts_b[bm.halfEdges[b0.next].rootVertex];
            const Vector3 axis = (qa - pa).cross(qb - pb);
            const float len2 = axis.length2();
            if (len2 != 0) {
                normal = axis * (1.f / sqrtf(len2));
                if (normal.dot(pa - center_a) < 0.0f) normal = -normal;
                sep = normal.dot(pb - pa);
            }
        }
        if (sep > e_sep) {
            e_sep = sep;
            e_pair = (i32)p;
            e_normal = normal;
            if (sep > 0) break;
        }
    }
    {
        const float my_sep = e_sep;
        const i32 my_pair = e_pair;
        const Winner ew = groupSequentialWinner(gm, e_sep, e_pair, my_pair != 0x7fffffff);
        e_sep = ew.sep;
        e_pair = ew.idx;
        const unsigned owner = __ballot_sync(gm, my_pair == e_pair && my_pair != 0x7fffffff &&
                                                 my_sep == e_sep);
        if (owner) {
            const int src = __ffs(owner) - 1;
            e_normal.x = __shfl_sync(gm, e_normal.x, src);
            e_normal.y = __shfl_sync(gm, e_normal.y, src);
            e_normal.z = __shfl_sync(gm, e_normal.z, src);
        } else {
            // nothing beat the initial -FLT_MAX: the scalar scan keeps its defaults
            e_sep = -FLT_MAX;
            e_pair = 0;
            e_normal = Vector3::zero();
        }
    }
    if (e_sep > 0.0f) return false;

    // -- contact generation on the group's first lane (data already in shared memory)
    bool made = false;
    if (sub == 0) {
        const bool face_contact_a = sep_a > e_sep;
        const bool face_contact_b = sep_b > e_sep;
        if (face_contact_a || face_contact_b) {
            const bool a_is_ref = sep_a >= sep_b;
            const Plane ref_plane = a_is_ref ? planes_a[face_a] : planes_b[face_b];
            const i32 ref_face = a_is_ref ? face_a : face_b;
            const HullInWorld &ref = a_is_ref ? a : b;
            const HullInWorld &inc = a_is_ref ? b : a;
            const i32 inc_face = mostOpposedFace(inc, ref_plane.normal);
            ManifoldOut m = faceFaceManifold(ref_plane, ref_face, inc_face, ref, inc,
                                             scratch.clipA, scratch.clipB);
            if (m.count > 0) {
                if (a_is_ref) {
                    writeContact(out, ps.aArch, ps.aRow, ps.bArch, ps.bRow, m);
                    out.refInfo = ps.aInfo; out.altInfo = ps.bInfo;
                } else {
                    writeContact(out, ps.bArch, ps.bRow, ps.aArch, ps.aRow, m);
                    out.refInfo = ps.bInfo; out.altInfo = ps.aInfo;
                }
                made = true;
            }
        } else {
            // edge - edge: contact point on A's edge, depth = -separation, A is ref
            const u32 ha = ((u32)e_pair / eb) * 2, hb = ((u32)e_pair % eb) * 2;
            const HalfEdge he_a = am.halfEdges[ha];
            const HalfEdge he_b = bm.halfEdges[hb];
            const Vector3 p = closestOnFirstSegment(
                verts_a[he_a.rootVertex], verts_a[am.halfEdges[he_a.next].rootVertex],
                verts_b[he_b.rootVertex], verts_b[bm.halfEdges[he_b.next].rootVertex]);
            writeContact(out, ps.aArch, ps.aRow, ps.bArch, ps.bRow, singlePoint(p, e_normal, -e_sep));
            out.refInfo = ps.aInfo; out.altInfo = ps.bInfo;
            made = true;
        }
    }
    return __shfl_sync(gm, made ? 1 : 0, (__ffs(gm) - 1)) != 0;
}

// ---- narrowphase, dense over the candidates of ALL worlds ------------------------------------
// The contact of candidate i of world w lives in slot (w, i), so nothing here
// needs per-world ordering:
//   physNarrowSimpleKernel  one THREAD per candidate (a block flattens the candidate
//       lists of kNarrowWorldsPerBlock worlds, so lanes stay busy whatever the
//       per-world counts are): pair setup + primitive-box reject; sphere / plane
//       pair types are finished on the spot, hull - hull survivors are queued;
//   physNarrowHullKernel    one 8-lane GROUP per queued hull - hull pair, groups
//       stride over the queue (4 pairs in flight per warp, every lane busy);
//   orderContacts (prologue of the position solve) lists each world's hits in
//       candidate order and assigns the dependency levels.
#ifndef MB2_NS_MINB
#define MB2_NS_MINB 8      // B200, room: 6 blocks/SM (85 regs) 1.094 ms/step, 8 (64 regs) 1.074
#endif
#ifndef MB2_NH_MINB
#define MB2_NH_MINB 12     // 8 (128 regs): 1.094, 12 (85): 1.074, 16 (64): 1.081
#endif
constexpr int kNarrowWorldsPerBlock = 8;   // 4 worlds x 64 threads: 1.105
constexpr int kNarrowSimpleThreads = 128;

template <bool SPHERE_HULL>
__global__ void __launch_bounds__(kNarrowSimpleThreads, MB2_NS_MINB)
physNarrowSimpleKernel(EngineState *Sp)
{
    EngineState &S = *Sp;
    const PhysicsState &P = *S.physics;
    fillColCache(S, P);
    __shared__ i32 first[kNarrowWorldsPerBlock + 1];
    const i32 w0 = (i32)blockIdx.x * kNarrowWorldsPerBlock;
    if (threadIdx.x == 0) {
        i32 acc = 0;
        for (int k = 0; k < kNarrowWorldsPerBlock; k++) {
            first[k] = acc;
            if (w0 + k < (i32)S.numWorlds) acc += P.candCounts[w0 + k];
        }
        first[kNarrowWorldsPerBlock] = acc;
    }
    __syncthreads();
    const i32 total = first[kNarrowWorldsPerBlock];
    const int lane = threadIdx.x & 31;

    for (i32 j0 = 0; j0 < total; j0 += kNarrowSimpleThreads) {
        const i32 j = j0 + (i32)threadIdx.x;
        const bool have = j < total;
        i32 w = w0, i = 0;
        u32 test = 0;
        if (have) {
            int k = 0;
            while (j >= first[k + 1]) k++;
            w = w0 + k;
            i = j - first[k];
            const size_t slot = (size_t)w * P.maxCandidatesPerWorld + i;
            const ObjectManager &objs = worldObjects(S, P, w);
            const PairSetup ps = setupPair(S, P, objs, P.candidates[slot]);
            test = ps.test;
            bool hit = false;
            if (test != 0 && test != 2) {
                Contact c;
                hit = narrowphaseSimple<SPHERE_HULL>(S, ps, c);
                if (hit) {
                    // single-point and hull - plane contacts store (ref, alt) = (b, a)
                    c.refInfo = ps.bInfo;
                    c.altInfo = ps.aInfo;
                    P.contacts[slot] = c;
                }
            }
            P.candHit[slot] = hit ? 1 : 0;
        }
        // queue the hull - hull survivors (one atomic per warp)
        const unsigned hh = __ballot_sync(0xffffffffu, have && test == 2);
        if (hh) {
            const int leader = __ffs(hh) - 1;
            i32 base = 0;
            if (lane == leader) base = atomicAdd(P.hullQueueCount, __popc(hh));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (have && test == 2) {
                P.hullQueue[base + __popc(hh & ((1u << lane) - 1u))] = HullQueueEntry { w, i };
            }
        }
    }
}

constexpr int kNarrowHullThreads = 64;

__global__ void __launch_bounds__(kNarrowHullThreads, MB2_NH_MINB)
physNarrowHullKernel(EngineState *Sp)
{
    EngineState &S = *Sp;
    const PhysicsState &P = *S.physics;
    fillColCache(S, P);
    __shared__ HullScratch scratch[kNarrowHullThreads / kGroupLanes];
    const int lane = threadIdx.x & 31;
    const int sub = lane % kGroupLanes;
    const int group_in_warp = lane / kGroupLanes;
    const int group_in_block = threadIdx.x / kGroupLanes;
    const unsigned gm = ((1u << kGroupLanes) - 1u) << (group_in_warp * kGroupLanes);
    const i32 count = *P.hullQueueCount;
    const i32 groups_per_block = kNarrowHullThreads / kGroupLanes;
    for (i32 e = (i32)blockIdx.x * groups_per_block + group_in_block; e < count;
         e += (i32)gridDim.x * groups_per_block) {
        const HullQueueEntry ent = P.hullQueue[e];
        const size_t slot = (size_t)ent.world * P.maxCandidatesPerWorld + ent.cand;
        const ObjectManager &objs = worldObjects(S, P, ent.world);
        const PairSetup ps = setupPairImpl<false>(S, P, objs, P.candidates[slot]);
        const bool made = hullHullGroup(S, ps, scratch[group_in_block], gm, sub, P.contacts[slot]);
        if (sub == 0 && made) P.candHit[slot] = 1;
        __syncwarp(gm);
    }
}

// Prologue of the position solve, run by the LPW lanes that own world w: list
// the world's contact slots in candidate order and give every contact its
// dependency level (see Contact::level) -- a sequential scan by the group's
// first lane over flags / body infos its lanes fetched in parallel.
template <int LPW>
__device__ __forceinline__ void orderContacts(EngineState &S, const PhysicsState &P, const i32 w, const bool valid,
                                              const int lane, i32 *last_level /* [kMaxLevelBodies] of this world */)
{
    constexpr unsigned kGroupMask = LPW == 32 ? 0xffffffffu : ((1u << (LPW & 31)) - 1u);
    const int sub = lane & (LPW - 1);
    const int group_shift = (lane / LPW) * LPW;
    const unsigned gm = kGroupMask << group_shift;

    for (int i = sub; i < kMaxLevelBodies; i += LPW) last_level[i] = 0;
    __syncwarp(gm);

    const i32 n = valid ? P.candCounts[w] : 0;
    const size_t base_slot = (size_t)w * P.maxCandidatesPerWorld;
    Contact *contacts = P.contacts + base_slot;
    i32 *order = P.contactOrder + (size_t)w * P.maxContactsPerWorld;
    i32 running = 0, max_level = 0, seq_level = 0;

    for (i32 base = 0; base < n; base += LPW) {
        const i32 i = base + sub;
        const bool hit = i < n && P.candHit[base_slot + i] != 0;
        u32 a = 0, b = 0;
        if (hit) {
            a = contacts[i].refInfo;
            b = contacts[i].altInfo;
        }
        const unsigned hits = (__ballot_sync(gm, hit) >> group_shift) & kGroupMask;
        i32 my_level = 0;
        unsigned todo = hits;
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const u32 sa_info = __shfl_sync(gm, a, group_shift + src);
            const u32 sb_info = __shfl_sync(gm, b, group_shift + src);
            i32 lvl = 0;
            if (sub == 0) {
                const u32 sa = sa_info >> 1, sb = sb_info >> 1;
                if (sa >= (u32)kMaxLevelBodies || sb >= (u32)kMaxLevelBodies) {
                    lvl = max_level + 1;          // unknown body: strictly after everything so far
                    seq_level = lvl;
                } else {
                    i32 dep = seq_level;
                    if (sa_info & 1u) dep = max(dep, last_level[sa]);
                    if (sb_info & 1u) dep = max(dep, last_level[sb]);
                    lvl = dep + 1;
                    if (sa_info & 1u) last_level[sa] = lvl;
                    if (sb_info & 1u) last_level[sb] = lvl;
                }
                if (lvl > max_level) max_level = lvl;
            }
            lvl = __shfl_sync(gm, lvl, group_shift);
            if (sub == src) my_level = lvl;
        }
        if (hit) {
            const i32 at = running + __popc(hits & ((1u << sub) - 1u));
            contacts[i].level = my_level;
            if (at < P.maxContactsPerWorld) order[at] = i;
        }
        running += __popc(hits);
    }
    if (valid && sub == 0) {
        if (running > P.maxContactsPerWorld) {
            atomicOr(&S.errorFlags, (u32)ErrPhysicsOverflow);
            running = P.maxContactsPerWorld;
        }
        P.contactCounts[w] = running;
        P.contactMaxLevel[w] = max_level;
    }
    __syncwarp(gm);
}

// =============================================================================================
// XPBD constraint solve (per world, sequential Gauss-Seidel in contact order)
// =============================================================================================

struct BodyPair {
    float invM1, invM2;
    Vector3 invI1, invI2;
};

__device__ __forceinline__ float positionalLambda(Vector3 tq1, Vector3 tq2, Vector3 ra1, Vector3 ra2,
                                                  float inv_m1, float inv_m2, float c, float alpha)
{
    float w1 = inv_m1 + dot(tq1, ra1);
    float w2 = inv_m2 + dot(tq2, ra2);
    return -c / (w1 + w2 + alpha);
}

__device__ __forceinline__ void applyPositional(Vector3 &x1, Vector3 &x2, Quat &q1, Quat &q2,
                                                Vector3 rot_axis1, Vector3 rot_axis2,
                                                float inv_m1, float inv_m2, Vector3 n, float lambda)
{
    x1 += lambda * inv_m1 * n;
    x2 -= lambda * inv_m2 * n;
    const float half = 0.5f * lambda;
    const Vector3 w1 = q1.rotateVec(half * rot_axis1);
    const Vector3 w2 = q2.rotateVec(half * rot_axis2);
    q1 += Quat::fromAngularVec(w1) * q1;
    q2 -= Quat::fromAngularVec(w2) * q2;
    q1 = q1.normalize();
    q2 = q2.normalize();
}

__device__ __forceinline__ float positionalCorrection(Vector3 &x1, Vector3 &x2, Quat &q1, Quat &q2,
                                                      Vector3 r1, Vector3 r2, const BodyPair &bp,
                                                      Vector3 n_world, float c, float alpha)
{
    const Vector3 n1 = q1.inv().rotateVec(n_world);
    const Vector3 n2 = q2.inv().rotateVec(n_world);
    const Vector3 tq1 = cross(r1, n1);
    const Vector3 tq2 = cross(r2, n2);
    const Vector3 ra1 = mulDiag(bp.invI1, tq1);
    const Vector3 ra2 = mulDiag(bp.invI2, tq2);
    const float lambda = positionalLambda(tq1, tq2, ra1, ra2, bp.invM1, bp.invM2, c, alpha);
    applyPositional(x1, x2, q1, q2, ra1, ra2, bp.invM1, bp.invM2, n_world, lambda);
    return lambda;
}

// depth-weighted mean contact point + deepest penetration (xpbd.cpp:421-449);
// false when all depths are zero
__device__ bool meanContact(const Contact &c, Vector3 *mean, float *deepest)
{
    float max_pen = -FLT_MAX, sum = 0.f;
    for (int i = 0; i < c.numPoints; i++) {
        float pen = c.points[i][3];
        if (pen > max_pen) max_pen = pen;
        sum += pen;
    }
    if (sum == 0.f) return false;
    Vector3 acc = Vector3::zero();
    for (int i = 0; i < c.numPoints; i++) {
        acc += c.points[i][3] / sum * Vector3 { c.points[i][0], c.points[i][1], c.points[i][2] };
    }
    *mean = acc;
    *deepest = max_pen;
    return true;
}

__device__ __forceinline__ void localArms(const PreSolvePositional &pre1, const PreSolvePositional &pre2,
                                          Vector3 p1, float depth, Vector3 n, Vector3 *r1, Vector3 *r2)
{
    const Vector3 p2 = p1 - n * depth;
    *r1 = pre1.q.inv().rotateVec(p1 - pre1.x);
    *r2 = pre2.q.inv().rotateVec(p2 - pre2.x);
}

__device__ __forceinline__ BodyPair bodyPair(const EngineState &S, const PhysicsState &P,
                                             const ObjectManager &objs, u32 a1, i32 r1, u32 a2, i32 r2,
                                             float *mu_s, float *mu_d)
{
    const RigidBodyMetadata m1 = objs.metadata[locCol<i32>(S, P, a1, r1, PCObjectID)];
    const RigidBodyMetadata m2 = objs.metadata[locCol<i32>(S, P, a2, r2, PCObjectID)];
    BodyPair bp { m1.mass.invMass, m2.mass.invMass, m1.mass.invInertiaTensor, m2.mass.invInertiaTensor };
    if (locCol<ResponseType>(S, P, a1, r1, PCResponseType) == ResponseType::Static) {
        bp.invM1 = 0.f;
        bp.invI1 = Vector3::zero();
    }
    if (locCol<ResponseType>(S, P, a2, r2, PCResponseType) == ResponseType::Static) {
        bp.invM2 = 0.f;
        bp.invI2 = Vector3::zero();
    }
    *mu_s = 0.5f * (m1.friction.muS + m2.friction.muS);
    *mu_d = 0.5f * (m1.friction.muD + m2.friction.muD);
    return bp;
}

// normal push-out along the contact normal + static friction (xpbd.cpp:347-419, 454-550)
__device__ void solveContactPosition(EngineState &S, const PhysicsState &P, const ObjectManager &objs,
                                     Contact &c)
{
    c.lambdaN = 0.f;

    Vector3 &x1_ref = locCol<Vector3>(S, P, c.refArch, c.refRow, PCPosition);
    Vector3 &x2_ref = locCol<Vector3>(S, P, c.altArch, c.altRow, PCPosition);
    Quat &q1_ref = locCol<Quat>(S, P, c.refArch, c.refRow, PCRotation);
    Quat &q2_ref = locCol<Quat>(S, P, c.altArch, c.altRow, PCRotation);
    const SubstepPrevState prev1 = locCol<SubstepPrevState>(S, P, c.refArch, c.refRow, PCPrevState);
    const SubstepPrevState prev2 = locCol<SubstepPrevState>(S, P, c.altArch, c.altRow, PCPrevState);
    const PreSolvePositional pre1 = locCol<PreSolvePositional>(S, P, c.refArch, c.refRow, PCPreSolvePos);
    const PreSolvePositional pre2 = locCol<PreSolvePositional>(S, P, c.altArch, c.altRow, PCPreSolvePos);

    float mu_s, mu_d;
    const BodyPair bp = bodyPair(S, P, objs, c.refArch, c.refRow, c.altArch, c.altRow, &mu_s, &mu_d);

    Vector3 x1 = x1_ref, x2 = x2_ref;
    Quat q1 = q1_ref, q2 = q2_ref;

    Vector3 mean;
    float deepest;
    if (!meanContact(c, &mean, &deepest)) return;

    const Vector3 n = c.normal;
    Vector3 r1, r2;
    localArms(pre1, pre2, mean, deepest, n, &r1, &r2);

    Vector3 p1 = q1.rotateVec(r1) + x1;
    Vector3 p2 = q2.rotateVec(r2) + x2;
    const float d = dot(p1 - p2, n);
    if (d > 0) {
        const float lambda_n = positionalCorrection(x1, x2, q1, q2, r1, r2, bp, n, d, 0);
        c.lambdaN = lambda_n;

        const Vector3 p1_hat = prev1.prevRotation.rotateVec(r1) + prev1.prevPosition;
        const Vector3 p2_hat = prev2.prevRotation.rotateVec(r2) + prev2.prevPosition;
        p1 = q1.rotateVec(r1) + x1;
        p2 = q2.rotateVec(r2) + x2;
        const Vector3 dp = (p1 - p1_hat) - (p2 - p2_hat);
        const Vector3 dp_t = dp - dot(dp, n) * n;
        const float slide = dp_t.length();
        if (slide > 0.f) {
            const Vector3 t_world = dp_t / slide;
            const Vector3 t1 = q1.inv().rotateVec(t_world);
            const Vector3 t2 = q2.inv().rotateVec(t_world);
            const Vector3 tq1 = cross(r1, t1);
            const Vector3 tq2 = cross(r2, t2);
            const Vector3 ra1 = mulDiag(bp.invI1, tq1);
            const Vector3 ra2 = mulDiag(bp.invI2, tq2);
            const float lambda_t = positionalLambda(tq1, tq2, ra1, ra2, bp.invM1, bp.invM2, slide, 0);
            if (lambda_t > lambda_n * mu_s) {
                applyPositional(x1, x2, q1, q2, ra1, ra2, bp.invM1, bp.invM2, t_world, lambda_t);
            }
        }
    }

    x1_ref = x1;
    x2_ref = x2;
    q1_ref = q1;
    q2_ref = q2;
}

__device__ void angularCorrection(Quat &q1, Quat &q2, const BodyPair &bp, Vector3 axis_world, float theta)
{
    const Vector3 n1 = q1.inv().rotateVec(axis_world);
    const Vector3 n2 = q2.inv().rotateVec(axis_world);
    const Vector3 ra1 = mulDiag(bp.invI1, n1);
    const Vector3 ra2 = mulDiag(bp.invI2, n2);
    const float w1 = dot(n1, ra1);
    const float w2 = dot(n2, ra2);
    const float lambda = -theta / (w1 + w2 + 0);
    const float half = 0.5f * lambda;
    const Quat u1 = Quat::fromAngularVec(q1.rotateVec(half * ra1));
    const Quat u2 = Quat::fromAngularVec(q2.rotateVec(half * ra2));
    q1 = (q1 + u1 * q1).normalize();
    q2 = (q2 - u2 * q2).normalize();
}

// fixed / hinge joints (xpbd.cpp:552-718)
__device__ void solveJoint(EngineState &S, const PhysicsState &P, const ObjectManager &objs,
                           const JointConstraint &j)
{
    if (j.e1.id < 0 || j.e2.id < 0 || j.e1.id >= S.entityCapacity || j.e2.id >= S.entityCapacity) return;
    const EntitySlot s1 = S.entitySlots[j.e1.id];
    const EntitySlot s2 = S.entitySlots[j.e2.id];
    if (s1.gen != j.e1.gen || s2.gen != j.e2.gen) return;
    const u32 a1 = (u32)s1.a, a2 = (u32)s2.a;
    const i32 r1row = s1.b, r2row = s2.b;
    if (!isBodyArchetype(a1) || !isBodyArchetype(a2)) return;

    Vector3 &x1_ref = locCol<Vector3>(S, P, a1, r1row, PCPosition);
    Vector3 &x2_ref = locCol<Vector3>(S, P, a2, r2row, PCPosition);
    Quat &q1_ref = locCol<Quat>(S, P, a1, r1row, PCRotation);
    Quat &q2_ref = locCol<Quat>(S, P, a2, r2row, PCRotation);
    Vector3 x1 = x1_ref, x2 = x2_ref;
    Quat q1 = q1_ref, q2 = q2_ref;

    float mu_s, mu_d;
    const BodyPair bp = bodyPair(S, P, objs, a1, r1row, a2, r2row, &mu_s, &mu_d);

    Vector3 correction;
    if (j.type == JointConstraint::Type::Fixed) {
        const Quat o1 = (q1 * j.fixed.attachRot1).normalize();
        const Quat o2 = (q2 * j.fixed.attachRot2).normalize();
        const Quat diff = o1 * o2.inv();
        Vector3 dq = 2.f * Vector3 { diff.x, diff.y, diff.z };
        const float mag = dq.length();
        if (mag > 0) {
            dq /= mag;
            angularCorrection(q1, q2, bp, dq, mag);
        }
        const Vector3 p1 = q1.rotateVec(j.r1) + x1;
        const Vector3 p2 = q2.rotateVec(j.r2) + x2;
        const Vector3 delta = p2 - p1;
        const Quat frame = (q1 * j.fixed.attachRot1).normalize();
        const Vector3 ax_a = frame.rotateVec(madrona::math::fwd);
        const Vector3 ax_b = frame.rotateVec(madrona::math::right);
        const Vector3 ax_c = cross(ax_a, ax_b);
        correction = Vector3::zero();
        correction -= (dot(delta, ax_a) - j.fixed.separation) * ax_a;
        correction -= dot(delta, ax_b) * ax_b;
        correction -= dot(delta, ax_c) * ax_c;
    } else {
        const Vector3 w1 = q1.rotateVec(j.hinge.a1Local);
        const Vector3 w2 = q2.rotateVec(j.hinge.a2Local);
        Vector3 dq = cross(w1, w2);
        const float mag = dq.length();
        if (mag > 0) {
            dq /= mag;
            angularCorrection(q1, q2, bp, dq, mag);
        }
        const Vector3 p1 = q1.rotateVec(j.r1) + x1;
        const Vector3 p2 = q2.rotateVec(j.r2) + x2;
        correction = p2 - p1;
    }

    const float cmag = correction.length();
    if (cmag > 0.f) {
        correction /= cmag;
        positionalCorrection(x1, x2, q1, q2, j.r1, j.r2, bp, correction, cmag, 0);
    }
    x1_ref = x1;
    x2_ref = x2;
    q1_ref = q1;
    q2_ref = q2;
}

// Contact sweep of one world by a group of LPW lanes (32 / LPW worlds share a
// warp).  Contacts are swept level by level (Contact::level): the contacts of a
// level run concurrently, levels run in order -- same floats as the reference's
// one-thread-per-world sequential sweep (xpbd.cpp:720-736).  Contacts are taken
// in chunks of 32, chunk-major: a later chunk only holds later contacts and the
// levels inside a chunk run in order, so any two contacts sharing a mutable body
// keep their sequential order.  Inside a level the members are compacted onto
// the group's first lanes (ballot + find-nth-set).
// The solves are latency bound with ~4 contacts per level, so several worlds per
// warp multiply the worlds in flight per SM at no register cost (measured on B200, room
// 8192 worlds: 32 lanes/world 1.103 ms/step, 16: 1.097, 8: 1.080).
#ifndef MB2_SOLVER_LPW
#define MB2_SOLVER_LPW 8
#endif
constexpr int kSolverLanes = MB2_SOLVER_LPW;

template <int LPW, typename Fn>
__device__ __forceinline__ void sweepContactLevels(const Contact *contacts, const i32 *order, const i32 n,
                                                   const i32 levels, const int lane, Fn &&solve)
{
    constexpr int kPerLane = 32 / LPW;
    constexpr unsigned kGroupMask = LPW == 32 ? 0xffffffffu : ((1u << (LPW & 31)) - 1u);
    const int sub = lane & (LPW - 1);
    const int group_shift = (lane / LPW) * LPW;

    i32 n_max = n, levels_max = levels;
#pragma unroll
    for (int o = LPW; o < 32; o <<= 1) {
        n_max = max(n_max, __shfl_xor_sync(0xffffffffu, n_max, o));
        levels_max = max(levels_max, __shfl_xor_sync(0xffffffffu, levels_max, o));
    }

    for (i32 base = 0; base < n_max; base += 32) {
        i32 lv[kPerLane];
#pragma unroll
        for (int r = 0; r < kPerLane; r++) {
            const i32 i = base + r * LPW + sub;
            lv[r] = i < n ? contacts[order[i]].level : 0;
        }
        for (i32 lvl = 1; lvl <= levels_max; lvl++) {
            unsigned members = 0;
#pragma unroll
            for (int r = 0; r < kPerLane; r++) {
                const unsigned b = __ballot_sync(0xffffffffu, lv[r] == lvl);
                members |= ((b >> group_shift) & kGroupMask) << (r * LPW);
            }
            const int count = __popc(members);
            for (int k = sub; k < count; k += LPW) {
                // member bit m = r * LPW + lane-in-group: fetch that lane's slot[r]
                const int m = (int)__fns(members, 0, k + 1);
                solve(order[base + m]);
            }
            __syncwarp();
        }
    }
}

// Joints follow the contacts, sequentially.
__device__ void phaseSolvePositions(EngineState &S, const PhysicsState &P, const i32 w, const bool valid,
                                    const int lane)
{
    const ObjectManager &objs = worldObjects(S, P, w);

    Contact *contacts = P.contacts + (size_t)w * P.maxCandidatesPerWorld;
    const i32 *order = P.contactOrder + (size_t)w * P.maxContactsPerWorld;
    const i32 n = valid ? P.contactCounts[w] : 0;
    const i32 levels = valid ? P.contactMaxLevel[w] : 0;
    sweepContactLevels<kSolverLanes>(contacts, order, n, levels, lane, [&](i32 i) {
        solveContactPosition(S, P, objs, contacts[i]);
    });

    const TableDesc &jt = S.tables[P.jointArchetype];
    if (valid && (lane & (kSolverLanes - 1)) == 0 && jt.numRows > 0) {
        const JointConstraint *joints = (const JointConstraint *)jt.columns[P.jointCol];
        const i32 *jw = (const i32 *)jt.columns[1];
        const i32 first = jt.worldOffsets[w];
        const i32 count = jt.worldCounts[w];
        for (i32 r = first; r < first + count; r++) {
            if (jw[r] < 0) continue;
            solveJoint(S, P, objs, joints[r]);
        }
    }
}

__device__ __forceinline__ Vector3 relativeVelocity(Vector3 v1, Vector3 v2, Vector3 o1, Vector3 o2,
                                                    Vector3 d1, Vector3 d2)
{
    return (v1 + cross(o1, d1)) - (v2 + cross(o2, d2));
}

// restitution on the mean contact, then dynamic friction per contact point
// (xpbd.cpp:781-1039)
__device__ void solveContactVelocity(EngineState &S, const PhysicsState &P, const ObjectManager &objs,
                                     const Contact &c, float h, float restitution_threshold)
{
    Velocity &vel1_ref = locCol<Velocity>(S, P, c.refArch, c.refRow, PCVelocity);
    Velocity &vel2_ref = locCol<Velocity>(S, P, c.altArch, c.altRow, PCVelocity);
    const Quat q1 = locCol<Quat>(S, P, c.refArch, c.refRow, PCRotation);
    const Quat q2 = locCol<Quat>(S, P, c.altArch, c.altRow, PCRotation);
    const PreSolvePositional pre1 = locCol<PreSolvePositional>(S, P, c.refArch, c.refRow, PCPreSolvePos);
    const PreSolvePositional pre2 = locCol<PreSolvePositional>(S, P, c.altArch, c.altRow, PCPreSolvePos);
    const PreSolveVelocity pv1 = locCol<PreSolveVelocity>(S, P, c.refArch, c.refRow, PCPreSolveVel);
    const PreSolveVelocity pv2 = locCol<PreSolveVelocity>(S, P, c.altArch, c.altRow, PCPreSolveVel);

    float mu_s, mu_d;
    const BodyPair bp = bodyPair(S, P, objs, c.refArch, c.refRow, c.altArch, c.altRow, &mu_s, &mu_d);

    Vector3 v1 = vel1_ref.linear, o1 = vel1_ref.angular;
    Vector3 v2 = vel2_ref.linear, o2 = vel2_ref.angular;
    const Vector3 n = c.normal;

    {
        Vector3 mean;
        float deepest;
        if (!meanContact(c, &mean, &deepest)) return;
        Vector3 r1, r2;
        localArms(pre1, pre2, mean, deepest, n, &r1, &r2);

        const Vector3 v_bar = relativeVelocity(pv1.v, pv2.v, pv1.omega, pv2.omega,
                                               pre1.q.rotateVec(r1), pre2.q.rotateVec(r2));
        const float vn_bar = dot(n, v_bar);
        const Vector3 r1_world = q1.rotateVec(r1);
        const Vector3 r2_world = q2.rotateVec(r2);
        const Vector3 tq1 = cross(r1, q1.inv().rotateVec(n));
        const Vector3 tq2 = cross(r2, q2.inv().rotateVec(n));

        const Vector3 v = relativeVelocity(v1, v2, o1, o2, r1_world, r2_world);
        const float vn = dot(n, v);
        float e = 0.3f;
        if (fabsf(vn_bar) <= restitution_threshold) e = 0.f;
        const float target = fminf(-e * vn_bar, 0) - vn;
        const Vector3 ra1 = mulDiag(bp.invI1, tq1);
        const Vector3 ra2 = mulDiag(bp.invI2, tq2);
        const float w1 = bp.invM1 + dot(tq1, ra1);
        const float w2 = bp.invM2 + dot(tq2, ra2);
        const float inv_w = 1.f / (w1 + w2);
        const float impulse = target * inv_w;
        if (impulse != 0.f) {
            v1 += n * impulse * bp.invM1;
            v2 -= n * impulse * bp.invM2;
            o1 += q1.rotateVec(impulse * ra1);
            o2 -= q2.rotateVec(impulse * ra2);
        }
    }

    float pen_sum = 0.f;
    for (int i = 0; i < c.numPoints; i++) pen_sum += c.points[i][3];

    for (int i = 0; i < c.numPoints; i++) {
        Vector3 r1, r2;
        localArms(pre1, pre2, Vector3 { c.points[i][0], c.points[i][1], c.points[i][2] },
                  c.points[i][3], n, &r1, &r2);
        const Vector3 r1_world = q1.rotateVec(r1);
        const Vector3 r2_world = q2.rotateVec(r2);
        const float lambda = c.lambdaN * (c.points[i][3] / pen_sum);

        const Vector3 v = relativeVelocity(v1, v2, o1, o2, r1_world, r2_world);
        const float vn = dot(n, v);
        const Vector3 vt = v - n * vn;
        const float vt_len = vt.length();
        if (vt_len == 0.f) continue;
        const Vector3 dir = vt / vt_len;
        const Vector3 d1 = q1.inv().rotateVec(dir);
        const Vector3 d2 = q2.inv().rotateVec(dir);
        const Vector3 tq1 = cross(r1, d1);
        const Vector3 tq2 = cross(r2, d2);
        const Vector3 ra1 = mulDiag(bp.invI1, tq1);
        const Vector3 ra2 = mulDiag(bp.invI2, tq2);
        const float w1 = bp.invM1 + dot(tq1, ra1);
        const float w2 = bp.invM2 + dot(tq2, ra2);
        const float inv_w = 1.f / (w1 + w2);
        const float friction = mu_d * fabsf(lambda) * inv_w / h;
        const float corrected = -fminf(friction, vt_len);
        const float impulse = corrected * inv_w;
        if (impulse == 0.f) continue;
        v1 += dir * impulse * bp.invM1;
        v2 -= dir * impulse * bp.invM2;
        o1 += q1.rotateVec(impulse * ra1);
        o2 -= q2.rotateVec(impulse * ra2);
    }

    vel1_ref = Velocity { v1, o1 };
    vel2_ref = Velocity { v2, o2 };
}

__device__ void phaseSolveVelocities(EngineState &S, const PhysicsState &P, const i32 w, const bool valid,
                                     const int lane)
{
    const ObjectManager &objs = worldObjects(S, P, w);
    const PhysicsSystemState &params = worldParams(S, P, w);
    const Contact *contacts = P.contacts + (size_t)w * P.maxCandidatesPerWorld;
    const i32 *order = P.contactOrder + (size_t)w * P.maxContactsPerWorld;
    const i32 n = valid ? P.contactCounts[w] : 0;
    const i32 levels = valid ? P.contactMaxLevel[w] : 0;
    sweepContactLevels<kSolverLanes>(contacts, order, n, levels, lane, [&](i32 i) {
        solveContactVelocity(S, P, objs, contacts[i], params.h, params.restitutionThreshold);
    });
}

// =============================================================================================
// Launchers.  Row-parallel phases (leaf update, refit, integrate, velocity
// update) are grid-stride kernels over all rows of every body archetype;
// per-world phases (candidates, narrowphase, solves) give each world a warp.
// (A single fused warp-per-world kernel for the whole step was measured 2.4x
// SLOWER on B200: 18.7k SASS instructions with warps spread over every phase
// thrash the instruction cache, and the light phases inherit the narrowphase's
// 128-register occupancy.)
// =============================================================================================

enum PhysPhase : u32 {
    PhaseUpdateLeaves = 1, PhaseRebuild, PhaseRefit, PhaseFindCandidates, PhaseIntegrate,
    PhaseNarrowphase, PhaseSolvePositions, PhaseSetVelocities, PhaseSolveVelocities,
    PhaseNarrowphaseSpheres,      // narrowphase incl. the sphere - hull (GJK) path
    PhaseTGSVelocities, PhaseTGSPositions,
};

// (B200, room 8192 worlds, one box: 32-register build + a full wave of 8 blocks per SM
// 1.091 ms/step, unconstrained registers + 4 blocks per SM 1.067: the default)
#ifndef MB2_BODY_MINB
#define MB2_BODY_MINB 1
#endif
#ifndef MB2_BODY_BLOCKS_PER_SM
#define MB2_BODY_BLOCKS_PER_SM 4
#endif
template <u32 OP>
__global__ void __launch_bounds__(256, MB2_BODY_MINB)
physBodyKernel(EngineState *Sp)
{
    const EngineState &S = *Sp;
    const PhysicsState &P = *S.physics;
    if (blockIdx.y >= P.numBodyArchetypes) return;
    const BodyArchetype &b = P.bodies[blockIdx.y];
    const TableDesc &t = S.tables[b.archetype];
    const i32 n = t.numRows;
    const i32 *world_col = (const i32 *)t.columns[1];
    for (i32 row = blockIdx.x * blockDim.x + threadIdx.x; row < n; row += gridDim.x * blockDim.x) {
        const i32 w = world_col[row];
        if (w < 0) continue;
        if constexpr (OP == PhaseUpdateLeaves) {
            // leaf update, then straight into the refit of that leaf (it only
            // needs the leaf's own new box) -- unless the world asked for a
            // rebuild, whose thread refits all leaves afterwards
            rowUpdateLeaf(S, P, b, row, w);
            if (!worldBVH(S, P, w).forceRebuild) rowRefit(S, P, b, row, w);
        }
        else if constexpr (OP == PhaseRefit) rowRefit(S, P, b, row, w);
        else if constexpr (OP == PhaseIntegrate) rowIntegrate(S, P, b, row, w);
        else if constexpr (OP == PhaseSetVelocities) rowSetVelocity(S, P, b, row, w);
        else if constexpr (OP == PhaseTGSVelocities) rowTGSVelocities(S, P, b, row, w);
        else if constexpr (OP == PhaseTGSPositions) rowTGSPositions(S, P, b, row, w);
    }
}

__global__ void __launch_bounds__(128)
physRebuildKernel(EngineState *Sp)
{
    const EngineState &S = *Sp;
    const i32 w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= (i32)S.numWorlds) return;
    phaseRebuild(S, *S.physics, w, 0);
}

// lanes of a world's warp stride over its bodies (tables are world-sorted)
template <typename Fn>
__device__ __forceinline__ void forEachWorldBody(const EngineState &S, const PhysicsState &P, const i32 w,
                                                 const int lane, Fn &&fn)
{
    for (u32 bi = 0; bi < P.numBodyArchetypes; bi++) {
        const BodyArchetype &b = P.bodies[bi];
        const TableDesc &t = S.tables[b.archetype];
        const i32 first_row = t.worldOffsets[w];
        const i32 num_rows = t.worldCounts[w];
        for (i32 row = first_row + lane; row < first_row + num_rows; row += 32) {
            if (((const i32 *)t.columns[1])[row] != w) continue;   // destroyed, awaiting compaction
            fn(b, row);
        }
    }
}

// One warp per world; kPhysWarps worlds per block.  (Fusing neighbouring phases
// into one launch -- integrate -> narrowphase, position solve -> velocity update
// -> velocity solve -- was measured: no gain, and the bigger kernels miss the
// 32 KB instruction cache more; see DESIGN.md 3.2.)
template <u32 OP>
__global__ void __launch_bounds__(32 * kPhysWarps, 8)
physWorldKernel(EngineState *Sp)
{
    EngineState &S = *Sp;
    const PhysicsState &P = *S.physics;
    fillColCache(S, P);
    const int lane = threadIdx.x & 31;
    const int warp = threadIdx.x >> 5;
    if constexpr (OP == PhaseSolvePositions || OP == PhaseSolveVelocities) {
        // kSolverLanes lanes per world; the lanes of a warp past the last world idle along
        const i32 first_w = (i32)((blockIdx.x * blockDim.x + (threadIdx.x & ~31u)) / kSolverLanes);
        if (first_w >= (i32)S.numWorlds) return;
        const i32 my_w = (i32)((blockIdx.x * blockDim.x + threadIdx.x) / kSolverLanes);
        const bool valid = my_w < (i32)S.numWorlds;
        const i32 w = valid ? my_w : (i32)S.numWorlds - 1;
        if constexpr (OP == PhaseSolvePositions) {
            // the hull queue of this substep has been consumed: empty it for the next one
            if (blockIdx.x == 0 && threadIdx.x == 0) *P.hullQueueCount = 0;
            __shared__ i32 last_level[32 * kPhysWarps / kSolverLanes][kMaxLevelBodies];
            orderContacts<kSolverLanes>(S, P, w, valid, lane, last_level[threadIdx.x / kSolverLanes]);
            phaseSolvePositions(S, P, w, valid, lane);
        } else {
            phaseSolveVelocities(S, P, w, valid, lane);
        }
    } else {
        const i32 w = (i32)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
        if (w >= (i32)S.numWorlds) return;
        if constexpr (OP == PhaseFindCandidates) {
            // a new step: the hull - hull queue starts empty (solvers that never run the
            // position solve -- TGS -- would otherwise let it grow)
            if (blockIdx.x == 0 && threadIdx.x == 0) *P.hullQueueCount = 0;
            __shared__ CandidateScratch cand_scratch;
            phaseFindCandidates(S, P, w, lane, warp, cand_scratch);
        }
    }
}

// =============================================================================================
// Host side
// =============================================================================================

bool physicsHostCreate(Executor *ex, std::string *err)
{
    PhysicsHost *ph = new PhysicsHost();
    ex->physics = ph;
    memset(&ph->hPhys, 0, sizeof(PhysicsState));
    if (!devAlloc(ex, (void **)&ph->dPhys, sizeof(PhysicsState))) {
        *err = "physics state allocation failed";
        return false;
    }
    ex->hState->physics = ph->dPhys;
    return true;
}

bool physicsHostAfterRegistry(Executor *ex, const mb2_render_config *, std::string *err)
{
    PhysicsHost *ph = ex->physics;
    EngineState &S = *ex->hState;
    cudaMemcpy(&ph->hPhys, ph->dPhys, sizeof(PhysicsState), cudaMemcpyDeviceToHost);
    PhysicsState &P = ph->hPhys;
    if (!P.registered) return true;   // simulator without physics
    ph->active = true;

    // archetypes that carry the whole RigidBody bundle, ascending id == the
    // CPU backend's query iteration order
    P.numBodyArchetypes = 0;
    memset(P.bodyIndex, 0xff, sizeof(P.bodyIndex));
    for (uint32_t a = 0; a < S.numArchetypes; a++) {
        if (!S.archetypes[a].registered) continue;
        BodyArchetype b;
        b.archetype = a;
        bool all = true;
        for (int pc = 0; pc < PCCount; pc++) {
            int col = S.columnLookup[a][P.componentIDs[pc]];
            // TGS keeps no per-body solver state (its RigidBody bundle ends at ExternalTorque)
            const bool solver_state = pc == PCPrevState || pc == PCPreSolvePos || pc == PCPreSolveVel;
            if (col < 0 && !(solver_state && P.solver == 1u)) { all = false; break; }
            b.cols[pc] = col;
        }
        if (!all) continue;
        if (P.numBodyArchetypes >= (uint32_t)kMaxBodyArchetypes) {
            *err = "too many rigid-body archetypes";
            return false;
        }
        P.bodyIndex[a] = (signed char)P.numBodyArchetypes;
        P.bodies[P.numBodyArchetypes++] = b;
    }
    P.jointCol = S.columnLookup[P.jointArchetype][P.cidJointConstraint];

    P.maxCandidatesPerWorld = (i32)envU64("MADRONA_B200_MAX_CANDIDATES_PER_WORLD", 256);
    P.maxContactsPerWorld = (i32)envU64("MADRONA_B200_MAX_CONTACTS_PER_WORLD", 128);
    const size_t W = S.numWorlds;
    if (!devAlloc(ex, (void **)&P.candidates, sizeof(Candidate) * W * P.maxCandidatesPerWorld) ||
        !devAlloc(ex, (void **)&P.candCounts, sizeof(i32) * W) ||
        !devAlloc(ex, (void **)&P.contacts, sizeof(Contact) * W * P.maxCandidatesPerWorld) ||
        !devAlloc(ex, (void **)&P.candHit, sizeof(i32) * W * P.maxCandidatesPerWorld) ||
        !devAlloc(ex, (void **)&P.contactOrder, sizeof(i32) * W * P.maxContactsPerWorld) ||
        !devAlloc(ex, (void **)&P.hullQueue, sizeof(HullQueueEntry) * W * P.maxCandidatesPerWorld) ||
        !devAlloc(ex, (void **)&P.hullQueueCount, sizeof(i32) * 4) ||
        !devAlloc(ex, (void **)&P.contactCounts, sizeof(i32) * W) ||
        !devAlloc(ex, (void **)&P.contactMaxLevel, sizeof(i32) * W)) {
        *err = "physics buffers allocation failed";
        return false;
    }
    cudaMemcpy(ph->dPhys, &P, sizeof(PhysicsState), cudaMemcpyHostToDevice);
    return true;
}

void physicsBeforeGraphCapture(Executor *ex)
{
    PhysicsHost *ph = ex->physics;
    if (!ph || !ph->active) return;
    u32 flag = 0;
    cudaMemcpy(&flag, &ph->dPhys->hasSpherePrims, sizeof(u32), cudaMemcpyDeviceToHost);
    ph->spheres = flag != 0;
}

void physicsHostDestroy(Executor *ex)
{
    delete ex->physics;
    ex->physics = nullptr;
}

static dim3 bodyGrid(Executor *ex)
{
    const PhysicsState &P = ex->physics->hPhys;
    int max_cap = 256;
    for (uint32_t i = 0; i < P.numBodyArchetypes; i++) {
        max_cap = std::max(max_cap, ex->hState->tables[P.bodies[i].archetype].capacity);
    }
    int blocks = std::min((max_cap + 255) / 256, ex->numSMs * MB2_BODY_BLOCKS_PER_SM);
    return dim3((unsigned)std::max(blocks, 1), std::max(P.numBodyArchetypes, 1u));
}

bool physicsEnqueueNodes(Executor *ex, const NodeRecord *recs, uint32_t count, cudaStream_t s,
                         std::string *err)
{
    PhysicsHost *ph = ex->physics;
    if (!ph || !ph->active) {
        *err = "physics task recorded but PhysicsSystem::registerTypes was never called";
        return false;
    }
    EngineState *d = ex->dState;
    const unsigned W = ex->hState->numWorlds;
    const unsigned wgrid = (W + kPhysWarps - 1) / kPhysWarps;
    const unsigned wblock = 32 * kPhysWarps;
    const unsigned worlds_per_block = wblock / kSolverLanes;
    const unsigned sgrid = (W + worlds_per_block - 1) / worlds_per_block;
    const dim3 bgrid = bodyGrid(ex);
    for (uint32_t i = 0; i < count; i++) {
        const NodeRecord &rec = recs[i];
        switch (rec.kind) {
        case NodePhysBroadphaseUpdate:
            // tag 0 (post-integration) never rebuilds in the reference either; a
            // pending rebuild request then simply waits for the next tag-1 node,
            // and the un-refitted leaves are refitted by that rebuild
            physBodyKernel<PhaseUpdateLeaves><<<bgrid, 256, 0, s>>>(d);
            if (rec.userTag == 1) physRebuildKernel<<<(W + 127) / 128, 128, 0, s>>>(d);
            break;
        case NodePhysFindCandidates:
            // joints are iterated per world by the solver: keep their table in
            // world order (the reference sorts Joint here too, xpbd.cpp:1092-1096)
            launchSortArchetype(ex, ph->hPhys.jointArchetype, 1, s);
            physWorldKernel<PhaseFindCandidates><<<wgrid, wblock, 0, s>>>(d);
            break;
        case NodePhysSubstepBegin:
            physBodyKernel<PhaseIntegrate><<<bgrid, 256, 0, s>>>(d);
            break;
        case NodePhysNarrowphase:
            {
                const unsigned sgrid_n = (W + kNarrowWorldsPerBlock - 1) / kNarrowWorldsPerBlock;
                if (ph->spheres) physNarrowSimpleKernel<true><<<sgrid_n, kNarrowSimpleThreads, 0, s>>>(d);
                else physNarrowSimpleKernel<false><<<sgrid_n, kNarrowSimpleThreads, 0, s>>>(d);
                physNarrowHullKernel<<<(unsigned)ex->numSMs * (unsigned)MB2_NH_MINB, kNarrowHullThreads, 0, s>>>(d);
            }
            break;
        case NodePhysSolvePositions:
            physWorldKernel<PhaseSolvePositions><<<sgrid, wblock, 0, s>>>(d);
            break;
        case NodePhysTGSVelocities:
            physBodyKernel<PhaseTGSVelocities><<<bgrid, 256, 0, s>>>(d);
            break;
        case NodePhysTGSPositions:
            physBodyKernel<PhaseTGSPositions><<<bgrid, 256, 0, s>>>(d);
            break;
        case NodePhysSetVelocities:
            physBodyKernel<PhaseSetVelocities><<<bgrid, 256, 0, s>>>(d);
            break;
        case NodePhysSolveVelocities:
            physWorldKernel<PhaseSolveVelocities><<<sgrid, wblock, 0, s>>>(d);
            break;
        default:
            *err = "unknown physics node kind " + std::to_string(rec.kind);
            return false;
        }
    }
    return true;
}

bool physicsEnqueueNode(Executor *ex, const NodeRecord &rec, cudaStream_t s, std::string *err)
{
    return physicsEnqueueNodes(ex, &rec, 1, s, err);
}

uint64_t physicsNodeBytes(Executor *ex, const NodeRecord &rec, const char **name, int64_t *rows)
{
    // SURVEY.md 8(d) algorithmic bytes per unit
    PhysicsHost *ph = ex->physics;
    *rows = 0;
    *name = "physics";
    if (!ph || !ph->active) return 0;
    const PhysicsState &P = ph->hPhys;
    const unsigned W = ex->hState->numWorlds;

    int64_t bodies = 0;
    std::vector<TableDesc> tables(ex->hState->numArchetypes);
    cudaMemcpy(tables.data(), ex->dState->tables, sizeof(TableDesc) * tables.size(), cudaMemcpyDeviceToHost);
    for (uint32_t i = 0; i < P.numBodyArchetypes; i++) bodies += tables[P.bodies[i].archetype].numRows;
    std::vector<i32> counts(W);
    auto total = [&](const i32 *dptr) {
        cudaMemcpy(counts.data(), dptr, sizeof(i32) * W, cudaMemcpyDeviceToHost);
        int64_t t = 0;
        for (i32 c : counts) t += c;
        return t;
    };
    switch (rec.kind) {
    case NodePhysBroadphaseUpdate: *name = "phys_broadphase_update"; *rows = bodies; return 136ull * bodies;
    case NodePhysFindCandidates: *name = "phys_find_candidates"; *rows = total(P.candCounts);
        return 24ull * (*rows) + 40ull * bodies;
    case NodePhysSubstepBegin: *name = "phys_substep"; *rows = bodies; return 192ull * bodies;
    case NodePhysNarrowphase: {
        *name = "phys_narrowphase";
        int64_t q = total(P.candCounts), k = total(P.contactCounts);
        *rows = q;
        return 24ull * q + 88ull * q + 96ull * k;
    }
    case NodePhysSolvePositions: *name = "phys_solve_positions"; *rows = total(P.contactCounts);
        return 368ull * (*rows);
    case NodePhysTGSVelocities: *name = "phys_tgs_velocities"; *rows = bodies; return 104ull * bodies;
    case NodePhysTGSPositions: *name = "phys_tgs_positions"; *rows = bodies; return 80ull * bodies;
    case NodePhysSetVelocities: *name = "phys_set_velocities"; *rows = bodies; return 80ull * bodies;
    case NodePhysSolveVelocities: *name = "phys_solve_velocities"; *rows = total(P.contactCounts);
        return 360ull * (*rows);
    default: return 0;
    }
}

}
