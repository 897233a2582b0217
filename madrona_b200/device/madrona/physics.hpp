// Rigid-body physics API for simulator code (reference:
// include/madrona/physics.hpp:12-222, src/physics/physics.cpp:75-390,
// src/physics/xpbd.cpp:1054-1144).
//
// Same component types, bundle composition (hence the fixed RigidBody column
// order RGDCols relies on, src/physics/physics_impl.hpp:43-58), object
// description structs and PhysicsSystem entry points as the reference.  What
// differs is WHERE the systems run: the reference compiles broadphase /
// narrowphase / XPBD as generic per-row ECS systems next to the simulator;
// here setupBroadphaseTasks / setupPhysicsStepTasks only record engine-owned
// nodes, executed by the ahead-of-time sm_100a kernels in
// csrc/kernels_physics.cu (candidates and contacts live in flat per-world
// buffers, produced in deterministic order, so no Contact / Joint sorts).
// The data-only layouts those kernels and the host asset builder read as well
// (Velocity, JointConstraint, CollisionPrimitive, ObjectManager,
// PhysicsSystemState, the xpbd per-body state ...) live in csrc/physics_state.h.
#pragma once

#include <madrona/math.hpp>
#include <madrona/components.hpp>
#include <madrona/span.hpp>
#include <madrona/taskgraph_builder.hpp>
#include <madrona/context.hpp>

#include <madrona/broadphase.hpp>
#include <madrona/geo.hpp>
#include <physics_state.h>

namespace madrona::phys {

struct ExternalForce : math::Vector3 {
    inline ExternalForce(math::Vector3 v) : Vector3(v) {}
};

struct ExternalTorque : math::Vector3 {
    inline ExternalTorque(math::Vector3 v) : Vector3(v) {}
};

struct SolverBundleAlias {};

struct RigidBody : Bundle<
    base::ObjectInstance,
    ResponseType,
    broadphase::LeafID,
    Velocity,
    ExternalForce,
    ExternalTorque,
    SolverBundleAlias
> {};

struct CandidateCollision {
    Loc a;
    Loc b;
    uint32_t aPrim;
    uint32_t bPrim;
};

struct ContactConstraint {
    Loc ref;
    Loc alt;
    math::Vector4 points[4];
    int32_t numPoints;
    math::Vector3 normal;
};

struct CollisionEvent {
    Entity a;
    Entity b;
};

struct CollisionEventTemporary : Archetype<CollisionEvent> {};

struct ObjectData {
    ObjectManager *mgr;
};

namespace xpbd {

struct XPBDRigidBodyState : Bundle<
    SubstepPrevState,
    PreSolvePositional,
    PreSolveVelocity
> {};

struct Joint : Archetype<JointConstraint> {};

}

namespace tgs {
// == tgs.cpp:15-18
struct TGSRigidBodyState : Bundle<
> {};
}

namespace xpbd {

// The reference keeps its contact / joint queries in this singleton
// (xpbd.cpp:20-23).  The engine does not need it, but registering it keeps the
// number and order of singleton archetypes -- and therefore every entity ID
// handed out afterwards -- identical to the CPU backend's.
struct SolverState {
    uint32_t reserved[4];
};

}

namespace PhysicsSystem {

enum class Solver : uint32_t {
    XPBD,
    TGS,
};

inline void registerTypes(ECSRegistry &registry, Solver solver = Solver::XPBD)
{
    registry.registerComponent<ResponseType>();
    registry.registerComponent<broadphase::LeafID>();
    registry.registerComponent<Velocity>();
    registry.registerComponent<ExternalForce>();
    registry.registerComponent<ExternalTorque>();

    registry.registerSingleton<broadphase::BVH>();

    registry.registerComponent<CollisionEvent>();
    registry.registerArchetype<CollisionEventTemporary>();

    registry.registerComponent<CandidateCollision>();
    registry.registerComponent<JointConstraint>();
    registry.registerComponent<ContactConstraint>();

    registry.registerSingleton<PhysicsSystemState>();
    registry.registerSingleton<ObjectData>();

    // solver state: xpbd::registerTypes (xpbd.cpp:1055-1069) / tgs::registerTypes
    // (tgs.cpp:28-43).  TGS keeps no per-body state: its bundle is empty.
    registry.registerComponent<xpbd::SubstepPrevState>();
    registry.registerComponent<xpbd::PreSolvePositional>();
    registry.registerComponent<xpbd::PreSolveVelocity>();
    registry.registerArchetype<xpbd::Joint>();
    registry.registerSingleton<xpbd::SolverState>();
    if (solver == Solver::TGS) {
        registry.registerBundle<tgs::TGSRigidBodyState>();
        registry.registerBundleAlias<SolverBundleAlias, tgs::TGSRigidBodyState>();
    } else {
        registry.registerBundle<xpbd::XPBDRigidBodyState>();
        registry.registerBundleAlias<SolverBundleAlias, xpbd::XPBDRigidBodyState>();
    }

    registry.registerBundle<RigidBody>();

    // tell the engine which components / archetypes are the physics ones
    mb2::PhysicsState &P = *mwGPU::engine().physics;
    P.solver = (uint32_t)solver;
    P.componentIDs[mb2::PCPosition] = TypeTracker::typeID<base::Position>();
    P.componentIDs[mb2::PCRotation] = TypeTracker::typeID<base::Rotation>();
    P.componentIDs[mb2::PCScale] = TypeTracker::typeID<base::Scale>();
    P.componentIDs[mb2::PCObjectID] = TypeTracker::typeID<base::ObjectID>();
    P.componentIDs[mb2::PCResponseType] = TypeTracker::typeID<ResponseType>();
    P.componentIDs[mb2::PCLeafID] = TypeTracker::typeID<broadphase::LeafID>();
    P.componentIDs[mb2::PCVelocity] = TypeTracker::typeID<Velocity>();
    P.componentIDs[mb2::PCExtForce] = TypeTracker::typeID<ExternalForce>();
    P.componentIDs[mb2::PCExtTorque] = TypeTracker::typeID<ExternalTorque>();
    P.componentIDs[mb2::PCPrevState] = TypeTracker::typeID<xpbd::SubstepPrevState>();
    P.componentIDs[mb2::PCPreSolvePos] = TypeTracker::typeID<xpbd::PreSolvePositional>();
    P.componentIDs[mb2::PCPreSolveVel] = TypeTracker::typeID<xpbd::PreSolveVelocity>();
    P.cidJointConstraint = TypeTracker::typeID<JointConstraint>();
    P.bvhArchetype = TypeTracker::typeID<SingletonArchetype<broadphase::BVH>>();
    P.paramsArchetype = TypeTracker::typeID<SingletonArchetype<PhysicsSystemState>>();
    P.objectDataArchetype = TypeTracker::typeID<SingletonArchetype<ObjectData>>();
    P.jointArchetype = TypeTracker::typeID<xpbd::Joint>();
    P.registered = 1;
}

// Per-world setup, called from the simulator's world constructor
// (reference: src/physics/physics.cpp:98-141, broadphase.cpp:13-46).
inline void init(Context &ctx,
                 ObjectManager *obj_mgr,
                 float delta_t,
                 CountT num_substeps,
                 math::Vector3 gravity,
                 CountT max_dynamic_objects,
                 Solver = Solver::XPBD)
{
    mb2::EngineState &S = mwGPU::engine();
    mb2::WorldBVH &bvh = ctx.singleton<broadphase::BVH>().storage();

    const CountT max_leaves = max_dynamic_objects;
    // node budget as broadphase.cpp:38-45
    CountT third = (max_leaves - 1 + 2) / 3;
    const CountT num_nodes = (third > 1 ? third : 1) + max_leaves;

    auto carve = [&S](uint64_t bytes) -> char * {
        bytes = (bytes + 127ull) & ~127ull;
        unsigned long long off = atomicAdd((unsigned long long *)&S.persistOffset,
                                           (unsigned long long)bytes);
        if (off + bytes > S.persistCapacity) {
            mwGPU::raiseError(mb2::ErrPersistOverflow);
            return S.persistArena;
        }
        return S.persistArena + off;
    };

    bvh.nodes = (mb2::BVHNode *)carve(sizeof(mb2::BVHNode) * num_nodes);
    bvh.leafEntities = (mb2::u64 *)carve(8 * max_leaves);
    bvh.objMgr = obj_mgr;
    bvh.leafObjIDs = (int32_t *)carve(4 * max_leaves);
    bvh.leafAABBs = (math::AABB *)carve(sizeof(math::AABB) * max_leaves);
    bvh.leafTransforms = (mb2::LeafTransform *)carve(sizeof(mb2::LeafTransform) * max_leaves);
    bvh.leafParents = (uint32_t *)carve(4 * max_leaves);
    bvh.sortedLeaves = (int32_t *)carve(4 * max_leaves);
    bvh.traversalOrder = (int32_t *)carve(4 * max_leaves);
    bvh.orderedBoxes = (mb2::PVec4 *)carve(sizeof(mb2::PVec4) * 2 * max_leaves);
    bvh.leafOrderPos = (int32_t *)carve(4 * max_leaves);
    bvh.numTraversal = 0;
    bvh.numNodes = 0;
    bvh.numAllocatedNodes = (int32_t)num_nodes;
    bvh.numLeaves = 0;
    bvh.numAllocatedLeaves = (int32_t)max_leaves;
    // expansion: 2 * dt of velocity, 100 * dt^2 of acceleration (physics.cpp:106-111)
    bvh.velExpansion = 2.f * delta_t;
    bvh.accelExpansion = 100.f * delta_t * delta_t;
    bvh.forceRebuild = 1;

    float h = delta_t / (float)num_substeps;
    float g_mag = gravity.length();
    ctx.singleton<PhysicsSystemState>() = PhysicsSystemState {
        delta_t, h, gravity, g_mag, 2.f * g_mag * h,
        0xFFFFFFFFu, TypeTracker::typeID<xpbd::Joint>(),
    };
    ctx.singleton<ObjectData>() = ObjectData { obj_mgr };
}

inline void reset(Context &ctx)
{
    broadphase::BVH &bvh = ctx.singleton<broadphase::BVH>();
    bvh.rebuildOnUpdate();
    bvh.clearLeaves();
}

inline broadphase::LeafID registerEntity(Context &ctx, Entity e, base::ObjectID obj_id)
{
    broadphase::BVH &bvh = ctx.singleton<broadphase::BVH>();
    // tell the executor when spheres are in play (it then launches the narrowphase
    // variant that carries the sphere - hull path)
    {
        const ObjectManager *obj_mgr = bvh.storage().objMgr;
        const uint32_t first = obj_mgr->rigidBodyPrimitiveOffsets[obj_id.idx];
        const uint32_t count = obj_mgr->rigidBodyPrimitiveCounts[obj_id.idx];
        for (uint32_t i = 0; i < count; i++) {
            if (obj_mgr->collisionPrimitives[first + i].type == CollisionPrimitive::Type::Sphere) {
                mb2::PhysicsState *P = mwGPU::engine().physics;
                if (!P->hasSpherePrims) atomicOr(&P->hasSpherePrims, 1u);
            }
        }
    }
    return bvh.reserveLeaf(e, obj_id);
}

inline Entity makeFixedJoint(Context &ctx, Entity e1, Entity e2,
                             math::Quat attach_rot1, math::Quat attach_rot2,
                             math::Vector3 r1, math::Vector3 r2, float separation)
{
    Entity e = ctx.makeEntity<xpbd::Joint>();
    JointConstraint &j = ctx.get<JointConstraint>(e);
    j.e1 = e1;
    j.e2 = e2;
    j.type = JointConstraint::Type::Fixed;
    j.fixed.attachRot1 = attach_rot1;
    j.fixed.attachRot2 = attach_rot2;
    j.fixed.separation = separation;
    j.r1 = r1;
    j.r2 = r2;
    return e;
}

inline Entity makeHingeJoint(Context &ctx, Entity e1, Entity e2,
                             math::Vector3 a1_local, math::Vector3 a2_local,
                             math::Vector3 b1_local, math::Vector3 b2_local,
                             math::Vector3 r1, math::Vector3 r2)
{
    Entity e = ctx.makeEntity<xpbd::Joint>();
    JointConstraint &j = ctx.get<JointConstraint>(e);
    j.e1 = e1;
    j.e2 = e2;
    j.type = JointConstraint::Type::Hinge;
    j.hinge.a1Local = a1_local;
    j.hinge.a2Local = a2_local;
    j.hinge.b1Local = b1_local;
    j.hinge.b2Local = b2_local;
    j.r1 = r1;
    j.r2 = r2;
    return e;
}

// Leaf update -> (rebuild if requested) -> refit
// (reference: broadphase.cpp:995-1017 setupBVHTasks).
inline TaskGraphNodeID setupBroadphaseTasks(TaskGraphBuilder &builder,
                                            Span<const TaskGraphNodeID> deps)
{
    return mwGPU::pushBuiltin(builder, deps, mb2::NodePhysBroadphaseUpdate, 0, 0, 1);
}

// Candidate search, num_substeps x (integrate, narrowphase, position solve,
// velocity update, velocity solve), post-integration leaf update + refit
// (reference: physics.cpp:351-384, xpbd.cpp:1085-1144).
inline TaskGraphNodeID setupPhysicsStepTasks(TaskGraphBuilder &builder,
                                             Span<const TaskGraphNodeID> deps,
                                             CountT num_substeps,
                                             Solver solver = Solver::XPBD)
{
    TaskGraphNodeID cur = mwGPU::pushBuiltin(builder, deps, mb2::NodePhysFindCandidates);
    if (solver == Solver::TGS) {
        // tgs::setupTGSSolverTasks (src/physics/tgs.cpp:213-302): the narrowphase runs once,
        // then every substep integrates velocities and positions; the reference's contact /
        // joint prepare, warm-start and solve systems are empty bodies there (:59-90,
        // 144-205), so the solver is a collision-free integrator -- reproduced as it is.
        cur = mwGPU::pushBuiltin(builder, { cur }, mb2::NodePhysNarrowphase);
        for (CountT i = 0; i < num_substeps; i++) {
            cur = mwGPU::pushBuiltin(builder, { cur }, mb2::NodePhysTGSVelocities);
            cur = mwGPU::pushBuiltin(builder, { cur }, mb2::NodePhysTGSPositions);
        }
        return mwGPU::pushBuiltin(builder, { cur }, mb2::NodePhysBroadphaseUpdate, 0, 0, 0);
    }
    for (CountT i = 0; i < num_substeps; i++) {
        cur = mwGPU::pushBuiltin(builder, { cur }, mb2::NodePhysSubstepBegin);
        cur = mwGPU::pushBuiltin(builder, { cur }, mb2::NodePhysNarrowphase);
        cur = mwGPU::pushBuiltin(builder, { cur }, mb2::NodePhysSolvePositions);
        cur = mwGPU::pushBuiltin(builder, { cur }, mb2::NodePhysSetVelocities);
        cur = mwGPU::pushBuiltin(builder, { cur }, mb2::NodePhysSolveVelocities);
    }
    // post-integration: leaf update + refit, no rebuild (broadphase.cpp:1029-1052)
    return mwGPU::pushBuiltin(builder, { cur }, mb2::NodePhysBroadphaseUpdate, 0, 0, 0);
}

inline TaskGraphNodeID setupCleanupTasks(TaskGraphBuilder &builder,
                                         Span<const TaskGraphNodeID> deps)
{
    return builder.addToGraph<ClearTmpNode<CollisionEventTemporary>>(deps);
}

}

// ---- ray casts against the broadphase tree (used by lidar-style systems) ----

namespace broadphase {

namespace detail {

inline bool rayIntoPlane(math::Vector3 ray_o, math::Vector3 ray_d, float t_min,
                         float t_max, float *hit_t, math::Vector3 *hit_normal)
{
    // object space: the plane is z = 0 with normal +z
    float denom = ray_d.z;
    if (denom == 0) return false;
    float t = -ray_o.z / denom;
    if (t < t_min || t > t_max) return false;
    *hit_t = t;
    *hit_normal = math::Vector3 { 0, 0, 1 };
    return true;
}

// Ray vs convex polyhedron as an intersection of half-spaces (RTCD 5.3.8);
// face normals point outwards.  A ray that only crosses back faces is a miss.
inline bool rayIntoHull(const geo::HalfEdgeMesh &mesh, math::Vector3 ray_o,
                        math::Vector3 ray_d, float t_min, float t_max,
                        float *hit_t, math::Vector3 *hit_normal)
{
    float t_enter = t_min;
    float t_exit = t_max;
    math::Vector3 enter_normal = math::Vector3::zero();
    const CountT num_faces = (CountT)mesh.numFaces;
    for (CountT f = 0; f < num_faces; f++) {
        geo::Plane plane = mesh.facePlanes[f];
        float denom = dot(plane.normal, ray_d);
        float neg_dist = plane.d - dot(plane.normal, ray_o);
        if (denom == 0.0f) {
            if (neg_dist < 0.0f) return false;
        } else {
            float t = neg_dist / denom;
            if (denom < 0.0f) {
                if (t >= t_enter) {
                    t_enter = t;
                    enter_normal = plane.normal;
                }
            } else if (t <= t_exit) {
                t_exit = t;
            }
            if (t_enter > t_exit) return false;
        }
    }
    if (enter_normal.x == 0 && enter_normal.y == 0 && enter_normal.z == 0) return false;
    *hit_t = t_enter;
    *hit_normal = enter_normal;
    return true;
}

}

bool BVH::traceRayIntoLeaf(int32_t leaf_idx, math::Vector3 world_ray_o,
                           math::Vector3 world_ray_d, float t_min, float t_max,
                           float *hit_t, math::Vector3 *hit_normal)
{
    const ObjectManager *obj_mgr = s_.objMgr;
    const int32_t obj = s_.leafObjIDs[leaf_idx];
    const mb2::LeafTransform txfm = s_.leafTransforms[leaf_idx];
    const math::Quat rot = txfm.rot;
    const math::Vector3 pos = txfm.pos;
    const math::Quat to_local = rot.inv();

    math::Vector3 obj_o = to_local.rotateVec(world_ray_o - pos);
    obj_o.x /= txfm.scale.x;
    obj_o.y /= txfm.scale.y;
    obj_o.z /= txfm.scale.z;
    math::Vector3 obj_d = rot.inv().rotateVec(world_ray_d);
    obj_d.x /= txfm.scale.x;
    obj_d.y /= txfm.scale.y;
    obj_d.z /= txfm.scale.z;
    math::Diag3x3 inv_d = math::Diag3x3::fromVec(1.f / obj_d);

    const CountT prim_offset = (CountT)obj_mgr->rigidBodyPrimitiveOffsets[obj];
    const CountT num_prims = (CountT)obj_mgr->rigidBodyPrimitiveCounts[obj];

    math::Vector3 obj_normal;
    bool hit_leaf = false;
    for (CountT i = 0; i < num_prims; i++) {
        const CountT prim_idx = prim_offset + i;
        math::AABB prim_aabb = obj_mgr->primitiveAABBs[prim_idx];
        if (!prim_aabb.rayIntersects(obj_o, inv_d, 0.f, t_max)) continue;

        const CollisionPrimitive *prim = &obj_mgr->collisionPrimitives[prim_idx];
        bool hit = false;
        if (prim->type == CollisionPrimitive::Type::Hull) {
            hit = detail::rayIntoHull(prim->hull.halfEdgeMesh, obj_o, obj_d,
                                      t_min, t_max, hit_t, &obj_normal);
        } else if (prim->type == CollisionPrimitive::Type::Plane) {
            hit = detail::rayIntoPlane(obj_o, obj_d, t_min, t_max, hit_t, &obj_normal);
        }
        if (hit) {
            hit_leaf = true;
            t_max = *hit_t;
        }
    }
    if (!hit_leaf) return false;
    *hit_normal = rot.rotateVec(obj_normal);
    return true;
}

Entity BVH::traceRay(math::Vector3 o, math::Vector3 d, float *out_hit_t,
                     math::Vector3 *out_hit_normal, float t_max)
{
    math::Diag3x3 inv_d = math::Diag3x3::fromVec(d).inv();

    // The reference walks the 4-wide tree with a stack (src/physics/
    // broadphase.cpp:658-724), testing child i of a popped node against the
    // t_max current at that moment:
    //   max(mins.x, mins.y, mins.z, 0) <= min(maxes.x, maxes.y, maxes.z, t_max)
    // (math.inl:1670-1696, NaN-skipping fminf / fmaxf).  A leaf is entered iff
    // its own slot box passes that test when its turn comes: every ancestor box
    // contains it (the slab expressions are monotonic in the box bounds and
    // t_max only shrinks), and leaves are met in the tree's fixed report order.
    // So the walk is a linear scan over WorldBVH::orderedBoxes -- same leaves,
    // same order, same floats, no stack and no node pointer chasing.
    //
    //
    // Mechanism (results identical by construction): boxes are handled in chunks of 64.
    //   1. uniform pass: every lane slab-tests the chunk's boxes against its CURRENT t_max and
    //      keeps the passing ones as a 64-bit mask -- all lanes run the same loop, no divergence.
    //      t_max only shrinks afterwards and a smaller t_max can only turn a pass into a fail
    //      (exit = min(..., t_max)), so the mask is a superset of the leaves the walk enters;
    //   2. ordered pass over the mask bits: the slab test is REPEATED with the t_max of that
    //      moment -- the reference's exact decision, same expression, same floats -- and the
    //      leaves that pass are entered in order.  Each round every lane first moves on to its
    //      next entered leaf, then the lanes that called together run the (expensive) leaf
    //      test together; the warp votes keep the compiler from folding the two phases back
    //      into one divergent loop.
    // (The one-phase scan over all boxes spent most of its instructions in the divergent
    // "walk to my next entered leaf" loop: ncu round 1, 9 of 32 lanes active.  Tried and
    // rejected on B200, room 8192 worlds: seeding t_max with the hit of the nearest-entry leaf
    // before the walk -- 1.091 vs 1.019 ms/step, the extra pass costs more than the leaf tests
    // it saves.)
    const unsigned peers = __activemask();
    const mb2::PVec4 *boxes = s_.orderedBoxes;
    const int32_t num_boxes = s_.numTraversal;
    Entity closest = Entity::none();
    math::Vector3 closest_normal { 0, 0, 0 };

    auto entered = [&](int32_t j, int32_t *leaf) {
        const mb2::PVec4 b0 = boxes[2 * j], b1 = boxes[2 * j + 1];
        const float lx = inv_d.d0 * (b0.x - o.x), ux = inv_d.d0 * (b0.w - o.x);
        const float ly = inv_d.d1 * (b0.y - o.y), uy = inv_d.d1 * (b1.x - o.y);
        const float lz = inv_d.d2 * (b0.z - o.z), uz = inv_d.d2 * (b1.y - o.z);
        const float entry = fmaxf(fminf(lx, ux), fmaxf(fminf(ly, uy), fmaxf(fminf(lz, uz), 0.f)));
        const float exit = fminf(fmaxf(lx, ux), fminf(fmaxf(ly, uy), fminf(fmaxf(lz, uz), t_max)));
        *leaf = __float_as_int(b1.z);
        return entry <= exit;
    };

    // (every peer runs the same number of chunk iterations: lanes of one warp may belong to
    // worlds with different leaf counts)
    for (int32_t base = 0; __any_sync(peers, base < num_boxes); base += 64) {
        const int32_t left = num_boxes - base;
        const int32_t chunk = left < 0 ? 0 : (left < 64 ? left : 64);
        unsigned long long cand = 0;
        for (int32_t j = 0; j < chunk; j++) {
            int32_t leaf;
            if (entered(base + j, &leaf)) cand |= 1ull << j;
        }
        while (__any_sync(peers, cand != 0)) {
            int32_t leaf_idx = -1;
            while (cand != 0) {
                const int32_t j = __ffsll((long long)cand) - 1;
                cand &= cand - 1;
                int32_t leaf;
                if (entered(base + j, &leaf)) {
                    leaf_idx = leaf;
                    break;
                }
            }
            __syncwarp(peers);

            if (leaf_idx >= 0) {
                float hit_t;
                math::Vector3 leaf_normal;
                if (traceRayIntoLeaf(leaf_idx, o, d, 0.f, t_max, &hit_t, &leaf_normal)) {
                    t_max = hit_t;
                    closest = unpackEntity(s_.leafEntities[leaf_idx]);
                    closest_normal = leaf_normal;
                }
            }
        }
    }
    if (closest == Entity::none()) return Entity::none();
    *out_hit_t = t_max;
    *out_hit_normal = closest_normal;
    return closest;
}

}

}
