// physics_state.h -- layouts shared by the NVRTC-side physics API
// (device/madrona/physics.hpp: what simulator code calls), the ahead-of-time
// physics kernels (kernels_physics.cu) and the host asset builder
// (physics_assets.cpp).  Plain structs; every header included here compiles
// under g++, nvcc and NVRTC.
//
// The public component structs (Velocity, CollisionPrimitive, ObjectManager,
// RigidBodyMetadata, HalfEdgeMesh ...) keep the reference's field order and
// sizes (include/madrona/physics.hpp:12-153, geo.hpp:7-45) so a simulator's
// ObjectManager blob is interchangeable between the reference CPU backend and
// this engine.  Engine-internal state (candidate / contact buffers, per-world
// BVH storage) is laid out for the GPU instead of being ECS archetypes.
#pragma once

#include <cstddef>
#include <madrona/math.hpp>
#include <madrona/geo.hpp>
#include <madrona/ecs.hpp>

#include "mb2_state.h"

namespace madrona::phys {

enum class ResponseType : uint32_t {
    Dynamic,
    Kinematic,
    Static,
};

struct Velocity {
    math::Vector3 linear;
    math::Vector3 angular;
};

struct JointConstraint {
    enum class Type {
        Fixed,
        Hinge
    };

    struct Fixed {
        math::Quat attachRot1;
        math::Quat attachRot2;
        float separation;
    };

    struct Hinge {
        math::Vector3 a1Local;
        math::Vector3 a2Local;
        math::Vector3 b1Local;
        math::Vector3 b2Local;
    };

    Entity e1;
    Entity e2;
    Type type;

    union {
        Fixed fixed;
        Hinge hinge;
    };

    math::Vector3 r1;
    math::Vector3 r2;
};

struct RigidBodyMassData {
    float invMass;
    math::Vector3 invInertiaTensor;
    math::Vector3 toCenterOfMass;
    math::Quat toInteriaFrame;
};

struct RigidBodyFrictionData {
    float muS;
    float muD;
};

struct RigidBodyMetadata {
    RigidBodyMassData mass;
    RigidBodyFrictionData friction;
};

struct CollisionPrimitive {
    enum class Type : uint32_t {
        Sphere = 1 << 0,
        Hull = 1 << 1,
        Plane = 1 << 2,
    };

    struct Sphere {
        float radius;
    };

    struct Hull {
        geo::HalfEdgeMesh halfEdgeMesh;
    };

    struct Plane {};

    Type type;
    union {
        Sphere sphere;
        Plane plane;
        Hull hull;
    };
};

struct ObjectManager {
    CollisionPrimitive *collisionPrimitives;
    math::AABB *primitiveAABBs;

    math::AABB *rigidBodyAABBs;
    uint32_t *rigidBodyPrimitiveOffsets;
    uint32_t *rigidBodyPrimitiveCounts;
    RigidBodyMetadata *metadata;
};

// == src/physics/physics_impl.hpp:7-15 (a singleton component, per world)
struct PhysicsSystemState {
    float deltaT;
    float h;
    math::Vector3 g;
    float gMagnitude;
    float restitutionThreshold;
    uint32_t contactArchetypeID;
    uint32_t jointArchetypeID;
};

namespace xpbd {

// == src/physics/xpbd.cpp:26-46
struct SubstepPrevState {
    math::Vector3 prevPosition;
    math::Quat prevRotation;
};

struct PreSolvePositional {
    math::Vector3 x;
    math::Quat q;
};

struct PreSolveVelocity {
    math::Vector3 v;
    math::Vector3 omega;
};

}

// The kernels read these through ECS columns and the uploaded ObjectManager blob,
// and RigidBodyAssets.host_arrays (executor.py) decodes the blob by offset.
static_assert(sizeof(Velocity) == 24, "Velocity layout");
static_assert(sizeof(JointConstraint) == 92, "JointConstraint layout");
static_assert(sizeof(RigidBodyMetadata) == 52, "RigidBodyMetadata layout");
static_assert(sizeof(CollisionPrimitive) == 56, "CollisionPrimitive layout");
static_assert(sizeof(ObjectManager) == 48, "ObjectManager layout");
static_assert(sizeof(PhysicsSystemState) == 36, "PhysicsSystemState layout");
static_assert(sizeof(geo::HalfEdge) == 12 && sizeof(geo::Plane) == 16 && sizeof(math::AABB) == 24,
              "object description element layouts");
#ifndef __CUDACC_RTC__    // NVRTC has no constant offsetof
static_assert(offsetof(CollisionPrimitive, sphere) == 8 && offsetof(CollisionPrimitive, hull) == 8,
              "CollisionPrimitive layout");
static_assert(offsetof(geo::HalfEdgeMesh, halfEdges) == 0 && offsetof(geo::HalfEdgeMesh, faceBaseHalfEdges) == 8 &&
              offsetof(geo::HalfEdgeMesh, facePlanes) == 16 && offsetof(geo::HalfEdgeMesh, vertices) == 24 &&
              offsetof(geo::HalfEdgeMesh, numHalfEdges) == 32 && offsetof(geo::HalfEdgeMesh, numFaces) == 36 &&
              offsetof(geo::HalfEdgeMesh, numVertices) == 40, "HalfEdgeMesh layout");
#endif

}

namespace mb2 {

struct alignas(16) PVec4 { float x, y, z, w; };

// == broadphase::BVH::Node (include/madrona/broadphase.hpp:62-78): 4-wide node,
// child boxes in SoA, leaf children tagged with bit 31, sentinel = -1.
struct BVHNode {
    float minX[4];
    float minY[4];
    float minZ[4];
    float maxX[4];
    float maxY[4];
    float maxZ[4];
    i32 children[4];
    i32 parentID;
};
static_assert(sizeof(BVHNode) == 116, "BVH node layout");

struct LeafTransform {
    madrona::math::Vector3 pos;
    madrona::math::Quat rot;
    madrona::math::Vector3 scale;
};

// One per world: the payload of the broadphase::BVH singleton component.
struct WorldBVH {
    BVHNode *nodes;
    u64 *leafEntities;        // Entity {gen,id} packed as in the table column
    const madrona::phys::ObjectManager *objMgr;
    i32 *leafObjIDs;
    madrona::math::AABB *leafAABBs;
    LeafTransform *leafTransforms;
    u32 *leafParents;         // (node << 2) | child
    i32 *sortedLeaves;
    // Leaves in the order an un-pruned traversal reports them (children 0..3
    // scanned in order, inner children visited LIFO).  Pruning never reorders
    // the survivors, so a query's result list is this list filtered by box
    // overlap -- which lets the candidate search run as a uniform loop.
    i32 *traversalOrder;
    // The same list with the boxes inlined, 32 B per entry: the leaf's slot box in
    // its parent node (grow-only between rebuilds) + the leaf index --
    //   {min.x, min.y, min.z, max.x}, {max.y, max.z, leaf (int bits), 0}
    // kept current by rebuild / refit, read by the candidate search and by
    // BVH::traceRay as a flat, coalesced array (no node pointer chasing).
    PVec4 *orderedBoxes;
    i32 *leafOrderPos;        // leaf -> position in the list
    i32 numNodes;
    i32 numAllocatedNodes;
    i32 numLeaves;
    i32 numAllocatedLeaves;
    float velExpansion;
    float accelExpansion;
    i32 forceRebuild;
    i32 numTraversal;
};

// Role of phys::CandidateCollision (physics.hpp:52-57: two Locs + two primitive
// indices, 24 B), packed to 16 B and extended with what the narrowphase would
// otherwise look up again per contact:
//   archPrim = aArch | bArch << 8 | aPrim << 16 | bPrim << 24
//   slots    = aSlot | aMutable << 15 | ... same for b in the high half, i.e.
//              ((slot << 1) | mutable) per side with slot = index of the body in
//              its world's body list (0x7fff: unknown) and mutable = "writing the
//              body back can change it" (see rotationIsNormalizeFixpoint).
struct Candidate {
    u32 archPrim;
    i32 aRow;
    i32 bRow;
    u32 slots;
};
static_assert(sizeof(Candidate) == 16, "candidate layout");

struct HullQueueEntry {
    i32 world;
    i32 cand;
};

// == phys::ContactConstraint (physics.hpp:59-65) + xpbd::XPBDContactState
struct Contact {
    u32 refArch; i32 refRow;
    u32 altArch; i32 altRow;
    float points[4][4];       // xyz + penetration depth
    i32 numPoints;
    madrona::math::Vector3 normal;
    float lambdaN;            // XPBDContactState::lambdaN[0], the only one ever read (xpbd.cpp:1028)
    u32 refInfo;              // (world body slot << 1) | mutable of ref / alt (Candidate::slots)
    u32 altInfo;
    // Dependency level inside the world's contact list: contacts of one level
    // touch disjoint (mutable) bodies and every earlier contact they could
    // depend on has a lower level, so solving level by level in parallel is
    // bit-identical to the reference's sequential Gauss-Seidel sweep.
    i32 level;
};
static_assert(sizeof(Contact) == 112, "contact layout");

enum PhysCol : int {
    PCPosition = 0, PCRotation, PCScale, PCObjectID, PCResponseType, PCLeafID,
    PCVelocity, PCExtForce, PCExtTorque, PCPrevState, PCPreSolvePos, PCPreSolveVel,
    PCCount
};

constexpr int kMaxBodyArchetypes = 16;
constexpr int kMaxHullVerts = 16;     // narrowphase per-thread staging caps
constexpr int kMaxHullFaces = 16;
constexpr int kMaxFaceVerts = 8;
constexpr int kMaxLevelBodies = 128;  // bodies per world tracked by the contact level scan

struct BodyArchetype {
    u32 archetype;
    i32 cols[PCCount];
};

struct PhysicsState {
    // ---- written by the device-side PhysicsSystem::registerTypes (1 thread)
    u32 registered;
    u32 solver;
    u32 componentIDs[PCCount];
    u32 cidJointConstraint;
    u32 bvhArchetype;            // singleton archetypes
    u32 paramsArchetype;
    u32 objectDataArchetype;
    u32 jointArchetype;
    // set by PhysicsSystem::registerEntity when an object with a sphere primitive
    // joins a world: selects the narrowphase kernel that carries the sphere-hull
    // (GJK) path
    u32 hasSpherePrims;

    // ---- filled by the host after registerTypes
    u32 numBodyArchetypes;
    BodyArchetype bodies[kMaxBodyArchetypes];   // ascending archetype id
    signed char bodyIndex[kMaxArchetypes];      // archetype id -> index into bodies[] or -1
    i32 jointCol;

    Candidate *candidates;       // [numWorlds][maxCandidatesPerWorld]
    i32 *candCounts;             // [numWorlds]
    i32 maxCandidatesPerWorld;
    // A candidate's contact lives in the slot of the same index (so the dense
    // narrowphase kernels need no per-world ordering); candHit marks the slots
    // that hold a contact this substep, contactOrder lists them in candidate
    // order (== the CPU backend's contact order) for the solvers.
    Contact *contacts;           // [numWorlds][maxCandidatesPerWorld]
    i32 *candHit;                // [numWorlds][maxCandidatesPerWorld]
    i32 *contactOrder;           // [numWorlds][maxContactsPerWorld] -> slot
    i32 *contactCounts;
    i32 *contactMaxLevel;        // [numWorlds]
    i32 maxContactsPerWorld;
    // hull - hull candidates that passed the primitive-box test, any order
    HullQueueEntry *hullQueue;   // [numWorlds * maxCandidatesPerWorld]
    i32 *hullQueueCount;
};

}
