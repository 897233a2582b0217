// broadphase::BVH -- the per-world singleton simulator code reaches through
// ctx.singleton<broadphase::BVH>() (reference: include/madrona/broadphase.hpp
// :18-115, broadphase.inl, src/physics/broadphase.cpp:663-888 for traceRay).
// Storage is an mb2::WorldBVH (physics_state.h) so the ahead-of-time physics
// kernels (leaf update, rebuild, refit, candidate search) share it.  Tree
// shape, child order and traversal order follow the reference exactly: the
// order in which overlaps are reported decides contact order and therefore the
// Gauss-Seidel solver's floats.
#pragma once

#include <madrona/math.hpp>
#include <madrona/context.hpp>
#include <madrona/components.hpp>
#include <madrona/geo.hpp>
#include <physics_state.h>

namespace madrona::phys::broadphase {

struct LeafID {
    int32_t id;
};

class BVH {
public:
    inline LeafID reserveLeaf(Entity e, base::ObjectID obj_id)
    {
        int32_t leaf_idx = atomicAdd(&s_.numLeaves, 1);
        if (leaf_idx >= s_.numAllocatedLeaves) {
            mwGPU::raiseError(mb2::ErrPhysicsOverflow);
            return LeafID { 0 };
        }
        s_.leafEntities[leaf_idx] =
            ((unsigned long long)(uint32_t)e.id << 32) | (unsigned long long)e.gen;
        s_.leafObjIDs[leaf_idx] = obj_id.idx;
        return LeafID { leaf_idx };
    }

    inline math::AABB getLeafAABB(LeafID leaf_id) const
    {
        return s_.leafAABBs[leaf_id.id];
    }

    template <typename Fn>
    inline void findIntersecting(const math::AABB &aabb, Fn &&fn) const
    {
        int32_t stack[32];
        stack[0] = 0;
        CountT stack_size = 1;
        while (stack_size > 0) {
            const mb2::BVHNode &node = s_.nodes[stack[--stack_size]];
            for (int i = 0; i < 4; i++) {
                int32_t child = node.children[i];
                if (child == -1) continue;
                math::AABB box { { node.minX[i], node.minY[i], node.minZ[i] },
                                 { node.maxX[i], node.maxY[i], node.maxZ[i] } };
                if (!aabb.overlaps(box)) continue;
                if (child & 0x80000000) {
                    fn(unpackEntity(s_.leafEntities[child & 0x7fffffff]));
                } else {
                    stack[stack_size++] = child;
                }
            }
        }
    }

    template <typename Fn>
    inline void findLeafIntersecting(LeafID leaf_id, Fn &&fn) const
    {
        findIntersecting(getLeafAABB(leaf_id), (Fn &&)fn);
    }

    inline Entity traceRay(math::Vector3 o, math::Vector3 d, float *out_hit_t,
                           math::Vector3 *out_hit_normal,
                           float t_max = float(INFINITY));

    inline void rebuildOnUpdate() { s_.forceRebuild = 1; }
    inline void clearLeaves() { s_.numLeaves = 0; }

    inline mb2::WorldBVH &storage() { return s_; }

private:
    static inline Entity unpackEntity(unsigned long long v)
    {
        return Entity { (uint32_t)(v & 0xFFFFFFFFull), (int32_t)(uint32_t)(v >> 32) };
    }

    inline bool traceRayIntoLeaf(int32_t leaf_idx, math::Vector3 world_ray_o,
                                 math::Vector3 world_ray_d, float t_min, float t_max,
                                 float *hit_t, math::Vector3 *hit_normal);

    mb2::WorldBVH s_;
};

}
