// kernels_render.cu -- hot system 3: batch ray-cast renderer (SURVEY.md 8 rows
// a13-a15).
//
// Per step (render-prepare node, inside the step graph; role of the reference's
// instanceTransformUpdate / viewTransformUpdate / lightUpdate / mortonCodeUpdate /
// three archetype sorts / bvhBuildFast / bvhConstructAABBs / bvhWidenTree /
// exportCountsGPU: src/render/ecs_system.cpp:100-348, 486-597 and
// src/mw/device/bvh.cpp:731-1217):
//   renderGatherInstancesKernel  every world's renderable instances -> InstanceData +
//                                world box (mesh root box under TRS)
//   renderLightKernels           carriers refresh their LightDesc, lights gathered per world
//   renderGatherViewsKernel      PerspectiveCameraData per view
//   renderBuildTLASKernel        ONE WARP PER WORLD, all in shared memory: 30-bit Morton
//                                codes of the box centres inside the world's bounds, rank
//                                sort, Karras' parallel LBVH, bottom-up boxes, collapse to
//                                4-wide nodes, quantise -> QBVHNode[] (the reference's
//                                traversal format)
// Render graph: renderRaycastKernel, one thread per pixel, one block per view
// (8 x 4 pixel tiles per warp): TLAS -> instance -> object-space ray -> BLAS
// (reference-format MeshBVH: quantised 4-wide nodes over de-indexed triangles)
// -> watertight ray / triangle test; materials (override colour / material
// table), lights with shadow rays, RGBA8 + f32 depth.
//
// Image formation follows the reference's CUDA ray tracer
// (src/mw/device/bvh_raycast.cpp): ray generation :58-88, object-space ray and
// t rescaling :620-645 / :744-751, watertight ray-triangle test :317-448
// (explicit fmaf kept), colour / normal of a hit :756-815, lighting :848-938,
// depth / RGBA8 output :820-838, 940-1029.  How the structures are built and
// walked is this engine's own (the reference builds the TLAS with ~10 megakernel
// nodes and global atomics and walks it with a packed-group traversal); a
// closest hit does not depend on the tree that found it.
//
// Parity: the reference can only render on its GPU backend (the CPU backend
// forces the ray caster off, src/render/ecs_system.cpp:684-689), so there is no
// reference image to compare with -- "parity unpinned".  tests/test_render_bvh.py
// pins every pixel's (instance, triangle, depth) to a brute-force float64
// closest hit over ALL triangles of the world; tests/test_render.py keeps the
// numpy restatement of the image-formation formulas.
#include "physics_host.hpp"
#include "render_state.h"

#include <madrona/math.hpp>
#include <cfloat>
#include <algorithm>
#include <vector>

namespace mb2 {

using madrona::math::Vector3;
using madrona::math::Quat;
using madrona::math::Diag3x3;
using madrona::math::AABB;
using madrona::math::cross;
using madrona::math::dot;
using madrona::render::LightDesc;
using madrona::render::RenderCamera;

struct RenderHost {
    RenderState *dRender = nullptr;
    RenderState hRender;
    bool active = false;
    size_t tlasSmem = 0;
};

// ---- render-prepare: instances ---------------------------------------------------------
__global__ void __launch_bounds__(128)
renderGatherInstancesKernel(EngineState *Sp)
{
    EngineState &S = *Sp;
    RenderState &R = *S.render;
    const int lane = threadIdx.x & 31;
    const i32 w = (i32)((blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    if (w >= (i32)S.numWorlds) return;

    RenderInstance *out = R.instances + (size_t)w * R.maxInstancesPerWorld;
    i32 running = 0;
    for (u32 ai = 0; ai < R.numRenderArchetypes; ai++) {
        const RenderArchetype &ra = R.renderables[ai];
        const TableDesc &t = S.tables[ra.archetype];
        const i32 first = t.worldOffsets[w];
        const i32 count = t.worldCounts[w];
        for (i32 base = 0; base < count; base += 32) {
            const i32 row = first + base + lane;
            bool valid = base + lane < count && ((const i32 *)t.columns[1])[row] == w;
            if (valid) {
                const u64 marker = ((const u64 *)t.columns[ra.cols[RCRenderable]])[row];
                valid = (i32)(u32)(marker >> 32) != -1;     // Renderable{Entity::none()} => hidden
            }
            const u32 keep = __ballot_sync(0xffffffffu, valid);
            if (valid) {
                const i32 at = running + __popc(keep & ((1u << lane) - 1u));
                if (at < R.maxInstancesPerWorld) {
                    RenderInstance inst;
                    const Vector3 p = ((const Vector3 *)t.columns[ra.cols[RCPosition]])[row];
                    const Quat q = ((const Quat *)t.columns[ra.cols[RCRotation]])[row];
                    const Diag3x3 s = ((const Diag3x3 *)t.columns[ra.cols[RCScale]])[row];
                    inst.position = p;
                    inst.rotation = q;
                    inst.scale = Vector3 { s.d0, s.d1, s.d2 };
                    inst.objectID = ((const i32 *)t.columns[ra.cols[RCObjectID]])[row];
                    // instanceTransformUpdate (no material components: mesh default) /
                    // instanceTransformUpdateWithMat (ecs_system.cpp:100-159, 211-250); a
                    // ColorOverride without a MaterialOverride means "use this colour"
                    inst.color = ra.colorCol >= 0 ? ((const u32 *)t.columns[ra.colorCol])[row] : 0xFFFFFFu;
                    inst.matID = ra.matCol >= 0 ? ((const i32 *)t.columns[ra.matCol])[row]
                                                : (ra.colorCol >= 0 ? -2 : -1);
                    AABB box { { 0, 0, 0 }, { 0, 0, 0 } };
                    if (inst.objectID >= 0 && (u32)inst.objectID < R.numMeshes) {
                        const MeshBVH &m = R.meshes[inst.objectID];
                        box = AABB { { m.rootAABBMin[0], m.rootAABBMin[1], m.rootAABBMin[2] },
                                     { m.rootAABBMax[0], m.rootAABBMax[1], m.rootAABBMax[2] } }.applyTRS(p, q, s);
                    }
                    inst.aabbMin[0] = box.pMin.x; inst.aabbMin[1] = box.pMin.y; inst.aabbMin[2] = box.pMin.z;
                    inst.aabbMax[0] = box.pMax.x; inst.aabbMax[1] = box.pMax.y; inst.aabbMax[2] = box.pMax.z;
                    out[at] = inst;
                }
            }
            running += __popc(keep);
        }
    }
    if (lane == 0) {
        if (running > R.maxInstancesPerWorld) {
            atomicOr(&S.errorFlags, (u32)ErrPhysicsOverflow);
            running = R.maxInstancesPerWorld;
        }
        R.instanceCounts[w] = running;
        atomicAdd(&R.totalNumInstances, (u32)running);
    }
}

// ---- render-prepare: lights -------------------------------------------------------------
// lightUpdate (ecs_system.cpp:183-209): every light carrier writes its current
// description into its light entity; then each world's LightDescs are listed.
__global__ void __launch_bounds__(256)
renderLightUpdateKernel(EngineState *Sp, u32 archetype, i32 carrier_col, i32 pos_col, i32 dir_col, i32 type_col,
                        i32 shadow_col, i32 cutoff_col, i32 intensity_col, i32 active_col)
{
    EngineState &S = *Sp;
    const RenderState &R = *S.render;
    const TableDesc &t = S.tables[archetype];
    const i32 n = t.numRows;
    for (i32 row = blockIdx.x * blockDim.x + threadIdx.x; row < n; row += gridDim.x * blockDim.x) {
        if (((const i32 *)t.columns[1])[row] < 0) continue;
        const u64 packed = ((const u64 *)t.columns[carrier_col])[row];
        const i32 id = (i32)(u32)(packed >> 32);
        const u32 gen = (u32)(packed & 0xFFFFFFFFull);
        if (id < 0 || id >= S.entityCapacity) continue;
        const EntitySlot slot = S.entitySlots[id];
        if (slot.gen != gen || (u32)slot.a != R.lightArchetype) continue;
        LightDesc &d = ((LightDesc *)S.tables[R.lightArchetype].columns[R.lightCol])[slot.b];
        const Vector3 p = ((const Vector3 *)t.columns[pos_col])[row];
        const Vector3 dir = ((const Vector3 *)t.columns[dir_col])[row];
        d.type = ((const LightDesc::Type *)t.columns[type_col])[row];
        d.castShadow = ((const bool *)t.columns[shadow_col])[row];
        d.position = p;
        d.direction = dir;
        d.cutoff = ((const float *)t.columns[cutoff_col])[row];
        d.intensity = ((const float *)t.columns[intensity_col])[row];
        d.active = ((const bool *)t.columns[active_col])[row];
    }
}

__global__ void __launch_bounds__(256)
renderGatherLightsKernel(EngineState *Sp)
{
    EngineState &S = *Sp;
    RenderState &R = *S.render;
    const TableDesc &t = S.tables[R.lightArchetype];
    const i32 W = (i32)S.numWorlds;
    for (i32 w = blockIdx.x * blockDim.x + threadIdx.x; w < W; w += gridDim.x * blockDim.x) {
        const i32 first = t.worldOffsets[w];
        const i32 count = t.worldCounts[w];
        i32 kept = 0;
        for (i32 r = first; r < first + count && kept < kMaxLightsPerWorld; r++) {
            if (((const i32 *)t.columns[1])[r] != w) continue;
            const LightDesc d = ((const LightDesc *)t.columns[R.lightCol])[r];
            RenderLight l;
            l.directional = d.type ? 1u : 0u;
            l.castShadow = d.castShadow ? 1u : 0u;
            l.position = d.position;
            l.direction = d.direction;
            l.cutoff = d.cutoff;
            l.intensity = d.intensity;
            l.active = d.active ? 1u : 0u;
            R.lights[(size_t)w * kMaxLightsPerWorld + kept++] = l;
        }
        R.lightCounts[w] = kept;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        // exportCountsGPU (ecs_system.cpp:317-348)
        R.totalNumViews = (u32)S.tables[R.outputArchetype].numRows;
    }
}

// ---- render-prepare: views (viewTransformUpdate, ecs_system.cpp:275-314) ----------------
__global__ void __launch_bounds__(256)
renderGatherViewsKernel(EngineState *Sp)
{
    EngineState &S = *Sp;
    RenderState &R = *S.render;
    if (blockIdx.y >= R.numViewArchetypes) return;
    const ViewArchetype &va = R.viewers[blockIdx.y];
    const TableDesc &t = S.tables[va.archetype];
    const i32 n = t.numRows;
    const i32 *world_col = (const i32 *)t.columns[1];
    for (i32 row = blockIdx.x * blockDim.x + threadIdx.x; row < n; row += gridDim.x * blockDim.x) {
        const i32 w = world_col[row];
        if (w < 0) continue;
        const RenderCamera cam = ((const RenderCamera *)t.columns[va.camCol])[row];
        const madrona::Entity out = cam.cameraEntity;
        if (out.id < 0 || out.id >= S.entityCapacity) continue;
        const EntitySlot slot = S.entitySlots[out.id];
        if (slot.gen != out.gen || (u32)slot.a != R.outputArchetype) continue;
        const i32 out_row = slot.b;
        if (out_row < 0 || out_row >= R.maxViews) continue;
        const Vector3 p = ((const Vector3 *)t.columns[va.posCol])[row];
        const Quat q = ((const Quat *)t.columns[va.rotCol])[row];
        const Vector3 cam_pos = p + cam.cameraOffset;
        const Quat inv = q.inv();
        RenderView v;
        v.position = cam_pos;
        v.rotation = inv;
        v.xScale = cam.fovScale;          // square output: aspect ratio 1
        v.yScale = -cam.fovScale;
        v.zNear = cam.zNear;
        v.worldIDX = w;
        v.outputRow = out_row;
        R.views[out_row] = v;
    }
}

struct RayShear {
    int kx, ky, kz;
    float Sx, Sy, Sz;
};

// Woop et al. 2013: permute so the dominant direction is z, shear onto it
__device__ __forceinline__ RayShear rayShear(Vector3 d, Diag3x3 inv_d)
{
    const float ax = fabsf(d.x), ay = fabsf(d.y), az = fabsf(d.z);
    int kz = (ax > ay && ax > az) ? 0 : (ay > az ? 1 : 2);
    int kx = kz + 1 == 3 ? 0 : kz + 1;
    int ky = kx + 1 == 3 ? 0 : kx + 1;
    auto pick = [](int k, float x, float y, float z) { return k == 0 ? x : (k == 1 ? y : z); };
    if (pick(kz, d.x, d.y, d.z) < 0.f) {
        int t = kx; kx = ky; ky = t;
    }
    const float inv_kz = pick(kz, inv_d.d0, inv_d.d1, inv_d.d2);
    return RayShear { kx, ky, kz, pick(kx, d.x, d.y, d.z) * inv_kz, pick(ky, d.x, d.y, d.z) * inv_kz, inv_kz };
}

// ---- render-prepare: per-world TLAS ----------------------------------------------------------
// One warp per world; everything lives in the warp's slice of dynamic shared
// memory until the 4-wide nodes are written out.
struct TLASScratch {
    unsigned long long *keys;     // [n] morton << 32 | gather index
    float *leafBox;               // [n][6] in SORTED order
    float *nodeBox;               // [n - 1][6] binary internal nodes
    short *left, *right;          // [n - 1] child: >= 0 internal, < 0: ~leaf (sorted position)
    short *parent;                // [2n - 1]: internal nodes first, then leaves
    int *flags;                   // [n - 1] arrival counters of the bottom-up pass
    short *wideBin;               // [n] binary node of each wide node
    int *order;                   // [n] sorted position -> gather index
};

__host__ __device__ inline size_t tlasScratchBytes(int n)
{
    return (size_t)n * (8 + 24 + 24 + 2 + 2 + 4 + 4 + 2 + 4) + 64;
}

__device__ __forceinline__ u32 expandBits10(u32 v)
{
    v = (v * 0x00010001u) & 0xFF0000FFu;
    v = (v * 0x00000101u) & 0x0F00F00Fu;
    v = (v * 0x00000011u) & 0xC30C30C3u;
    v = (v * 0x00000005u) & 0x49249249u;
    return v;
}

__device__ __forceinline__ int commonPrefix(const unsigned long long *keys, int n, int i, int j)
{
    if (j < 0 || j >= n) return -1;
    return __clzll((long long)(keys[i] ^ keys[j]));     // keys are unique (index in the low word)
}

__global__ void __launch_bounds__(32)
renderBuildTLASKernel(EngineState *Sp)
{
    extern __shared__ __align__(16) unsigned char tlas_smem[];
    EngineState &S = *Sp;
    RenderState &R = *S.render;
    const int lane = threadIdx.x;
    const i32 w = (i32)blockIdx.x;
    const i32 n = R.instanceCounts[w];
    const RenderInstance *inst = R.instances + (size_t)w * R.maxInstancesPerWorld;
    QBVHNode *out = R.tlasNodes + (size_t)w * R.maxInstancesPerWorld;
    if (n <= 0) {
        if (lane == 0) R.tlasNodeCounts[w] = 0;
        return;
    }
    const int cap = R.maxInstancesPerWorld;
    TLASScratch sc;
    {
        unsigned char *p = tlas_smem;
        sc.keys = (unsigned long long *)p; p += (size_t)cap * 8;
        sc.leafBox = (float *)p; p += (size_t)cap * 24;
        sc.nodeBox = (float *)p; p += (size_t)cap * 24;
        sc.flags = (int *)p; p += (size_t)cap * 4;
        sc.order = (int *)p; p += (size_t)cap * 4;
        sc.left = (short *)p; p += (size_t)cap * 2;
        sc.right = (short *)p; p += (size_t)cap * 2;
        sc.parent = (short *)p; p += (size_t)cap * 4;
        sc.wideBin = (short *)p;
    }

    // 1. world bounds of the box centres, Morton keys
    float lo[3] = { FLT_MAX, FLT_MAX, FLT_MAX }, hi[3] = { -FLT_MAX, -FLT_MAX, -FLT_MAX };
    for (int i = lane; i < n; i += 32) {
        for (int a = 0; a < 3; a++) {
            const float c = 0.5f * (inst[i].aabbMin[a] + inst[i].aabbMax[a]);
            lo[a] = fminf(lo[a], c);
            hi[a] = fmaxf(hi[a], c);
        }
    }
    for (int o = 16; o >= 1; o >>= 1) {
        for (int a = 0; a < 3; a++) {
            lo[a] = fminf(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmaxf(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
    }
    for (int i = lane; i < n; i += 32) {
        u32 code = 0;
        for (int a = 0; a < 3; a++) {
            const float c = 0.5f * (inst[i].aabbMin[a] + inst[i].aabbMax[a]);
            const float ext = hi[a] - lo[a];
            float u = ext > 0.f ? (c - lo[a]) / ext : 0.f;
            u = fminf(fmaxf(u * 1024.f, 0.f), 1023.f);
            code |= expandBits10((u32)u) << a;
        }
        sc.keys[i] = ((unsigned long long)code << 32) | (u32)i;
    }
    __syncwarp();

    // 2. rank sort (n is tens to a few hundred): sorted position of every instance
    for (int i = lane; i < n; i += 32) {
        const unsigned long long mine = sc.keys[i];
        int rank = 0;
        for (int j = 0; j < n; j++) rank += sc.keys[j] < mine ? 1 : 0;
        sc.order[rank] = i;
    }
    __syncwarp();
    // keys / boxes in sorted order (keys rewritten in place through registers)
    {
        unsigned long long mine[16];
        const int per = (n + 31) / 32;
        for (int k = 0; k < per && k < 16; k++) {
            const int pos = lane + 32 * k;
            mine[k] = pos < n ? sc.keys[sc.order[pos]] : 0ull;
        }
        __syncwarp();
        for (int k = 0; k < per && k < 16; k++) {
            const int pos = lane + 32 * k;
            if (pos < n) {
                sc.keys[pos] = mine[k];
                const RenderInstance &ri = inst[sc.order[pos]];
                for (int a = 0; a < 3; a++) {
                    sc.leafBox[pos * 6 + a] = ri.aabbMin[a];
                    sc.leafBox[pos * 6 + 3 + a] = ri.aabbMax[a];
                }
            }
        }
    }
    __syncwarp();

    if (n == 1) {
        if (lane == 0) {
            float cmin[kBVHWidth][3], cmax[kBVHWidth][3];
            for (int a = 0; a < 3; a++) {
                cmin[0][a] = sc.leafBox[a];
                cmax[0][a] = sc.leafBox[3 + a];
            }
            QBVHNode node;
            quantizeNode(node, 1, cmin, cmax);
            node.childrenIdx[0] = 0x80000000u | (u32)sc.order[0];
            node.triSize[0] = 0;
            out[0] = node;
            R.tlasNodeCounts[w] = 1;
        }
        return;
    }

    // 3. Karras 2012: internal node i covers a key range; leaves are sorted positions
    for (int i = lane; i < n - 1; i += 32) {
        const int d = commonPrefix(sc.keys, n, i, i + 1) - commonPrefix(sc.keys, n, i, i - 1) >= 0 ? 1 : -1;
        const int delta_min = commonPrefix(sc.keys, n, i, i - d);
        int lmax = 2;
        while (commonPrefix(sc.keys, n, i, i + lmax * d) > delta_min) lmax <<= 1;
        int l = 0;
        for (int t = lmax >> 1; t >= 1; t >>= 1) {
            if (commonPrefix(sc.keys, n, i, i + (l + t) * d) > delta_min) l += t;
        }
        const int j = i + l * d;
        const int delta_node = commonPrefix(sc.keys, n, i, j);
        int s = 0;
        for (int t = (l + 1) >> 1; ; t = (t + 1) >> 1) {
            if (commonPrefix(sc.keys, n, i, i + (s + t) * d) > delta_node) s += t;
            if (t == 1) break;
        }
        const int gamma = i + s * d + min(d, 0);
        const int first = min(i, j), last = max(i, j);
        const int lc = first == gamma ? ~gamma : gamma;             // leaf: ~position
        const int rc = last == gamma + 1 ? ~(gamma + 1) : gamma + 1;
        sc.left[i] = (short)lc;
        sc.right[i] = (short)rc;
        sc.parent[lc >= 0 ? lc : (n - 1) + (~lc)] = (short)i;
        sc.parent[rc >= 0 ? rc : (n - 1) + (~rc)] = (short)i;
        sc.flags[i] = 0;
    }
    if (lane == 0) sc.parent[0] = -1;
    __syncwarp();

    // 4. boxes, bottom-up: the second thread to reach a node owns it
    for (int leaf = lane; leaf < n; leaf += 32) {
        int node = sc.parent[(n - 1) + leaf];
        while (node >= 0) {
            __threadfence_block();
            if (atomicAdd(&sc.flags[node], 1) == 0) break;
            const int lc = sc.left[node], rc = sc.right[node];
            const float *lb = lc >= 0 ? sc.nodeBox + lc * 6 : sc.leafBox + (~lc) * 6;
            const float *rb = rc >= 0 ? sc.nodeBox + rc * 6 : sc.leafBox + (~rc) * 6;
            for (int a = 0; a < 3; a++) {
                sc.nodeBox[node * 6 + a] = fminf(lb[a], rb[a]);
                sc.nodeBox[node * 6 + 3 + a] = fmaxf(lb[3 + a], rb[3 + a]);
            }
            node = sc.parent[node];
        }
    }
    __syncwarp();

    // 5. collapse to 4-wide nodes, breadth first; flags[0] now counts wide nodes
    if (lane == 0) {
        sc.wideBin[0] = 0;
        sc.flags[0] = 1;
    }
    __syncwarp();
    // waves: nodes [done, count) exist and are not written yet; writing them appends
    // their inner children behind `count`
    for (int done = 0;;) {
        const int count_now = *(volatile int *)&sc.flags[0];
        if (done >= count_now) break;
        const int k = done + lane;
        __syncwarp();
        if (k < count_now) {
            const int bin = sc.wideBin[k];
            int kids[kBVHWidth];
            int nk = 2;
            kids[0] = sc.left[bin];
            kids[1] = sc.right[bin];
            while (nk < kBVHWidth) {
                int pick = -1;
                float best = -1.f;
                for (int c = 0; c < nk; c++) {
                    if (kids[c] < 0) continue;
                    const float *b = sc.nodeBox + kids[c] * 6;
                    const float dx = b[3] - b[0], dy = b[4] - b[1], dz = b[5] - b[2];
                    const float area = dx * dy + dy * dz + dz * dx;
                    if (area > best) {
                        best = area;
                        pick = c;
                    }
                }
                if (pick < 0) break;
                const int inner = kids[pick];
                kids[pick] = sc.left[inner];
                kids[nk++] = sc.right[inner];
            }
            float cmin[kBVHWidth][3], cmax[kBVHWidth][3];
            for (int c = 0; c < nk; c++) {
                const float *b = kids[c] >= 0 ? sc.nodeBox + kids[c] * 6 : sc.leafBox + (~kids[c]) * 6;
                for (int a = 0; a < 3; a++) {
                    cmin[c][a] = b[a];
                    cmax[c][a] = b[3 + a];
                }
            }
            QBVHNode node;
            quantizeNode(node, nk, cmin, cmax);
            for (int c = 0; c < nk; c++) {
                node.triSize[c] = 0;
                if (kids[c] < 0) {
                    node.childrenIdx[c] = 0x80000000u | (u32)sc.order[~kids[c]];
                } else {
                    const int id = atomicAdd(&sc.flags[0], 1);
                    sc.wideBin[id] = (short)kids[c];
                    node.childrenIdx[c] = (u32)id;
                }
            }
            out[k] = node;
        }
        __syncwarp();
        done = min(done + 32, count_now);
    }
    if (lane == 0) R.tlasNodeCounts[w] = sc.flags[0];
}

// ---- ray casting ------------------------------------------------------------------------------
// Closest hit of camera rays against one world.  Two ways to find the instances a ray enters:
//   * worlds with <= kFlatInstances instances (the simulators' case: Escape Room 33): the view's
//     block stages every instance ONCE in shared memory -- world -> object matrix, object-space
//     camera origin, world box -- sorted front to back; each warp culls that list against the
//     sub-frustum of its 8 x 4 pixel tile (one 64-bit mask), and a ray only slab-tests the
//     survivors.  No tree, no per-ray quaternion algebra, a uniform loop across the warp.
//   * larger worlds: stack traversal of the per-world TLAS (quantised 4-wide nodes).
// Inside an instance both run the same BLAS traversal (reference-format quantised MeshBVH,
// watertight triangle test).  Object-space rays keep the world ray's parametrisation (the
// direction is NOT renormalised), so t needs no rescaling.

struct RayHit {
    float t;
    int instance;           // gather index inside the world, -1: miss
    int triangle;           // triangle index inside the instance's mesh
};

constexpr int kTraceStack = 48;     // TLAS + BLAS entries of one ray
constexpr int kFlatInstances = 64;

__device__ __forceinline__ float safeRcp(float x)
{
    // 1 / x; a zero component behaves like +-1e-7 (mesh_bvh.inl:100-110)
    return x == 0.f ? copysignf(1e7f, x) : __frcp_rn(x);
}

// byte i of a packed 4 x u8 word as a float without an int -> float conversion:
// 0x4B0000qq is the float 2^23 + qq
template <int I>
__device__ __forceinline__ float byteAsFloat(u32 word)
{
    return __uint_as_float(__byte_perm(word, 0x4B000000u, 0x7650 + I)) - 8388608.f;
}

// world -> object map of an instance: x_obj = m * (x_world - pos), m = scale^-1 * R(q)^T;
// R(q) is the matrix of Quat::rotateVec (valid for slightly non-unit q as well)
struct InstanceXform {
    float m[9];
};

__device__ __forceinline__ InstanceXform instanceXform(const RenderInstance &inst)
{
    const float w = inst.rotation.w, x = inst.rotation.x, y = inst.rotation.y, z = inst.rotation.z;
    const float diag = 1.f - 2.f * (x * x + y * y + z * z);
    // R = diag * I + 2 u u^T + 2 w [u]x
    const float r00 = diag + 2.f * x * x, r01 = 2.f * (x * y - w * z), r02 = 2.f * (x * z + w * y);
    const float r10 = 2.f * (x * y + w * z), r11 = diag + 2.f * y * y, r12 = 2.f * (y * z - w * x);
    const float r20 = 2.f * (x * z - w * y), r21 = 2.f * (y * z + w * x), r22 = diag + 2.f * z * z;
    const float isx = __frcp_rn(inst.scale.x), isy = __frcp_rn(inst.scale.y), isz = __frcp_rn(inst.scale.z);
    InstanceXform X;
    X.m[0] = r00 * isx; X.m[1] = r10 * isx; X.m[2] = r20 * isx;
    X.m[3] = r01 * isy; X.m[4] = r11 * isy; X.m[5] = r21 * isy;
    X.m[6] = r02 * isz; X.m[7] = r12 * isz; X.m[8] = r22 * isz;
    return X;
}

__device__ __forceinline__ Vector3 applyLinear(const float *m, Vector3 v)
{
    return Vector3 { m[0] * v.x + m[1] * v.y + m[2] * v.z,
                     m[3] * v.x + m[4] * v.y + m[5] * v.z,
                     m[6] * v.x + m[7] * v.y + m[8] * v.z };
}

__device__ __forceinline__ bool instanceTraceable(const RenderState &R, const RenderInstance &inst)
{
    return inst.scale.x != 0.f && inst.scale.y != 0.f && inst.scale.z != 0.f && inst.objectID >= 0 &&
        (u32)inst.objectID < R.numMeshes;
}

// watertight ray-triangle test (Woop et al. 2013), t only
__device__ __forceinline__ bool rayTriangleT(const BVHVertex *v, const RayShear &rs, Vector3 org, float t_min,
                                             float t_max, float *out_t)
{
    const Vector3 A { v[0].pos[0] - org.x, v[0].pos[1] - org.y, v[0].pos[2] - org.z };
    const Vector3 B { v[1].pos[0] - org.x, v[1].pos[1] - org.y, v[1].pos[2] - org.z };
    const Vector3 C { v[2].pos[0] - org.x, v[2].pos[1] - org.y, v[2].pos[2] - org.z };
    // component selection by compares (a dynamically indexed Vector3 would live in local memory)
    auto pick = [](int k, const Vector3 &p) { return k == 0 ? p.x : (k == 1 ? p.y : p.z); };
    const float a_kz = pick(rs.kz, A), a_kx = pick(rs.kx, A), a_ky = pick(rs.ky, A);
    const float b_kz = pick(rs.kz, B), b_kx = pick(rs.kx, B), b_ky = pick(rs.ky, B);
    const float c_kz = pick(rs.kz, C), c_kx = pick(rs.kx, C), c_ky = pick(rs.ky, C);

    const float Ax = fmaf(-rs.Sx, a_kz, a_kx), Ay = fmaf(-rs.Sy, a_kz, a_ky);
    const float Bx = fmaf(-rs.Sx, b_kz, b_kx), By = fmaf(-rs.Sy, b_kz, b_ky);
    const float Cx = fmaf(-rs.Sx, c_kz, c_kx), Cy = fmaf(-rs.Sy, c_kz, c_ky);

    float U = fmaf(Cx, By, -Cy * Bx);
    float V = fmaf(Ax, Cy, -Ay * Cx);
    float W = fmaf(Bx, Ay, -By * Ax);

    constexpr float eps = 1e-7;
    if (U > -eps && U < eps) U = 0.f;
    if (V > -eps && V < eps) V = 0.f;
    if (W > -eps && W < eps) W = 0.f;

    if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return false;

    if (U == 0.0f || V == 0.0f || W == 0.0f) {
        // edge case: redo the edge functions in double precision
        U = (float)((double)Cx * (double)By - (double)Cy * (double)Bx);
        V = (float)((double)Ax * (double)Cy - (double)Ay * (double)Cx);
        W = (float)((double)Bx * (double)Ay - (double)By * (double)Ax);
        if ((U < 0.0f || V < 0.0f || W < 0.0f) && (U > 0.0f || V > 0.0f || W > 0.0f)) return false;
    }

    const float det = U + V + W;
    if (det == 0.f) return false;

    const float Az = rs.Sz * a_kz, Bz = rs.Sz * b_kz, Cz = rs.Sz * c_kz;
    const float T = fmaf(U, Az, fmaf(V, Bz, W * Cz));

    const u32 sign = __float_as_uint(det) & 0x80000000u;
    const float xor_T = __uint_as_float(__float_as_uint(T) ^ sign);
    const float abs_det = fabsf(det);
    if (xor_T < 0.0f || xor_T > t_max * abs_det) return false;

    const float t = T * __frcp_rn(det);
    if (!(t >= t_min)) return false;
    *out_t = t;
    return true;
}

// BLAS traversal of one mesh with an object-space ray; shrinks t_best, reports the triangle.
// `stack` entries [sp0, kTraceStack) are free.
template <bool ANY_HIT>
__device__ __forceinline__ bool traceMesh(const MeshBVH &mesh, const Vector3 oo, const Vector3 od,
                                          const float t_min, float &t_best, int &tri_best, int *stack,
                                          const int sp0)
{
    const float ix = safeRcp(od.x), iy = safeRcp(od.y), iz = safeRcp(od.z);
    const RayShear rs = rayShear(od, Diag3x3 { ix, iy, iz });
    const QBVHNode *nodes = mesh.nodes;
    const BVHVertex *verts = mesh.vertices;
    bool hit = false;
    int sp = sp0;
    if (sp < kTraceStack) stack[sp++] = 0;
    while (sp > sp0) {
        const QBVHNode &bn = nodes[stack[--sp]];
        // child boxes in the node's quantised frame (mesh_bvh.inl:100-160)
        const u32 exps = *(const u32 *)&bn.expX;
        const float sx = __uint_as_float((u32)((int)(signed char)(exps & 0xffu) + 127) << 23) * ix;
        const float sy = __uint_as_float((u32)((int)(signed char)((exps >> 8) & 0xffu) + 127) << 23) * iy;
        const float sz = __uint_as_float((u32)((int)(signed char)((exps >> 16) & 0xffu) + 127) << 23) * iz;
        const float bx = (bn.minPoint[0] - oo.x) * ix;
        const float by = (bn.minPoint[1] - oo.y) * iy;
        const float bz = (bn.minPoint[2] - oo.z) * iz;
        const u32 qnx = *(const u32 *)bn.qMinX, qny = *(const u32 *)bn.qMinY, qnz = *(const u32 *)bn.qMinZ;
        const u32 qfx = *(const u32 *)bn.qMaxX, qfy = *(const u32 *)bn.qMaxY, qfz = *(const u32 *)bn.qMaxZ;
        const u32 tri_sizes = *(const u32 *)bn.triSize;

        auto visit = [&](const u32 child, const float nx, const float fx, const float ny, const float fy,
                         const float nz, const float fz, const u32 tri_count) {
            if (child == 0xFFFFFFFFu) return;
            const float t_near = fmaxf(fminf(nx, fx), fmaxf(fminf(ny, fy), fmaxf(fminf(nz, fz), 0.f)));
            const float t_far = fminf(fmaxf(nx, fx), fminf(fmaxf(ny, fy), fminf(fmaxf(nz, fz), t_best)));
            if (!(t_near <= t_far)) return;
            if (!(child & 0x80000000u)) {
                if (sp < kTraceStack) stack[sp++] = (int)child;
                return;
            }
            const u32 first_tri = child & 0x7FFFFFFFu;
            for (u32 k = 0; k < tri_count; k++) {
                float t;
                if (rayTriangleT(verts + (size_t)(first_tri + k) * 3, rs, oo, t_min, t_best, &t)) {
                    t_best = t;
                    tri_best = (int)(first_tri + k);
                    hit = true;
                }
            }
        };
        visit(bn.childrenIdx[0], byteAsFloat<0>(qnx) * sx + bx, byteAsFloat<0>(qfx) * sx + bx,
              byteAsFloat<0>(qny) * sy + by, byteAsFloat<0>(qfy) * sy + by,
              byteAsFloat<0>(qnz) * sz + bz, byteAsFloat<0>(qfz) * sz + bz, tri_sizes & 0xffu);
        visit(bn.childrenIdx[1], byteAsFloat<1>(qnx) * sx + bx, byteAsFloat<1>(qfx) * sx + bx,
              byteAsFloat<1>(qny) * sy + by, byteAsFloat<1>(qfy) * sy + by,
              byteAsFloat<1>(qnz) * sz + bz, byteAsFloat<1>(qfz) * sz + bz, (tri_sizes >> 8) & 0xffu);
        visit(bn.childrenIdx[2], byteAsFloat<2>(qnx) * sx + bx, byteAsFloat<2>(qfx) * sx + bx,
              byteAsFloat<2>(qny) * sy + by, byteAsFloat<2>(qfy) * sy + by,
              byteAsFloat<2>(qnz) * sz + bz, byteAsFloat<2>(qfz) * sz + bz, (tri_sizes >> 16) & 0xffu);
        visit(bn.childrenIdx[3], byteAsFloat<3>(qnx) * sx + bx, byteAsFloat<3>(qfx) * sx + bx,
              byteAsFloat<3>(qny) * sy + by, byteAsFloat<3>(qfy) * sy + by,
              byteAsFloat<3>(qnz) * sz + bz, byteAsFloat<3>(qfz) * sz + bz, (tri_sizes >> 24) & 0xffu);
        if (ANY_HIT && hit) return true;
    }
    return hit;
}

// child boxes of a quantised TLAS node against a world-space ray
struct NodeRay {
    float dirX, dirY, dirZ;     // 2^exp / d
    float orgX, orgY, orgZ;     // (minPoint - o) / d
};

__device__ __forceinline__ NodeRay nodeRay(const QBVHNode &node, Vector3 o, float ix, float iy, float iz)
{
    NodeRay r;
    r.dirX = __uint_as_float((u32)(node.expX + 127) << 23) * ix;
    r.dirY = __uint_as_float((u32)(node.expY + 127) << 23) * iy;
    r.dirZ = __uint_as_float((u32)(node.expZ + 127) << 23) * iz;
    r.orgX = (node.minPoint[0] - o.x) * ix;
    r.orgY = (node.minPoint[1] - o.y) * iy;
    r.orgZ = (node.minPoint[2] - o.z) * iz;
    return r;
}

__device__ __forceinline__ bool childHit(const QBVHNode &node, const NodeRay &r, int i, float t_max)
{
    const float nx = node.qMinX[i] * r.dirX + r.orgX, fx = node.qMaxX[i] * r.dirX + r.orgX;
    const float ny = node.qMinY[i] * r.dirY + r.orgY, fy = node.qMaxY[i] * r.dirY + r.orgY;
    const float nz = node.qMinZ[i] * r.dirZ + r.orgZ, fz = node.qMaxZ[i] * r.dirZ + r.orgZ;
    const float t_near = fmaxf(fminf(nx, fx), fmaxf(fminf(ny, fy), fmaxf(fminf(nz, fz), 0.f)));
    const float t_far = fminf(fmaxf(nx, fx), fminf(fmaxf(ny, fy), fminf(fmaxf(nz, fz), t_max)));
    return t_near <= t_far;
}

// Closest hit (ANY_HIT: first hit) of a world-space ray through the world's TLAS.
template <bool ANY_HIT>
__device__ RayHit traceWorld(const RenderState &R, const QBVHNode *tlas, const i32 tlas_nodes,
                             const RenderInstance *instances, Vector3 o, Vector3 d, float t_min, float t_max,
                             int *stack)
{
    RayHit hit { t_max, -1, -1 };
    if (tlas_nodes <= 0) return hit;
    const float ix = safeRcp(d.x), iy = safeRcp(d.y), iz = safeRcp(d.z);
    int sp = 0;
    stack[sp++] = 0;
    while (sp > 0) {
        const QBVHNode &node = tlas[stack[--sp]];
        const NodeRay nr = nodeRay(node, o, ix, iy, iz);
#pragma unroll
        for (int c = 0; c < kBVHWidth; c++) {
            const u32 child = node.childrenIdx[c];
            if (child == 0xFFFFFFFFu) continue;
            if (!childHit(node, nr, c, hit.t)) continue;
            if (!(child & 0x80000000u)) {
                if (sp < kTraceStack) stack[sp++] = (int)child;
                continue;
            }
            const int ii = (int)(child & 0x7FFFFFFFu);
            const RenderInstance &inst = instances[ii];
            if (!instanceTraceable(R, inst)) continue;
            const InstanceXform X = instanceXform(inst);
            const Vector3 oo = applyLinear(X.m, o - inst.position);
            const Vector3 od = applyLinear(X.m, d);
            int tri = -1;
            if (traceMesh<ANY_HIT>(R.meshes[inst.objectID], oo, od, t_min, hit.t, tri, stack, sp)) {
                hit.instance = ii;
                hit.triangle = tri;
                if (ANY_HIT) return hit;
            }
        }
    }
    return hit;
}

// One instance staged for a view (shared memory)
struct FlatInstance {
    float m[9];             // world -> object, linear part
    float pos[3];           // instance position
    float oo[3];            // object-space origin of the view's primary rays
    float lo[3], hi[3];     // world box relative to the view origin
    i32 index;              // gather index inside the world (RayHit::instance)
    i32 mesh;               // MeshBVH index; -1: nothing to trace (bad scale / object id)
    i32 inView;             // reaches into the view frustum (camera rays only need these)
};

// world box (relative to o) against a ray from o: entered before t_max?
__device__ __forceinline__ bool boxHit(const float *lo, const float *hi, float ix, float iy, float iz, float t_max)
{
    const float nx = lo[0] * ix, fx = hi[0] * ix;
    const float ny = lo[1] * iy, fy = hi[1] * iy;
    const float nz = lo[2] * iz, fz = hi[2] * iz;
    const float t_near = fmaxf(fminf(nx, fx), fmaxf(fminf(ny, fy), fmaxf(fminf(nz, fz), 0.f)));
    const float t_far = fminf(fmaxf(nx, fx), fminf(fmaxf(ny, fy), fminf(fmaxf(nz, fz), t_max)));
    return t_near <= t_far;
}

// Closest / first hit against the staged instance list.  PRIMARY: the ray starts at the view
// origin (staged object-space origin and relative boxes are used as they are); otherwise
// `shift` = view origin - ray origin re-bases them.
template <bool ANY_HIT, bool PRIMARY>
__device__ __forceinline__ RayHit traceFlat(const RenderState &R, const FlatInstance *list, unsigned long long mask,
                                            Vector3 o, Vector3 d, Vector3 shift, float t_min, float t_max,
                                            int *stack)
{
    RayHit hit { t_max, -1, -1 };
    const float ix = safeRcp(d.x), iy = safeRcp(d.y), iz = safeRcp(d.z);
    while (mask) {
        const int k = __ffsll((long long)mask) - 1;
        mask &= mask - 1;
        const FlatInstance &fi = list[k];
        bool enter;
        if (PRIMARY) {
            enter = boxHit(fi.lo, fi.hi, ix, iy, iz, hit.t);
        } else {
            const float lo[3] = { fi.lo[0] + shift.x, fi.lo[1] + shift.y, fi.lo[2] + shift.z };
            const float hi[3] = { fi.hi[0] + shift.x, fi.hi[1] + shift.y, fi.hi[2] + shift.z };
            enter = boxHit(lo, hi, ix, iy, iz, hit.t);
        }
        if (!enter) continue;
        const Vector3 oo = PRIMARY ? Vector3 { fi.oo[0], fi.oo[1], fi.oo[2] }
                                   : applyLinear(fi.m, o - Vector3 { fi.pos[0], fi.pos[1], fi.pos[2] });
        const Vector3 od = applyLinear(fi.m, d);
        int tri = -1;
        if (traceMesh<ANY_HIT>(R.meshes[fi.mesh], oo, od, t_min, hit.t, tri, stack, 0)) {
            hit.instance = fi.index;
            hit.triangle = tri;
            if (ANY_HIT) return hit;
        }
    }
    return hit;
}

__device__ __forceinline__ Vector3 hexToRgb(u32 hex)
{
    return Vector3 { ((hex >> 16) & 0xFF) / 255.0f, ((hex >> 8) & 0xFF) / 255.0f, (hex & 0xFF) / 255.0f };
}

// is the box (lo, hi relative to the apex) completely on the negative side of the plane n . x = 0 ?
__device__ __forceinline__ bool boxOutside(const float *lo, const float *hi, Vector3 n)
{
    const float cx = 0.5f * (lo[0] + hi[0]), cy = 0.5f * (lo[1] + hi[1]), cz = 0.5f * (lo[2] + hi[2]);
    const float hx = 0.5f * (hi[0] - lo[0]), hy = 0.5f * (hi[1] - lo[1]), hz = 0.5f * (hi[2] - lo[2]);
    const float reach = n.x * cx + n.y * cy + n.z * cz + fabsf(n.x) * hx + fabsf(n.y) * hy + fabsf(n.z) * hz;
    return reach < 0.f;
}

#ifndef MB2_RAYCAST_MINB
#define MB2_RAYCAST_MINB 3
#endif
// FLAT: this launch traces the views of worlds with <= kFlatInstances instances, the other
// instantiation the rest (a view belongs to exactly one of the two launches)
template <bool FLAT>
__global__ void __launch_bounds__(256, MB2_RAYCAST_MINB)
renderRaycastKernel(EngineState *Sp)
{
    EngineState &S = *Sp;
    const RenderState &R = *S.render;
    const TableDesc &out_tbl = S.tables[R.outputArchetype];
    const i32 num_views = min(out_tbl.numRows, R.maxViews);
    const u32 res = R.resolution;
    // One block traces a whole view; a warp traces 8 x 4 pixel tiles: coherent
    // rays (same instances entered, same dominant axis) instead of 32-pixel row segments.
    const u32 tiles_x = (res + 7) / 8;
    const u32 num_tiles = tiles_x * ((res + 3) / 4);
    const size_t bytes_per_view = (size_t)res * res * 4;
    const int lane = threadIdx.x & 31;
    int stack[kTraceStack];

    __shared__ FlatInstance s_list[kFlatInstances];      // sorted front to back
    __shared__ FlatInstance s_unsorted[kFlatInstances];
    __shared__ float s_key[kFlatInstances];

    for (i32 v = blockIdx.y; v < num_views; v += gridDim.y) {
        const RenderView view = R.views[v];
        const i32 w = view.worldIDX;
        const QBVHNode *tlas = R.tlasNodes + (size_t)w * R.maxInstancesPerWorld;
        const i32 tlas_nodes = R.tlasNodeCounts[w];
        const RenderInstance *instances = R.instances + (size_t)w * R.maxInstancesPerWorld;
        const i32 num_instances = R.instanceCounts[w];
        const RenderLight *lights = R.lights + (size_t)w * kMaxLightsPerWorld;
        const i32 num_lights = R.lightCounts[w];
        constexpr bool flat = FLAT;
        if ((num_instances <= kFlatInstances) != FLAT) continue;

        // camera frame (shared by every pixel of the view)
        const Quat rot = view.rotation;
        const Vector3 ray_start = view.position;
        const Vector3 look_at = rot.inv().rotateVec({ 0, 1, 0 });
        const float h = 1.0f / (-view.yScale);
        const float viewport = 2 * h;
        const Vector3 forward = look_at.normalize();
        const Vector3 u = rot.inv().rotateVec({ 1, 0, 0 });
        const Vector3 vv = cross(forward, u).normalize();

        // ---- stage the world's instances, front to back, culled against the view frustum
        __syncthreads();        // the previous view's rays are done with the list
        if (flat) {
            const int i = (int)threadIdx.x;
            if (i < num_instances) {
                FlatInstance &fi = s_unsorted[i];
                const RenderInstance &inst = instances[i];
                fi.index = i;
                fi.mesh = instanceTraceable(R, inst) ? inst.objectID : -1;
                const InstanceXform X = instanceXform(inst);
#pragma unroll
                for (int k = 0; k < 9; k++) fi.m[k] = X.m[k];
                fi.pos[0] = inst.position.x; fi.pos[1] = inst.position.y; fi.pos[2] = inst.position.z;
                const Vector3 oo = applyLinear(X.m, ray_start - inst.position);
                fi.oo[0] = oo.x; fi.oo[1] = oo.y; fi.oo[2] = oo.z;
                float lo[3], hi[3];
                float dist2 = 0.f;
#pragma unroll
                for (int a = 0; a < 3; a++) {
                    lo[a] = inst.aabbMin[a] - ray_start[a];
                    hi[a] = inst.aabbMax[a] - ray_start[a];
                    fi.lo[a] = lo[a];
                    fi.hi[a] = hi[a];
                    const float gap = fmaxf(fmaxf(lo[a], -hi[a]), 0.f);    // distance to the box on this axis
                    dist2 += gap * gap;
                }
                // whole-view frustum: |a| <= h c, |b| <= h c, c >= 0 in the (u, vv, forward) frame
                const float pad = fabsf(h) * (1.f + 2.f / (float)res);
                const bool outside = boxOutside(lo, hi, forward) ||
                    boxOutside(lo, hi, u + pad * forward) || boxOutside(lo, hi, pad * forward - u) ||
                    boxOutside(lo, hi, vv + pad * forward) || boxOutside(lo, hi, pad * forward - vv);
                fi.inView = outside ? 0 : 1;
                s_key[i] = dist2;
            }
            __syncthreads();
            if (i < num_instances) {
                const float key = s_key[i];
                int rank = 0;
                for (int j = 0; j < num_instances; j++) {
                    const float kj = s_key[j];
                    rank += (kj < key || (kj == key && j < i)) ? 1 : 0;
                }
                const u32 *src = (const u32 *)&s_unsorted[i];
                u32 *dst = (u32 *)&s_list[rank];
#pragma unroll
                for (int k = 0; k < (int)(sizeof(FlatInstance) / 4); k++) dst[k] = src[k];
            }
            __syncthreads();
        }

        // instances a shadow ray may hit: all with a mesh (warp-uniform mask)
        unsigned long long mesh_mask = 0;
        if (flat && num_lights > 0) {
#pragma unroll
            for (int half = 0; half < kFlatInstances / 32; half++) {
                const int k = half * 32 + lane;
                const bool keep = k < num_instances && s_list[k].mesh >= 0;
                mesh_mask |= (unsigned long long)__ballot_sync(0xffffffffu, keep) << (32 * half);
            }
        }

        for (u32 tile = threadIdx.x >> 5; tile < num_tiles; tile += blockDim.x >> 5) {
            const u32 tx0 = (tile % tiles_x) * 8, ty0 = (tile / tiles_x) * 4;
            const u32 px = tx0 + (threadIdx.x & 7);
            const u32 py = ty0 + ((threadIdx.x & 31) >> 3);

            // ---- instances that reach into this tile's sub-frustum (warp-uniform mask)
            unsigned long long tile_mask = 0;
            if (flat) {
                const float inv_res = 1.f / (float)res;
                // tile edges, a quarter pixel wider (the rays go through pixel centres)
                const float a0 = ((float)tx0 * inv_res - 0.25f * inv_res - 0.5f) * viewport;
                const float a1 = ((float)(tx0 + 8) * inv_res + 0.25f * inv_res - 0.5f) * viewport;
                const float b0 = ((float)ty0 * inv_res - 0.25f * inv_res - 0.5f) * viewport;
                const float b1 = ((float)(ty0 + 4) * inv_res + 0.25f * inv_res - 0.5f) * viewport;
                // (a mirrored projection, h < 0, only swaps which edge is which)
                const float al = fminf(a0, a1), ar = fmaxf(a0, a1), bl = fminf(b0, b1), br = fmaxf(b0, b1);
                const Vector3 n_left = u - al * forward, n_right = ar * forward - u;
                const Vector3 n_bottom = vv - bl * forward, n_top = br * forward - vv;
#pragma unroll
                for (int half = 0; half < kFlatInstances / 32; half++) {
                    const int k = half * 32 + lane;
                    bool keep = false;
                    if (k < num_instances) {
                        const FlatInstance &fi = s_list[k];
                        keep = fi.mesh >= 0 && fi.inView && !boxOutside(fi.lo, fi.hi, n_left) && !boxOutside(fi.lo, fi.hi, n_right) &&
                            !boxOutside(fi.lo, fi.hi, n_bottom) && !boxOutside(fi.lo, fi.hi, n_top);
                    }
                    tile_mask |= (unsigned long long)__ballot_sync(0xffffffffu, keep) << (32 * half);
                }
            }
            if (px >= res || py >= res) continue;

            // ---- primary ray (bvh_raycast.cpp:58-88)
            const Vector3 horizontal = u * viewport;
            const Vector3 vertical = vv * viewport;
            const Vector3 lower_left = ray_start - horizontal / 2 - vertical / 2 + forward;
            const float pu = ((float)px + 0.5f) / (float)res;
            const float pv = ((float)py + 0.5f) / (float)res;
            Vector3 ray_dir = lower_left + pu * horizontal + pv * vertical - ray_start;
            ray_dir = ray_dir.normalize();

            const RayHit first = flat
                ? traceFlat<false, true>(R, s_list, tile_mask, ray_start, ray_dir, Vector3 { 0, 0, 0 }, 0.f, 10000.f, stack)
                : traceWorld<false>(R, tlas, tlas_nodes, instances, ray_start, ray_dir, 0.f, 10000.f, stack);
            const bool hit = first.instance >= 0;

            const size_t pix = (size_t)px + (size_t)py * res;
            const size_t off = (size_t)view.outputRow * bytes_per_view + 4 * pix;
            float *depth_out = (float *)((char *)out_tbl.columns[R.depthCol] + off);
            *depth_out = hit ? first.t : 0.f;
            if (R.hitIDs) {
                i32 *ids = R.hitIDs + ((size_t)view.outputRow * res * res + pix) * 2;
                ids[0] = hit ? first.instance : -1;
                ids[1] = hit ? first.triangle : -1;
            }
            if (!R.rgbd) continue;

            unsigned char *rgb = (unsigned char *)out_tbl.columns[R.rgbCol] + off;
            Vector3 color { 0.f, 0.f, 0.f };
            if (hit) {
                // colour of the hit (bvh_raycast.cpp:756-815, textures excepted)
                const RenderInstance &inst = instances[first.instance];
                const MeshBVH &mesh = R.meshes[inst.objectID];
                i32 material_idx = inst.matID;
                if (material_idx == -1) {
                    material_idx = mesh.materialIDX != -1 ? mesh.materialIDX
                                                          : mesh.leafMats[first.triangle].matIDX;
                }
                Vector3 base { 1.f, 1.f, 1.f };
                if (inst.matID == -2) {
                    base = hexToRgb(inst.color);
                } else if (material_idx >= 0 && R.materials) {
                    const RenderMaterial &m = R.materials[material_idx];
                    base = Vector3 { m.color[0], m.color[1], m.color[2] };
                }

                float light_contrib = 0.f;
                if (num_lights > 0) {
                    // geometric normal of the hit triangle: object space, rotated by the instance
                    // rotation (scale ignored, as the reference does)
                    const BVHVertex *tv = mesh.vertices + (size_t)first.triangle * 3;
                    const Vector3 ta { tv[0].pos[0], tv[0].pos[1], tv[0].pos[2] };
                    const Vector3 tb { tv[1].pos[0], tv[1].pos[1], tv[1].pos[2] };
                    const Vector3 tc { tv[2].pos[0], tv[2].pos[1], tv[2].pos[2] };
                    const Quat iq = inst.rotation;
                    const Vector3 normal = iq.rotateVec(madrona::math::normalize(cross(tb - ta, tc - ta)));

                    // lights (bvh_raycast.cpp:861-919)
                    const Vector3 hit_pos = ray_start + first.t * ray_dir;
                    for (i32 li = 0; li < num_lights; li++) {
                        const RenderLight &l = lights[li];
                        const Vector3 ldir_in = l.direction;
                        Vector3 light_dir = -ldir_in;
                        if (!l.directional) {
                            light_dir = (l.position - hit_pos).normalize();
                            if (l.cutoff != -1.f) {
                                float dd = dot(-light_dir, ldir_in);
                                dd /= (light_dir.length() * ldir_in.length());
                                const float angle = acosf(dd);
                                if (fabsf(angle) > fabsf(l.cutoff)) continue;
                            }
                        }
                        if (l.castShadow) {
                            if (dot(light_dir, normal) > 0.f) {
                                // The reference starts the shadow ray AT the fp32 hit point with tMin 1e-6
                                // (bvh_raycast.cpp:893-901): whether it re-hits its own triangle then
                                // depends on which side of the surface the rounded point fell (measured
                                // here: ~10 % of lit pixels flicker).  Deliberate deviation: the origin is
                                // lifted 1 mm along the surface normal (which faces the light in this branch).
                                const Vector3 so = hit_pos + 0.001f * normal;
                                const RayHit shadow = flat
                                    ? traceFlat<true, false>(R, s_list, mesh_mask, so, light_dir, ray_start - so,
                                                             0.000001f, 10000.f, stack)
                                    : traceWorld<true>(R, tlas, tlas_nodes, instances, so, light_dir, 0.000001f,
                                                       10000.f, stack);
                                if (shadow.instance < 0) {
                                    light_contrib += fminf(fmaxf(dot(normal, light_dir), 0.f), 1.f);
                                }
                            }
                        } else {
                            light_contrib += fminf(fmaxf(dot(normal, light_dir), 0.f), 1.f);
                        }
                    }
                }
                color = fmaxf(0.2f, light_contrib) * base;
                color.x = fminf(1.f, color.x);
                color.y = fminf(1.f, color.y);
                color.z = fminf(1.f, color.z);
            }
            rgb[0] = (unsigned char)(color.x * 255);
            rgb[1] = (unsigned char)(color.y * 255);
            rgb[2] = (unsigned char)(color.z * 255);
            rgb[3] = 255;
        }
    }
}

// ---- host side --------------------------------------------------------------------------------

struct LightCarrierArchetype {
    u32 archetype;
    i32 carrierCol, posCol, dirCol, typeCol, shadowCol, cutoffCol, intensityCol, activeCol;
};

static std::vector<LightCarrierArchetype> &lightCarriers(Executor *ex)
{
    static std::vector<std::pair<Executor *, std::vector<LightCarrierArchetype>>> all;
    for (auto &e : all) {
        if (e.first == ex) return e.second;
    }
    all.emplace_back(ex, std::vector<LightCarrierArchetype>());
    return all.back().second;
}

bool renderHostCreate(Executor *ex, const mb2_render_config *rc, std::string *err)
{
    RenderHost *rh = new RenderHost();
    ex->render = rh;
    memset(&rh->hRender, 0, sizeof(RenderState));
    if (!devAlloc(ex, (void **)&rh->dRender, sizeof(RenderState), false)) {
        *err = "render state allocation failed";
        return false;
    }
    RenderState &R = rh->hRender;
    if (rc && rc->render_resolution > 0) {
        if (!rc->geo_bvh_data.mesh_bvhs || rc->geo_bvh_data.num_bvhs == 0) {
            *err = "CudaBatchRenderConfig::geoBVHData is empty (build it with mb2_build_mesh_bvhs / "
                   "render::AssetProcessor::makeBVHData)";
            return false;
        }
        R.enabled = 1;
        R.resolution = rc->render_resolution;
        R.rgbd = rc->render_mode == 0 ? 1u : 0u;
        R.nearPlane = rc->near_plane;
        R.farPlane = rc->far_plane;
        // device pointers, adopted as they are (the reference frees them in its
        // destructor, cuda_exec.cpp:2449-2485; here their owner is whoever built them)
        R.meshes = (const MeshBVH *)rc->geo_bvh_data.mesh_bvhs;
        R.numMeshes = (u32)rc->geo_bvh_data.num_bvhs;
        R.materials = (const RenderMaterial *)rc->material_data.materials;
        const char *dbg = getenv("MADRONA_B200_RENDER_DEBUG");
        R.debugHits = (dbg && *dbg && *dbg != '0') ? 1u : 0u;
    }
    cudaMemcpy(rh->dRender, &R, sizeof(RenderState), cudaMemcpyHostToDevice);
    ex->hState->render = rh->dRender;
    return true;
}

bool renderHostAfterRegistry(Executor *ex, std::string *err)
{
    RenderHost *rh = ex->render;
    EngineState &S = *ex->hState;
    RenderState dev;
    cudaMemcpy(&dev, rh->dRender, sizeof(RenderState), cudaMemcpyDeviceToHost);
    RenderState &R = rh->hRender;
    R = dev;
    if (!R.registered) return true;
    if (!R.enabled) {
        // RenderingSystem used without a CudaBatchRenderConfig: the reference then
        // simply does not ray cast (raycastOutputResolution == 0)
        return true;
    }
    rh->active = true;

    auto col = [&](u32 a, u32 cid) -> int {
        return cid < S.numComponents ? S.columnLookup[a][cid] : -1;
    };
    for (u32 a = 0; a < S.numArchetypes; a++) {
        if (!S.archetypes[a].registered) continue;
        if (col(a, R.cidRenderable) >= 0 && col(a, R.cidPosition) >= 0 && col(a, R.cidRotation) >= 0 &&
                col(a, R.cidScale) >= 0 && col(a, R.cidObjectID) >= 0) {
            if (R.numRenderArchetypes >= (u32)kMaxRenderArchetypes) {
                *err = "too many renderable archetypes";
                return false;
            }
            RenderArchetype &ra = R.renderables[R.numRenderArchetypes++];
            ra.archetype = a;
            ra.cols[RCPosition] = col(a, R.cidPosition);
            ra.cols[RCRotation] = col(a, R.cidRotation);
            ra.cols[RCScale] = col(a, R.cidScale);
            ra.cols[RCObjectID] = col(a, R.cidObjectID);
            ra.cols[RCRenderable] = col(a, R.cidRenderable);
            ra.colorCol = col(a, R.cidColorOverride);
            ra.matCol = col(a, R.cidMaterialOverride);
        }
        if (col(a, R.cidRenderCamera) >= 0 && col(a, R.cidPosition) >= 0 && col(a, R.cidRotation) >= 0) {
            if (R.numViewArchetypes >= (u32)kMaxRenderArchetypes) {
                *err = "too many viewing archetypes";
                return false;
            }
            ViewArchetype &va = R.viewers[R.numViewArchetypes++];
            va.archetype = a;
            va.posCol = col(a, R.cidPosition);
            va.rotCol = col(a, R.cidRotation);
            va.camCol = col(a, R.cidRenderCamera);
        }
    }
    R.rgbCol = col(R.outputArchetype, R.cidRGB);
    R.depthCol = col(R.outputArchetype, R.cidDepth);
    R.lightCol = col(R.lightArchetype, R.cidLightDesc);
    {
        const char *v = getenv("MADRONA_B200_MAX_INSTANCES_PER_WORLD");
        int cap = (v && *v) ? atoi(v) : 128;
        R.maxInstancesPerWorld = std::min(std::max(cap, 8), 512);
    }
    R.maxViews = S.tables[R.outputArchetype].capacity;
    rh->tlasSmem = tlasScratchBytes(R.maxInstancesPerWorld);
    cudaFuncSetAttribute(renderBuildTLASKernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rh->tlasSmem);

    // light carriers: archetypes with LightCarrier + Position + every LightDesc* component
    // (component ids are consecutive from registration: LightDesc, Direction, Type, Shadow,
    // CutoffAngle, Intensity, Active, LightCarrier)
    {
        auto &carriers = lightCarriers(ex);
        carriers.clear();
        const u32 c0 = R.cidLightDesc;
        for (u32 a = 0; a < S.numArchetypes; a++) {
            if (!S.archetypes[a].registered) continue;
            LightCarrierArchetype lc;
            lc.archetype = a;
            lc.carrierCol = col(a, c0 + 7);
            lc.posCol = col(a, R.cidPosition);
            lc.dirCol = col(a, c0 + 1);
            lc.typeCol = col(a, c0 + 2);
            lc.shadowCol = col(a, c0 + 3);
            lc.cutoffCol = col(a, c0 + 4);
            lc.intensityCol = col(a, c0 + 5);
            lc.activeCol = col(a, c0 + 6);
            if (lc.carrierCol >= 0 && lc.posCol >= 0 && lc.dirCol >= 0 && lc.typeCol >= 0 && lc.shadowCol >= 0 &&
                    lc.cutoffCol >= 0 && lc.intensityCol >= 0 && lc.activeCol >= 0) {
                carriers.push_back(lc);
            }
        }
    }

    const size_t W = S.numWorlds;
    if (!devAlloc(ex, (void **)&R.instances, sizeof(RenderInstance) * W * R.maxInstancesPerWorld) ||
        !devAlloc(ex, (void **)&R.instanceCounts, sizeof(i32) * W) ||
        !devAlloc(ex, (void **)&R.tlasNodes, sizeof(QBVHNode) * W * R.maxInstancesPerWorld) ||
        !devAlloc(ex, (void **)&R.tlasNodeCounts, sizeof(i32) * W) ||
        !devAlloc(ex, (void **)&R.lights, sizeof(RenderLight) * W * kMaxLightsPerWorld) ||
        !devAlloc(ex, (void **)&R.lightCounts, sizeof(i32) * W) ||
        (R.debugHits && !devAlloc(ex, (void **)&R.hitIDs, sizeof(i32) * 2 * (size_t)R.maxViews * R.resolution *
                                                              R.resolution)) ||
        !devAlloc(ex, (void **)&R.views, sizeof(RenderView) * (size_t)R.maxViews)) {
        *err = "render buffers allocation failed";
        return false;
    }
    cudaMemcpy(rh->dRender, &R, sizeof(RenderState), cudaMemcpyHostToDevice);
    return true;
}

void renderHostDestroy(Executor *ex)
{
    delete ex->render;
    ex->render = nullptr;
}

__global__ void renderResetCountsKernel(EngineState *Sp)
{
    Sp->render->totalNumInstances = 0;
}

bool renderEnqueuePrepare(Executor *ex, cudaStream_t s, std::string *err)
{
    RenderHost *rh = ex->render;
    if (!rh || !rh->active) return true;   // rendering not configured: nothing to prepare
    (void)err;
    const RenderState &R = rh->hRender;
    const unsigned W = ex->hState->numWorlds;
    renderResetCountsKernel<<<1, 1, 0, s>>>(ex->dState);
    renderGatherInstancesKernel<<<(W * 32 + 127) / 128, 128, 0, s>>>(ex->dState);
    // lights: carriers refresh their light entities, the light table is brought into
    // world order (no-op when clean), then listed per world
    for (const LightCarrierArchetype &lc : lightCarriers(ex)) {
        const int cap = ex->hState->tables[lc.archetype].capacity;
        renderLightUpdateKernel<<<(unsigned)std::max(1, std::min((cap + 255) / 256, ex->numSMs * 2)), 256, 0, s>>>(
            ex->dState, lc.archetype, lc.carrierCol, lc.posCol, lc.dirCol, lc.typeCol,
            lc.shadowCol, lc.cutoffCol, lc.intensityCol, lc.activeCol);
    }
    launchSortArchetype(ex, R.lightArchetype, 1, s);
    renderGatherLightsKernel<<<(W + 255) / 256, 256, 0, s>>>(ex->dState);
    int max_cap = 256;
    for (u32 i = 0; i < R.numViewArchetypes; i++) {
        max_cap = std::max(max_cap, ex->hState->tables[R.viewers[i].archetype].capacity);
    }
    dim3 grid((unsigned)std::min((max_cap + 255) / 256, ex->numSMs * 4), std::max(R.numViewArchetypes, 1u));
    renderGatherViewsKernel<<<grid, 256, 0, s>>>(ex->dState);
    renderBuildTLASKernel<<<W, 32, rh->tlasSmem, s>>>(ex->dState);
    return true;
}

void *renderDebugHitBuffer(Executor *ex)
{
    RenderHost *rh = ex->render;
    return (rh && rh->active) ? (void *)rh->hRender.hitIDs : nullptr;
}

void *renderDebugBuffer(Executor *ex, int which, int64_t *stride_out)
{
    RenderHost *rh = ex->render;
    if (!rh || !rh->active) return nullptr;
    const RenderState &R = rh->hRender;
    *stride_out = R.maxInstancesPerWorld;
    switch (which) {
    case 1: return R.tlasNodes;
    case 2: return R.tlasNodeCounts;
    case 3: return R.instances;
    case 4: return R.instanceCounts;
    default: return nullptr;
    }
}

LaunchGraph *physicsBuildRenderGraph(Executor *ex, std::string *err)
{
    RenderHost *rh = ex->render;
    if (!rh || !rh->active) {
        *err = "buildRenderGraph: no CudaBatchRenderConfig was given (or the simulator never called "
               "RenderingSystem::registerTypes)";
        return nullptr;
    }
    const RenderState &R = rh->hRender;
    LaunchGraph *g = new LaunchGraph();
    g->owner = ex;
    cudaSetDevice(ex->gpu);
    if (cudaStreamBeginCapture(ex->stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        *err = "cudaStreamBeginCapture failed";
        delete g;
        return nullptr;
    }
    // persistent blocks striding over the views (the output table's capacity can be far above
    // the live view count: one block per capacity row cost 76 us of empty-block scheduling at
    // 1024 worlds); 8 rounds of resident blocks keep the tail short
    const unsigned view_blocks = (unsigned)std::max(1, std::min(R.maxViews, ex->numSMs * MB2_RAYCAST_MINB * 8));
    renderRaycastKernel<true><<<dim3(1, view_blocks), 256, 0, ex->stream>>>(ex->dState);
    renderRaycastKernel<false><<<dim3(1, view_blocks), 256, 0, ex->stream>>>(ex->dState);
    launchStatusCopy(ex, ex->stream);
    cudaError_t e = cudaStreamEndCapture(ex->stream, &g->graph);
    if (e != cudaSuccess || cudaGraphInstantiate(&g->exec, g->graph, 0) != cudaSuccess) {
        *err = std::string("render graph capture failed: ") + cudaGetErrorString(cudaGetLastError());
        if (g->graph) cudaGraphDestroy(g->graph);
        delete g;
        return nullptr;
    }
    g->numKernels = 3;
    return g;
}

// algorithmic bytes of one frame (SURVEY.md 8d): res^2 x 4 B depth (+ 4 B RGBA8) per view
uint64_t renderBytesPerFrame(Executor *ex, int64_t num_views)
{
    RenderHost *rh = ex->render;
    if (!rh || !rh->active) return 0;
    const RenderState &R = rh->hRender;
    return (uint64_t)num_views * R.resolution * R.resolution * (R.rgbd ? 8ull : 4ull);
}

}
