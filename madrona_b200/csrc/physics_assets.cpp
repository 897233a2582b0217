// physics_assets.cpp -- host-side physics asset pipeline: convex hull meshes +
// collision object descriptions -> the phys::ObjectManager a simulator's Config
// points at (half-edge meshes, face planes, primitive / object AABBs, mass
// properties with the inertia tensor diagonalised), uploaded to the GPU.
//
// Role of RigidBodyAssets::processRigidBodyAssets (src/physics/
// physics_assets.cpp:1268-1407, with build_convex_hulls = false: the inputs are
// convex polyhedra whose coplanar faces are already merged) followed by
// PhysicsLoader::loadRigidBodies / getObjectManager (src/physics/
// physics_loader.cpp), which copies the arrays to the GPU and hands out the
// ObjectManager.  What is computed follows the reference function by function
// (half-edge numbering :638-748, Newell planes :211-252, tetrahedron covariance
// accumulation :956-1134, McAdams Jacobi diagonalisation :802-954, AABBs
// :1171-1266), so the blob is interchangeable with the reference's;
// tests/test_physics_assets.py compares the two bit for bit.  Quickhull
// (build_convex_hulls = true) is not provided.
#include "../../include/madrona_b200.h"
#include "engine.hpp"
#include "physics_state.h"

#include <cfloat>
#include <cstring>
#include <unordered_map>
#include <vector>

namespace mb2 {

using madrona::math::Vector3;
using madrona::math::Quat;
using madrona::math::Diag3x3;
using madrona::math::Mat3x3;
using madrona::math::Symmetric3x3;
using madrona::math::AABB;
using madrona::geo::HalfEdge;
using madrona::geo::HalfEdgeMesh;
using madrona::geo::Plane;
using madrona::phys::CollisionPrimitive;
using madrona::phys::ObjectManager;
using madrona::phys::RigidBodyMetadata;

namespace {

struct HostHull {
    std::vector<HalfEdge> hedges;
    std::vector<uint32_t> faceBase;
    std::vector<Plane> planes;
    std::vector<Vector3> verts;
};

// RTCD 12.4.2 (physics_assets.cpp:211-252): normal from the projected areas, d through the centroid
Plane newellPlane(const Vector3 *verts, const uint32_t *indices, int64_t n)
{
    Vector3 centroid { 0, 0, 0 };
    Vector3 nrm { 0, 0, 0 };
    int64_t count = 0;
    for (int64_t i = n - 1, j = 0; j < n; i = j, j++) {
        const Vector3 vi = verts[indices[i]];
        const Vector3 vj = verts[indices[j]];
        nrm.x += (vi.y - vj.y) * (vi.z + vj.z);
        nrm.y += (vi.z - vj.z) * (vi.x + vj.x);
        nrm.z += (vi.x - vj.x) * (vi.y + vj.y);
        centroid += vj;
        count += 1;
    }
    centroid /= (float)count;
    nrm = madrona::math::normalize(nrm);
    return Plane { nrm, madrona::math::dot(centroid, nrm) };
}

// buildHalfEdgeMesh (physics_assets.cpp:638-748): an edge gets the next two half-edge
// ids when either direction is first seen; `next` of a half edge whose successor does
// not exist yet is the id that successor is about to get
bool buildHull(const mb2_source_hull &src, HostHull *out, std::string *err)
{
    auto face_verts = [&](uint32_t f) { return src.face_counts ? src.face_counts[f] : 3u; };
    uint32_t num_hedges = 0;
    for (uint32_t f = 0; f < src.num_faces; f++) num_hedges += face_verts(f);
    if (num_hedges % 2 != 0) {
        *err = "hull mesh is not closed (odd number of half edges)";
        return false;
    }
    out->verts.resize(src.num_vertices);
    memcpy(out->verts.data(), src.positions, sizeof(Vector3) * src.num_vertices);
    out->hedges.assign(num_hedges, HalfEdge { 0, 0, 0 });
    out->faceBase.resize(src.num_faces);
    out->planes.resize(src.num_faces);

    std::unordered_map<uint64_t, uint32_t> edge_to_hedge;
    auto edge_id = [](uint32_t a, uint32_t b) { return ((uint64_t)a << 32) | (uint64_t)b; };
    uint32_t assigned = 0;
    const uint32_t *idx = src.indices;
    for (uint32_t f = 0; f < src.num_faces; f++) {
        const uint32_t nv = face_verts(f);
        for (uint32_t k = 0; k < nv; k++) {
            if (idx[k] >= src.num_vertices) {
                *err = "hull index out of range";
                return false;
            }
        }
        out->planes[f] = newellPlane(out->verts.data(), idx, nv);
        for (uint32_t k = 0; k < nv; k++) {
            const uint32_t a = idx[k], b = idx[(k + 1) % nv], c = idx[(k + 2) % nv];
            auto it = edge_to_hedge.find(edge_id(a, b));
            if (it == edge_to_hedge.end()) {
                if (assigned + 2 > num_hedges) {
                    *err = "hull mesh is not a closed 2-manifold";
                    return false;
                }
                it = edge_to_hedge.emplace(edge_id(a, b), assigned).first;
                edge_to_hedge.emplace(edge_id(b, a), assigned + 1);
                assigned += 2;
            }
            const uint32_t hedge = it->second;
            if (k == 0) out->faceBase[f] = hedge;
            auto next_it = edge_to_hedge.find(edge_id(b, c));
            const uint32_t next = next_it == edge_to_hedge.end() ? assigned : next_it->second;
            out->hedges[hedge] = HalfEdge { next, a, f };
        }
        idx += nv;
    }
    if (assigned != num_hedges) {
        *err = "hull mesh is not a closed 2-manifold";
        return false;
    }
    return true;
}

inline float rsqrtApprox(float x)       // include/madrona/math.inl:14-24
{
    uint32_t bits;
    memcpy(&bits, &x, 4);
    bits = 0x5F1FFFF9u - (bits >> 1);
    float y;
    memcpy(&y, &bits, 4);
    return y * (0.703952253f * (2.38924456f - x * y * y));
}

// McAdams et al. 2011, Algorithm 2 (physics_assets.cpp:802-833)
void approxGivens(const Symmetric3x3 &m, float *ch_out, float *sh_out)
{
    constexpr float gamma = 5.82842712474619f;
    constexpr float c_star = 0.9238795325112867f;
    constexpr float s_star = 0.3826834323650898f;
    const float a11 = m.diag[0], a12 = m.off[0], a22 = m.diag[1];
    float ch = 2.f * (a11 - a22);
    float sh = a12;
    const float sh2 = sh * sh;
    if (sh2 < 1e-20f) {
        *ch_out = 1.f;
        *sh_out = 0.f;
        return;
    }
    const float ch2 = ch * ch;
    const bool b = (gamma * sh2) < ch2;
    const float omega = rsqrtApprox(ch2 + sh2);
    *ch_out = b ? (omega * ch) : c_star;
    *sh_out = b ? (omega * sh) : s_star;
}

Symmetric3x3 jacobiConjugation(const Symmetric3x3 &m, float ch, float sh)   // :836-877
{
    const float ch2 = ch * ch, sh2 = sh * sh;
    const float q_scale = ch2 + sh2;
    const float q11 = (ch2 - sh2) / q_scale;
    const float q12 = (-2.f * sh * ch) / q_scale;
    const float q21 = (2.f * sh * ch) / q_scale;
    const float q22 = (ch2 - sh2) / q_scale;
    const float m11 = m.diag.x, m22 = m.diag.y, m33 = m.diag.z;
    const float m12 = m.off.x, m13 = m.off.y, m23 = m.off.z;
    const float m11q11_m12q21 = m11 * q11 + m12 * q21;
    const float m11q12_m12q22 = m11 * q12 + m12 * q22;
    const float m12q11_m22q21 = m12 * q11 + m22 * q21;
    const float m12q12_m22q22 = m12 * q12 + m22 * q22;
    return Symmetric3x3 {
        { q11 * m11q11_m12q21 + q21 * m12q11_m22q21, q12 * m11q12_m12q22 + q22 * m12q12_m22q22, m33 },
        { q12 * m11q11_m12q21 + q22 * m12q11_m22q21, m13 * q11 + m23 * q21, m13 * q12 + m23 * q22 },
    };
}

void diagonalize(const Symmetric3x3 &m, Diag3x3 *out_diag, Quat *out_rot)   // :879-954
{
    Symmetric3x3 cur = m;
    Quat acc { 1, 0, 0, 0 };
    for (int i = 0; i < 8; i++) {
        float ch1, sh1, ch2, sh2, ch3, sh3;
        approxGivens(cur, &ch1, &sh1);
        cur = jacobiConjugation(cur, ch1, sh1);
        std::swap(cur.diag[1], cur.diag[2]);
        std::swap(cur.off[0], cur.off[1]);
        approxGivens(cur, &ch2, &sh2);
        cur = jacobiConjugation(cur, ch2, sh2);
        std::swap(cur.diag[0], cur.diag[2]);
        std::swap(cur.off[0], cur.off[2]);
        approxGivens(cur, &ch3, &sh3);
        cur = jacobiConjugation(cur, ch3, sh3);
        cur = Symmetric3x3 { { cur.diag[2], cur.diag[0], cur.diag[1] }, { cur.off[1], cur.off[2], cur.off[0] } };
        acc = Quat { ch1, 0, 0, sh1 } * Quat { ch2, 0, sh2, 0 } * Quat { ch3, sh3, 0, 0 } * acc;
    }
    const Quat rot = acc.normalize();
    const Mat3x3 q = Mat3x3::fromQuat(rot);
    const float m11 = m.diag.x, m22 = m.diag.y, m33 = m.diag.z;
    const float m12 = m.off.x, m13 = m.off.y, m23 = m.off.z;
    const float q11 = q[0].x, q21 = q[0].y, q31 = q[0].z;
    const float q12 = q[1].x, q22 = q[1].y, q32 = q[1].z;
    const float q13 = q[2].x, q23 = q[2].y, q33 = q[2].z;
    out_diag->d0 = q11 * (m11 * q11 + m12 * q21 + m13 * q31) + q21 * (m12 * q11 + m22 * q21 + m23 * q31) +
                   q31 * (m13 * q11 + m23 * q21 + m33 * q31);
    out_diag->d1 = q12 * (m11 * q12 + m12 * q22 + m13 * q32) + q22 * (m12 * q12 + m22 * q22 + m23 * q32) +
                   q32 * (m13 * q12 + m23 * q22 + m33 * q32);
    out_diag->d2 = q13 * (m11 * q13 + m12 * q23 + m13 * q33) + q23 * (m12 * q13 + m22 * q23 + m23 * q33) +
                   q33 * (m13 * q13 + m23 * q23 + m33 * q33);
    *out_rot = rot;
}

struct MassProps {
    Diag3x3 inertia;
    Vector3 com;
    Quat toDiagonal;
};

// computeMassProperties (physics_assets.cpp:956-1134): covariance of the solid as a sum
// of tetrahedra (origin + fan triangles of every face), moved to the centre of mass,
// turned into the inertia tensor of unit mass and diagonalised
MassProps massProperties(const std::vector<HostHull> &hulls, const mb2_source_object &obj)
{
    const Symmetric3x3 canonical { Vector3 { 1.f / 60.f, 1.f / 60.f, 1.f / 60.f },
                                   Vector3 { 1.f / 120.f, 1.f / 120.f, 1.f / 120.f } };
    Symmetric3x3 C_total { Vector3::zero(), Vector3::zero() };
    float m_total = 0;
    Vector3 x_total = Vector3::zero();
    auto tet = [&](Vector3 e1, Vector3 e2, Vector3 e3) {
        Mat3x3 A { { e1, e2, e3 } };
        const float det_A = A.determinant();
        const Symmetric3x3 C = det_A * Symmetric3x3::AXAT(A, canonical);
        const float volume = 1.f / 6.f * det_A;
        const float m = volume * 1.f;
        const Vector3 x = 0.25f * e1 + 0.25f * e2 + 0.25f * e3;
        const float old_m = m_total;
        m_total += m;
        x_total = (x * m + x_total * old_m) / m_total;
        C_total += C;
    };
    for (uint32_t p = 0; p < obj.num_prims; p++) {
        const mb2_source_prim &prim = obj.prims[p];
        if (prim.type == 1) {
            m_total += 1.f;
            const float r = prim.sphere_radius;
            const float v = 1.f / 5.f * r * r;
            C_total += Symmetric3x3 { Vector3 { v, v, v }, Vector3::zero() };
            continue;
        } else if (prim.type == 4) {
            return MassProps { Diag3x3 { INFINITY, INFINITY, INFINITY }, Vector3::zero(), Quat { 1, 0, 0, 0 } };
        }
        const HostHull &h = hulls[prim.hull_idx];
        for (size_t f = 0; f < h.faceBase.size(); f++) {
            const uint32_t root_idx = h.faceBase[f];
            const HalfEdge root = h.hedges[root_idx];
            const Vector3 v1 = h.verts[root.rootVertex];
            uint32_t cur_idx = root.next;
            while (true) {
                const HalfEdge cur = h.hedges[cur_idx];
                const uint32_t next_idx = cur.next;
                if (next_idx == root_idx) break;
                const HalfEdge next = h.hedges[next_idx];
                tet(v1, h.verts[cur.rootVertex], h.verts[next.rootVertex]);
                cur_idx = next_idx;
            }
        }
    }
    // translate the covariance to the centre of mass (delta = -x_total)
    {
        const Vector3 x = x_total, dx = -x_total;
        const Symmetric3x3 cross_terms {
            2.f * Vector3 { x.x * dx.x, x.y * dx.y, x.z * dx.z },
            Vector3 { x.x * dx.y + x.y * dx.x, x.x * dx.z + x.z * dx.x, x.y * dx.z + x.z * dx.y },
        };
        C_total = C_total + m_total * (cross_terms + Symmetric3x3::vvT(dx));
    }
    const float tr = C_total[0][0] + C_total[1][1] + C_total[2][2];
    Symmetric3x3 inertia = Symmetric3x3 { Vector3 { tr, tr, tr }, Vector3::zero() } - C_total;
    inertia *= 1.f / m_total;
    MassProps out;
    out.com = x_total;
    diagonalize(inertia, &out.inertia, &out.toDiagonal);
    return out;
}

struct Layout {
    size_t offsets[10];
    size_t total;
};

Layout layoutFor(const size_t sizes[10])
{
    // utils::computeBufferOffsets with 64-byte alignment (include/madrona/utils.hpp)
    Layout l;
    size_t cur = 0;
    for (int i = 0; i < 10; i++) {
        cur = (cur + 63) / 64 * 64;
        l.offsets[i] = cur;
        cur += sizes[i];
    }
    l.total = (cur + 63) / 64 * 64;
    return l;
}

}

struct ObjectManagerBundle {
    int gpu = -1;
    std::vector<char> hostBlob;        // arrays, pointers valid on the host
    ObjectManager hostMgr {};
    void *deviceBlob = nullptr;        // arrays + the ObjectManager struct at the end
    void *deviceMgr = nullptr;
    mb2_rigid_body_assets view {};
};

}

using namespace mb2;

extern "C" {

mb2_object_manager *mb2_process_rigid_body_assets(const mb2_source_hull *hulls, uint32_t num_hulls,
                                                  const mb2_source_object *objects, uint32_t num_objects,
                                                  int gpu_id)
{
    std::string err;
    std::vector<HostHull> built(num_hulls);
    for (uint32_t h = 0; h < num_hulls; h++) {
        if (!buildHull(hulls[h], &built[h], &err)) {
            setError("mb2_process_rigid_body_assets: hull " + std::to_string(h) + ": " + err);
            return nullptr;
        }
    }
    size_t n_he = 0, n_faces = 0, n_verts = 0, n_prims = 0;
    for (const HostHull &h : built) {
        n_he += h.hedges.size();
        n_faces += h.faceBase.size();
        n_verts += h.verts.size();
    }
    for (uint32_t o = 0; o < num_objects; o++) {
        n_prims += objects[o].num_prims;
        for (uint32_t p = 0; p < objects[o].num_prims; p++) {
            const mb2_source_prim &prim = objects[o].prims[p];
            if (prim.type != 1 && prim.type != 2 && prim.type != 4) {
                setError("mb2_process_rigid_body_assets: unknown primitive type");
                return nullptr;
            }
            if (prim.type == 2 && prim.hull_idx >= num_hulls) {
                setError("mb2_process_rigid_body_assets: hull index out of range");
                return nullptr;
            }
        }
    }
    // same buffer order as the reference: halfEdges, faceBaseHalfEdges, facePlanes, vertices,
    // primitives, primitiveAABBs, metadatas, objAABBs, primOffsets, primCounts
    const size_t sizes[10] = {
        sizeof(HalfEdge) * n_he, sizeof(uint32_t) * n_faces, sizeof(Plane) * n_faces, sizeof(Vector3) * n_verts,
        sizeof(CollisionPrimitive) * n_prims, sizeof(AABB) * n_prims, sizeof(RigidBodyMetadata) * num_objects,
        sizeof(AABB) * num_objects, sizeof(uint32_t) * num_objects, sizeof(uint32_t) * num_objects,
    };
    const Layout L = layoutFor(sizes);
    ObjectManagerBundle *b = new ObjectManagerBundle();
    b->gpu = gpu_id;
    b->hostBlob.assign(L.total + sizeof(ObjectManager), 0);
    char *base = b->hostBlob.data();
    HalfEdge *he_out = (HalfEdge *)(base + L.offsets[0]);
    uint32_t *fb_out = (uint32_t *)(base + L.offsets[1]);
    Plane *pl_out = (Plane *)(base + L.offsets[2]);
    Vector3 *vt_out = (Vector3 *)(base + L.offsets[3]);
    CollisionPrimitive *prims = (CollisionPrimitive *)(base + L.offsets[4]);
    AABB *prim_aabbs = (AABB *)(base + L.offsets[5]);
    RigidBodyMetadata *metas = (RigidBodyMetadata *)(base + L.offsets[6]);
    AABB *obj_aabbs = (AABB *)(base + L.offsets[7]);
    uint32_t *prim_offsets = (uint32_t *)(base + L.offsets[8]);
    uint32_t *prim_counts = (uint32_t *)(base + L.offsets[9]);

    std::vector<HalfEdgeMesh> meshes(num_hulls);
    size_t he_at = 0, f_at = 0, v_at = 0;
    for (uint32_t h = 0; h < num_hulls; h++) {
        const HostHull &hh = built[h];
        memcpy(he_out + he_at, hh.hedges.data(), sizeof(HalfEdge) * hh.hedges.size());
        memcpy(fb_out + f_at, hh.faceBase.data(), sizeof(uint32_t) * hh.faceBase.size());
        memcpy(pl_out + f_at, hh.planes.data(), sizeof(Plane) * hh.planes.size());
        memcpy(vt_out + v_at, hh.verts.data(), sizeof(Vector3) * hh.verts.size());
        meshes[h] = HalfEdgeMesh { he_out + he_at, fb_out + f_at, pl_out + f_at, vt_out + v_at,
                                   (uint32_t)hh.hedges.size(), (uint32_t)hh.faceBase.size(),
                                   (uint32_t)hh.verts.size() };
        he_at += hh.hedges.size();
        f_at += hh.faceBase.size();
        v_at += hh.verts.size();
    }

    // setupRigidBodyAABBsAndPrimitives (physics_assets.cpp:1214-1266)
    uint32_t prim_at = 0;
    for (uint32_t o = 0; o < num_objects; o++) {
        AABB obj_box = AABB::invalid();
        for (uint32_t p = 0; p < objects[o].num_prims; p++) {
            const mb2_source_prim &src = objects[o].prims[p];
            CollisionPrimitive &out = prims[prim_at + p];
            memset(&out, 0, sizeof(out));
            out.type = (CollisionPrimitive::Type)src.type;
            AABB box;
            if (src.type == 1) {
                out.sphere.radius = src.sphere_radius;
                const float r = src.sphere_radius;
                box = AABB { { -r, -r, -r }, { r, r, r } };
            } else if (src.type == 4) {
                box = AABB { { -FLT_MAX, -FLT_MAX, -FLT_MAX }, { FLT_MAX, FLT_MAX, 0 } };
            } else {
                const HalfEdgeMesh &m = meshes[src.hull_idx];
                box = AABB::point(m.vertices[0]);
                for (uint32_t v = 1; v < m.numVertices; v++) box.expand(m.vertices[v]);
                out.hull.halfEdgeMesh = m;
            }
            prim_aabbs[prim_at + p] = box;
            obj_box = AABB::merge(obj_box, box);
        }
        obj_aabbs[o] = obj_box;
        prim_offsets[o] = prim_at;
        prim_counts[o] = objects[o].num_prims;
        prim_at += objects[o].num_prims;
    }
    // computeRigidBodiesMetadata (:1153-1169) + toMassData (:1136-1151)
    for (uint32_t o = 0; o < num_objects; o++) {
        const MassProps mp = massProperties(built, objects[o]);
        const Diag3x3 inv_inertia = objects[o].inv_mass / mp.inertia;
        metas[o] = RigidBodyMetadata {
            { objects[o].inv_mass, Vector3 { inv_inertia.d0, inv_inertia.d1, inv_inertia.d2 }, mp.com, mp.toDiagonal },
            { objects[o].mu_s, objects[o].mu_d },
        };
    }
    b->view = mb2_rigid_body_assets { he_out, fb_out, pl_out, vt_out, (uint32_t)n_he, (uint32_t)n_faces,
                                      (uint32_t)n_verts, prims, prim_aabbs, metas, obj_aabbs, prim_offsets,
                                      prim_counts, num_hulls, (uint32_t)n_prims, num_objects };
    b->hostMgr = ObjectManager { prims, prim_aabbs, obj_aabbs, prim_offsets, prim_counts, metas };
    memcpy(base + L.total, &b->hostMgr, sizeof(ObjectManager));

    if (gpu_id >= 0) {
        // PhysicsLoader::loadRigidBodies: the same block on the GPU, pointers rebased
        cudaSetDevice(gpu_id);
        if (cudaMalloc(&b->deviceBlob, b->hostBlob.size()) != cudaSuccess) {
            setError("mb2_process_rigid_body_assets: device allocation failed");
            delete b;
            return nullptr;
        }
        std::vector<char> staged = b->hostBlob;
        const ptrdiff_t delta = (char *)b->deviceBlob - base;
        auto rebase = [&](void *p) { return p ? (void *)((char *)p + delta) : nullptr; };
        CollisionPrimitive *sp = (CollisionPrimitive *)(staged.data() + L.offsets[4]);
        for (size_t i = 0; i < n_prims; i++) {
            if (sp[i].type == CollisionPrimitive::Type::Hull) {
                HalfEdgeMesh &m = sp[i].hull.halfEdgeMesh;
                m.halfEdges = (HalfEdge *)rebase(m.halfEdges);
                m.faceBaseHalfEdges = (uint32_t *)rebase(m.faceBaseHalfEdges);
                m.facePlanes = (Plane *)rebase(m.facePlanes);
                m.vertices = (Vector3 *)rebase(m.vertices);
            }
        }
        ObjectManager dm = b->hostMgr;
        dm.collisionPrimitives = (CollisionPrimitive *)rebase(dm.collisionPrimitives);
        dm.primitiveAABBs = (AABB *)rebase(dm.primitiveAABBs);
        dm.rigidBodyAABBs = (AABB *)rebase(dm.rigidBodyAABBs);
        dm.rigidBodyPrimitiveOffsets = (uint32_t *)rebase(dm.rigidBodyPrimitiveOffsets);
        dm.rigidBodyPrimitiveCounts = (uint32_t *)rebase(dm.rigidBodyPrimitiveCounts);
        dm.metadata = (RigidBodyMetadata *)rebase(dm.metadata);
        memcpy(staged.data() + L.total, &dm, sizeof(dm));
        cudaMemcpy(b->deviceBlob, staged.data(), staged.size(), cudaMemcpyHostToDevice);
        b->deviceMgr = (char *)b->deviceBlob + L.total;
    }
    return (mb2_object_manager *)b;
}

void *mb2_object_manager_ptr(const mb2_object_manager *mgr, int device)
{
    const ObjectManagerBundle *b = (const ObjectManagerBundle *)mgr;
    if (!b) return nullptr;
    return device ? b->deviceMgr : (void *)(b->hostBlob.data() + b->hostBlob.size() - sizeof(ObjectManager));
}

void mb2_object_manager_host_assets(const mb2_object_manager *mgr, mb2_rigid_body_assets *out)
{
    const ObjectManagerBundle *b = (const ObjectManagerBundle *)mgr;
    *out = b ? b->view : mb2_rigid_body_assets {};
}

void mb2_object_manager_destroy(mb2_object_manager *mgr)
{
    ObjectManagerBundle *b = (ObjectManagerBundle *)mgr;
    if (!b) return;
    if (b->deviceBlob) {
        cudaSetDevice(b->gpu);
        cudaFree(b->deviceBlob);
    }
    delete b;
}

}
