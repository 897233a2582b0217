// render_state.h -- layouts shared by the NVRTC-side rendering API
// (device/madrona/render/ecs.hpp) and the ahead-of-time batch ray caster
// (kernels_render.cu).  SURVEY.md 8 rows a13-a15.
#pragma once

#include <madrona/math.hpp>
#include <madrona/ecs.hpp>

#include "mb2_state.h"
#include "render_bvh.h"

namespace madrona::render {

struct RenderCamera {
    Entity cameraEntity;      // the view's RaycastOutputArchetype entity
    float fovScale;
    float zNear;
    math::Vector3 cameraOffset;
};

// == include/madrona/render/ecs.hpp:65-115
struct LightDesc {
    enum Type : bool {
        Directional = true,
        Spotlight = false
    };
    Type type;
    bool castShadow;
    math::Vector3 position;
    math::Vector3 direction;
    float cutoff;
    float intensity;
    bool active;
};

static_assert(sizeof(RenderCamera) == 28, "RenderCamera layout");
static_assert(sizeof(LightDesc) == 40, "LightDesc layout");

}

namespace mb2 {

// == render::InstanceData (include/madrona/render/ecs.hpp:49-63) + the instance's
// world box (TLBVHNode in the reference)
struct RenderInstance {
    madrona::math::Vector3 position;
    madrona::math::Quat rotation;
    madrona::math::Vector3 scale;
    i32 matID;            // MaterialOverride: -1 mesh default, -2 use `color`, else material index
    i32 objectID;
    u32 color;            // 0xRRGGBB (ColorOverride)
    float aabbMin[3];
    float aabbMax[3];
};

// == render::LightDesc (include/madrona/render/ecs.hpp:65-89), unpacked
struct RenderLight {
    u32 directional;      // LightDesc::Type: true = Directional, false = Spotlight
    u32 castShadow;
    madrona::math::Vector3 position;
    madrona::math::Vector3 direction;
    float cutoff;
    float intensity;
    u32 active;
};

constexpr int kMaxLightsPerWorld = 8;

// == render::PerspectiveCameraData (include/madrona/render/ecs.hpp:38-46)
struct RenderView {
    madrona::math::Vector3 position;
    madrona::math::Quat rotation;       // inverse of the viewing entity's rotation
    float xScale;
    float yScale;
    float zNear;
    i32 worldIDX;
    i32 outputRow;        // row of the view's RaycastOutputArchetype entity
};

enum RenderCol : int { RCPosition = 0, RCRotation, RCScale, RCObjectID, RCRenderable, RCCount };

constexpr int kMaxRenderArchetypes = 16;

struct RenderArchetype {
    u32 archetype;
    i32 cols[RCCount];
    i32 colorCol;          // ColorOverride column or -1
    i32 matCol;            // MaterialOverride column or -1
};

struct ViewArchetype {
    u32 archetype;
    i32 posCol, rotCol, camCol;
};

struct RenderState {
    // ---- host config (before registerTypes)
    u32 enabled;
    u32 resolution;
    u32 rgbd;              // 1 = RGB + depth, 0 = depth only
    float nearPlane, farPlane;
    const MeshBVH *meshes;          // device, == CudaBatchRenderConfig::geoBVHData.meshBVHs
    u32 numMeshes;
    const RenderMaterial *materials;   // device, == materialData.materials (may be null)
    u32 debugHits;                  // MADRONA_B200_RENDER_DEBUG: keep (instance, triangle) per pixel

    // ---- written by the device-side RenderingSystem::registerTypes
    u32 registered;
    u32 cidRenderable, cidRenderCamera, cidColorOverride, cidMaterialOverride;
    u32 lightArchetype, cidLightDesc;
    u32 cidPosition, cidRotation, cidScale, cidObjectID;
    u32 outputArchetype;   // RaycastOutputArchetype
    u32 cidRGB, cidDepth;

    // ---- filled by the host after registerTypes
    u32 numRenderArchetypes;
    RenderArchetype renderables[kMaxRenderArchetypes];
    u32 numViewArchetypes;
    ViewArchetype viewers[kMaxRenderArchetypes];
    i32 rgbCol, depthCol;

    RenderInstance *instances;      // [numWorlds][maxInstancesPerWorld], gather order
    i32 *instanceCounts;            // [numWorlds]
    i32 maxInstancesPerWorld;
    QBVHNode *tlasNodes;            // [numWorlds][maxInstancesPerWorld], node 0 = root
    i32 *tlasNodeCounts;            // [numWorlds]
    RenderLight *lights;            // [numWorlds][kMaxLightsPerWorld]
    i32 *lightCounts;               // [numWorlds]
    i32 lightCol;
    RenderView *views;              // [capacity of the output archetype]
    i32 maxViews;
    i32 *hitIDs;                    // debug: [maxViews][res*res][2] = (instance, triangle) or -1
    // exportCountsGPU (src/render/ecs_system.cpp:317-348): totals of the last prepare
    u32 totalNumViews;
    u32 totalNumInstances;
};

}
