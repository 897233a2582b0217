// Rendering ECS API for simulator code (reference: include/madrona/render/ecs.hpp
// :10-216, src/render/ecs_system.cpp:486-745).  Same component names and
// RenderingSystem entry points; behind them the engine keeps flat per-world
// instance / view arrays (filled by the render-prepare node) for the batch ray
// caster in csrc/kernels_render.cu instead of the reference's render-entity
// archetypes + three sorts per step.  RenderCamera and LightDesc, which the
// ray caster reads too, are defined in csrc/render_state.h.
#pragma once

#include <madrona/math.hpp>
#include <madrona/taskgraph_builder.hpp>
#include <madrona/components.hpp>
#include <render_state.h>

namespace madrona::render {

struct Renderable {
    Entity renderEntity;      // none() => not drawn
};

struct LightCarrier {
    Entity light;
};

struct LightDescDirection : math::Vector3 {
    LightDescDirection(math::Vector3 v) : Vector3(v) {}
};
struct LightDescType { LightDesc::Type type; };
struct LightDescShadow { bool castShadow; };
struct LightDescCutoffAngle { float cutoff; };
struct LightDescIntensity { float intensity; };
struct LightDescActive { bool active; };

struct LightArchetype : public Archetype<LightDesc> {};

struct MaterialOverride {
    enum {
        UseDefaultMaterial = -1,
        UseOverrideColor = -2
    };
    int32_t matID;
};

struct ColorOverride {
    uint32_t color;
};

struct RenderOutputBuffer {
    char buffer[1];
};

struct RGBOutputBuffer : RenderOutputBuffer {};
struct DepthOutputBuffer : RenderOutputBuffer {};

struct RaycastOutputArchetype : public Archetype<
    RGBOutputBuffer,
    DepthOutputBuffer
> {};

struct RenderECSBridge;

namespace RenderingSystem {

inline void registerTypes(ECSRegistry &registry, const RenderECSBridge *)
{
    mb2::RenderState &R = *mwGPU::engine().render;
    registry.registerComponent<RenderCamera>();
    registry.registerComponent<Renderable>();
    registry.registerComponent<MaterialOverride>();
    registry.registerComponent<ColorOverride>();
    registry.registerComponent<LightDesc>();
    registry.registerComponent<LightDescDirection>();
    registry.registerComponent<LightDescType>();
    registry.registerComponent<LightDescShadow>();
    registry.registerComponent<LightDescCutoffAngle>();
    registry.registerComponent<LightDescIntensity>();
    registry.registerComponent<LightDescActive>();
    registry.registerComponent<LightCarrier>();

    // one output row per view: res x res RGBA8 and res x res f32 depth
    // (src/render/ecs_system.cpp: registerComponent<...OutputBuffer>(bytes))
    uint32_t pixels = R.resolution * R.resolution;
    uint32_t bytes = pixels * 4u;
    if (bytes == 0) bytes = 4;
    registry.registerComponent<RGBOutputBuffer>(bytes);
    registry.registerComponent<DepthOutputBuffer>(bytes);
    registry.registerArchetype<RaycastOutputArchetype>();
    registry.registerArchetype<LightArchetype>();

    R.cidMaterialOverride = TypeTracker::typeID<MaterialOverride>();
    R.lightArchetype = TypeTracker::typeID<LightArchetype>();
    R.cidLightDesc = TypeTracker::typeID<LightDesc>();
    R.cidRenderable = TypeTracker::typeID<Renderable>();
    R.cidRenderCamera = TypeTracker::typeID<RenderCamera>();
    R.cidColorOverride = TypeTracker::typeID<ColorOverride>();
    R.cidPosition = TypeTracker::typeID<base::Position>();
    R.cidRotation = TypeTracker::typeID<base::Rotation>();
    R.cidScale = TypeTracker::typeID<base::Scale>();
    R.cidObjectID = TypeTracker::typeID<base::ObjectID>();
    R.outputArchetype = TypeTracker::typeID<RaycastOutputArchetype>();
    R.cidRGB = TypeTracker::typeID<RGBOutputBuffer>();
    R.cidDepth = TypeTracker::typeID<DepthOutputBuffer>();
    R.registered = 1;
}

inline void init(Context &, const RenderECSBridge *) {}

inline void makeEntityRenderable(Context &ctx, Entity e)
{
    ctx.get<Renderable>(e).renderEntity = e;
}

inline void disableEntityRenderable(Context &ctx, Entity e)
{
    ctx.get<Renderable>(e).renderEntity = Entity::none();
}

inline void attachEntityToView(Context &ctx, Entity e, float vfov_degrees,
                               float z_near, const math::Vector3 &camera_offset)
{
    float fov_scale = 1.0f / tanf(math::toRadians(vfov_degrees * 0.5f));
    Entity out = ctx.makeEntity<RaycastOutputArchetype>();
    ctx.get<RenderCamera>(e) = RenderCamera { out, fov_scale, z_near, camera_offset };
}

inline void cleanupViewingEntity(Context &ctx, Entity e)
{
    Entity out = ctx.get<RenderCamera>(e).cameraEntity;
    ctx.destroyEntity(out);
}

inline void cleanupRenderableEntity(Context &ctx, Entity e)
{
    ctx.get<Renderable>(e).renderEntity = Entity::none();
}

// src/render/ecs_system.cpp:713-727: the light entity takes its description from
// the carrier's LightDesc* components; the prepare node refreshes position /
// direction / state from the carrier every step (lightUpdate, :183-209)
inline void makeEntityLightCarrier(Context &ctx, Entity e)
{
    Entity light_e = ctx.makeEntity<LightArchetype>();
    ctx.get<LightCarrier>(e).light = light_e;
    LightDesc desc;
    desc.type = ctx.get<LightDescType>(e).type;
    desc.castShadow = ctx.get<LightDescShadow>(e).castShadow;
    desc.position = ctx.get<base::Position>(e);
    desc.direction = ctx.get<LightDescDirection>(e);
    desc.cutoff = ctx.get<LightDescCutoffAngle>(e).cutoff;
    desc.intensity = ctx.get<LightDescIntensity>(e).intensity;
    desc.active = ctx.get<LightDescActive>(e).active;
    ctx.get<LightDesc>(light_e) = desc;
}

// Per step: gather instance transforms / world boxes and camera data for the
// ray caster (reference: instanceTransformUpdate, viewTransformUpdate,
// mortonCodeUpdate + 3 sorts, ecs_system.cpp:100-159, 275-314, 486-597).
inline TaskGraphNodeID setupTasks(TaskGraphBuilder &builder,
                                  Span<const TaskGraphNodeID> deps,
                                  bool = false)
{
    return mwGPU::pushBuiltin(builder, deps, mb2::NodeRenderPrepare);
}

}

}
