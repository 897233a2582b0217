// TaskGraph construction API (reference: include/madrona/taskgraph_builder.hpp
// :22-219; GPU node set src/mw/device/include/madrona/taskgraph.hpp:207-381).
//
// There is no megakernel here.  setupTasks runs once on the device (1 thread)
// and appends mb2::NodeRecords; every ParallelForNode instantiation owns a
// real __global__ kernel (mwGPU::nodeKern<NodeT>) that the host launches as a
// CUDA-graph kernel node.  The host pairs records with kernels through the
// address of mwGPU::nodeMeta<NodeT>, whose mangled name shares the <NodeT>
// encoding with the kernel's.
#pragma once
#include <madrona/fwd.hpp>
#include <madrona/context.hpp>
#include <madrona/custom_context.hpp>

namespace madrona {

struct NodeBase {};

struct TaskGraphNodeID {
    uint32_t id;
};

namespace mwGPU {

template <typename NodeT>
__device__ uint32_t nodeMeta = 0;

template <typename NodeT>
__global__ void __launch_bounds__(256) nodeKern(const mb2::NodeRecord *rec)
{
    NodeT::run(*rec);
}

template <auto K> struct KernelInstantiate { static constexpr int v = 1; };

template <typename C, typename D>
D *contextDataPtr(CustomContext<C, D> *);

template <typename T> struct RemovePtr { using type = T; };
template <typename T> struct RemovePtr<T *> { using type = T; };

}

class TaskGraphBuilder {
public:
    inline TaskGraphBuilder() : taskgraph_id_(0) {}

    template <typename NodeT>
    inline TaskGraphNodeID addToGraph(Span<const TaskGraphNodeID> dependencies)
    {
        return NodeT::addToGraph(*this, dependencies);
    }

    // Append a record; returns its (global) node index.
    inline TaskGraphNodeID pushNode(const mb2::NodeRecord &proto,
                                    Span<const TaskGraphNodeID> dependencies)
    {
        mb2::EngineState &S = mwGPU::engine();
        if (S.numNodes >= (uint32_t)mb2::kMaxNodes) {
            mwGPU::raiseError(mb2::ErrTooManyNodes);
            return { S.numNodes - 1 };
        }
        uint32_t idx = S.numNodes++;
        mb2::NodeRecord &r = S.nodes[idx];
        r = proto;
        r.taskgraph = taskgraph_id_;
        r.numDeps = 0;
        for (CountT i = 0; i < dependencies.size() && i < mb2::kMaxNodeDeps; i++) {
            r.deps[r.numDeps++] = dependencies[i].id;
        }
        return { idx };
    }

    inline uint32_t taskgraphID() const { return taskgraph_id_; }

private:
    uint32_t taskgraph_id_;
friend class TaskGraphManager;
};

class TaskGraphManager {
public:
    inline TaskGraphManager(uint32_t num_taskgraphs) : num_(num_taskgraphs) {}

    template <EnumType EnumT>
    inline TaskGraphBuilder &init(EnumT taskgraph_id) { return init((uint32_t)taskgraph_id); }

    inline TaskGraphBuilder &init(uint32_t taskgraph_id)
    {
        builders_[taskgraph_id].taskgraph_id_ = taskgraph_id;
        return builders_[taskgraph_id];
    }

private:
    TaskGraphBuilder builders_[mb2::kMaxTaskGraphs];
    uint32_t num_;
};

// ---- ParallelFor ----------------------------------------------------------
// One record (and one launch) per archetype matching the component list; the
// kernel grid-strides over the table's live row count read on the device, so
// the captured CUDA graph never needs a host-side size.
template <typename ContextT, auto Fn, int threads_per_invocation,
          int items_per_invocation, typename... ComponentTs>
class CustomParallelForNode : public NodeBase {
public:
    static inline void run(const mb2::NodeRecord &rec)
    {
        runImpl(rec, mwGPU::IntSeq<(int)sizeof...(ComponentTs)> {});
    }

    static inline TaskGraphNodeID addToGraph(
        TaskGraphBuilder &builder, Span<const TaskGraphNodeID> dependencies)
    {
        using Self = CustomParallelForNode;
        static_assert(mwGPU::KernelInstantiate<&mwGPU::nodeKern<Self>>::v == 1);
        static_assert(sizeof...(ComponentTs) <= (size_t)mb2::kMaxNodeCols);

        auto &q = Query<ComponentTs...>::data();
        if (q.resolved == 0) {
            mwGPU::getStateManager()->template resolveQuery<ComponentTs...>(q);
        }

        mb2::NodeRecord rec {};
        rec.kind = mb2::NodeUserParallelFor;
        rec.numCols = (int32_t)sizeof...(ComponentTs);
        rec.userTag = (uint32_t)threads_per_invocation;
        // identity of this instantiation for the host (see header comment)
        unsigned long long meta_addr =
            (unsigned long long)(void *)&mwGPU::nodeMeta<Self>;
        rec.kernelID = (uint32_t)(meta_addr & 0xFFFFFFFFull);
        rec.component = (uint32_t)(meta_addr >> 32);

        TaskGraphNodeID last { 0xFFFFFFFFu };
        Span<const TaskGraphNodeID> deps = dependencies;
        for (int qa = 0; qa < q.numArchetypes; qa++) {
            rec.archetype = (uint32_t)q.archetypes[qa];
            for (int i = 0; i < rec.numCols; i++) rec.cols[i] = q.cols[qa][i];
            last = builder.pushNode(rec, deps);
        }
        if (q.numArchetypes == 0) {
            // nothing matches: keep a no-op record so dependency IDs stay valid
            rec.kind = mb2::NodeResetTmpAlloc;
            rec.userTag = 0xFFFFFFFFu;
            last = builder.pushNode(rec, deps);
        }
        return last;
    }

private:
    template <int... Is>
    static inline void runImpl(const mb2::NodeRecord &rec, mwGPU::IntList<Is...>)
    {
        using DataT = typename mwGPU::RemovePtr<
            decltype(mwGPU::contextDataPtr((ContextT *)nullptr))>::type;
        mb2::EngineState &S = mwGPU::engine();
        const mb2::TableDesc &t = S.tables[rec.archetype];
        const int32_t n = t.numRows;
        const WorldID *world_col = (const WorldID *)t.columns[1];
        const int32_t stride =
            (int32_t)((gridDim.x * blockDim.x) / threads_per_invocation);
        int32_t row =
            (int32_t)((blockIdx.x * blockDim.x + threadIdx.x) / threads_per_invocation);
        for (; row < n; row += stride) {
            WorldID w = world_col[row];
            if (w.idx < 0) continue;   // destroyed row awaiting compaction
            ContextT ctx((DataT *)(S.worldData + (size_t)w.idx * S.worldDataStride),
                         WorkerInit { w });
            Fn(ctx, ((ComponentTs *)t.columns[rec.cols[Is]])[row]...);
        }
    }
};

template <typename ContextT, auto Fn, typename... ComponentTs>
using ParallelForNode = CustomParallelForNode<ContextT, Fn, 1, 1, ComponentTs...>;

// ---- engine-owned nodes: recorded here, executed by ahead-of-time kernels --
namespace mwGPU {
inline TaskGraphNodeID pushBuiltin(TaskGraphBuilder &builder,
                                   Span<const TaskGraphNodeID> deps,
                                   uint32_t kind, uint32_t archetype = 0,
                                   uint32_t component = 0, uint32_t tag = 0)
{
    mb2::NodeRecord rec {};
    rec.kind = kind;
    rec.archetype = archetype;
    rec.component = component;
    rec.userTag = tag;
    return builder.pushNode(rec, deps);
}
}

class ResetTmpAllocNode : public NodeBase {
public:
    static inline TaskGraphNodeID addToGraph(
        TaskGraphBuilder &builder, Span<const TaskGraphNodeID> deps)
    {
        return mwGPU::pushBuiltin(builder, deps, mb2::NodeResetTmpAlloc);
    }
};

template <typename ArchetypeT>
class ClearTmpNode : public NodeBase {
public:
    static inline TaskGraphNodeID addToGraph(
        TaskGraphBuilder &builder, Span<const TaskGraphNodeID> deps)
    {
        return mwGPU::pushBuiltin(builder, deps, mb2::NodeClearTmp,
                                  TypeTracker::typeID<ArchetypeT>());
    }
};

class RecycleEntitiesNode : public NodeBase {
public:
    static inline TaskGraphNodeID addToGraph(
        TaskGraphBuilder &builder, Span<const TaskGraphNodeID> deps)
    {
        return mwGPU::pushBuiltin(builder, deps, mb2::NodeRecycleEntities);
    }
};

class SortArchetypeNodeBase : public NodeBase {
public:
    static inline TaskGraphNodeID addToGraph(
        TaskGraphBuilder &builder, Span<const TaskGraphNodeID> deps,
        uint32_t archetype_id, int32_t component_id)
    {
        return mwGPU::pushBuiltin(builder, deps, mb2::NodeSortArchetype,
                                  archetype_id, (uint32_t)component_id);
    }
};

template <typename ArchetypeT, typename ComponentT>
class SortArchetypeNode : public SortArchetypeNodeBase {
public:
    static inline TaskGraphNodeID addToGraph(
        TaskGraphBuilder &builder, Span<const TaskGraphNodeID> deps)
    {
        return SortArchetypeNodeBase::addToGraph(builder, deps,
            TypeTracker::typeID<ArchetypeT>(), (int32_t)TypeTracker::typeID<ComponentT>());
    }
};

template <typename ArchetypeT>
class CompactArchetypeNode : public NodeBase {
public:
    static inline TaskGraphNodeID addToGraph(
        TaskGraphBuilder &builder, Span<const TaskGraphNodeID> deps)
    {
        return mwGPU::pushBuiltin(builder, deps, mb2::NodeCompactArchetype,
                                  TypeTracker::typeID<ArchetypeT>(), 1u);
    }
};

}
