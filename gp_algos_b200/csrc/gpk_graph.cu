// gpk_graph.cu -- CUDA-graph replay of launch sequences that callers repeat verbatim.
//
// One logLikelihoodWithDerivatives call at n = 8192 is ~400 kernel launches plus ~300 event records / waits on 8 streams, and
// an optimiser (GpPredictor.scala:126-142 -> optimization/Optimization.scala:30-61) repeats exactly that sequence 25-60 times
// with new hyper-parameters; an EP run (EpParameterEstimator.scala:37-67) repeats the same ~450-launch sweep until its stop
// criterion fires.  A sequence is identified by a key (buffers, shape, kernel family) plus the workspace epoch.  The first
// `eager_calls` calls with a key run eagerly (the first one also sizes the arenas and sets kernel attributes), the next is
// stream-captured on the handle's stream -- the fork/join structure over the side streams becomes graph edges -- instantiated
// once and launched, later calls only launch the instantiated graph.  Capturing + instantiating ~400 nodes costs ~25 ms once;
// a replay saves the host ~10 ms of enqueueing and the device 0.2 - 0.9 ms of launch gaps, so `eager_calls` is the caller's
// break-even estimate (rent-or-buy: never more than twice the cost of the better choice).  Values that change between calls travel through device memory, never
// through kernel arguments, so the graph itself is immutable.
//
// Stream priorities matter to the look-ahead factorisation (its serial spine must overtake the bulk updates): every captured
// kernel node gets the priority of the stream it was launched on, and the graph is instantiated with
// cudaGraphInstantiateFlagUseNodePriority (without it all nodes run at the launch stream's priority: 20.1 instead of 17.4 ms
// per evaluation at n = 8192, profiles/r01_graph_check.log).
#include "gpk_internal.cuh"

#include <stdlib.h>

#include <new>
#include <utility>
#include <vector>

struct gpk_capture_log {
    std::vector<std::pair<cudaGraphNode_t, int>> nodes;   // kernel node, priority of the stream it was launched on
};

struct gpk_graph_slot {
    GraphKey key;
    unsigned arena_epoch;
    int calls;               // eager calls seen with this key
    int failed;              // capture was refused once: stay eager
    cudaGraphExec_t exec;    // null until captured
    int kernels;             // kernel nodes per replay (gpk_launch_count)
};

void gpk_capture_note(gpk_handle h) {
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    const cudaGraphNode_t* deps = nullptr;
    size_t nd = 0;
    if (cudaStreamGetCaptureInfo(h->stream, &st, nullptr, nullptr, &deps, &nd) != cudaSuccess) { cudaGetLastError(); return; }
    if (st != cudaStreamCaptureStatusActive || nd != 1) return;   // right after a launch the stream depends on exactly that node
    // stream classes: 0 main (the spine) and the batch-group streams, 1 side (forked GEMMs of a recursion node), 2.. the
    // look-ahead driver's bulk streams
    int cls = 0;
    for (int i = 0; i < GPK_NSIDE; ++i) if (h->stream == h->side[i]) cls = 1;
    for (int i = 0; i < GPK_NPIPE; ++i) if (h->stream == h->pipe[i]) cls = 2 + i;
    int prio = cls == 0 ? h->prio_main : cls == 1 ? h->prio_side : h->prio_pipe;
    static int over[2 + GPK_NPIPE], have = -1;
    if (have < 0) {   // GPK_GRAPH_PRIO="main,side,pipe0,pipe1,pipe2" (tuning aid; the defaults measured best, profiles/r01_graph_sweep.log)
        const char* e = getenv("GPK_GRAPH_PRIO");
        have = e && sscanf(e, "%d,%d,%d,%d,%d", &over[0], &over[1], &over[2], &over[3], &over[4]) == 5;
    }
    if (have) prio = over[cls];
    h->cap->nodes.emplace_back(deps[0], prio);
}

static void slot_drop(gpk_handle h, int slot) {
    gpk_graph_slot* s = h->slots[slot];
    if (!s) return;
    if (s->exec) cudaGraphExecDestroy(s->exec);
    delete s;
    h->slots[slot] = nullptr;
}

void gpk_graph_drop_all(gpk_handle h) {
    if (!h) return;
    for (int i = 0; i < GPK_NSLOTS; ++i) slot_drop(h, i);
}

int gpk_graph_run_impl(gpk_handle h, int slot, const GraphKey& key, int eager_calls, int (*body)(void*), void* ctx, const char* what) {
    gpk_graph_slot* g = h->slots[slot];
    if (!g || memcmp(&g->key, &key, sizeof(GraphKey)) != 0 || g->arena_epoch != h->arena_epoch) {
        slot_drop(h, slot);
        g = new (std::nothrow) gpk_graph_slot();
        if (!g) return gpk_set_error(h, GPK_ENOMEM, "host allocation failed");
        memset(g, 0, sizeof(*g));
        g->key = key;
        g->arena_epoch = h->arena_epoch;
        h->slots[slot] = g;
    }
    if (g->exec) {
        GPK_CUDA(h, cudaGraphLaunch(g->exec, h->stream));
        h->launches += g->kernels;
        return GPK_OK;
    }
    if (h->graph_mode >= 2) eager_calls = 1;                        // gpk_set_graph_mode(h, 2): capture at the first repetition
    if (g->failed || g->calls++ < eager_calls) return body(ctx);   // the first calls with this key: eager
    // second call: record the same launch sequence instead of running it
    gpk_capture_log log;
    const int64_t l0 = h->launches;
    GPK_CUDA(h, cudaStreamBeginCapture(h->stream, cudaStreamCaptureModeThreadLocal));
    h->cap = &log;
    int rc = body(ctx);
    h->cap = nullptr;
    cudaGraph_t graph = nullptr;
    cudaError_t ce = cudaStreamEndCapture(h->stream, &graph);
    const int kernels = (int)(h->launches - l0);
    h->launches = l0;
    if (rc == GPK_OK && ce == cudaSuccess && graph) {
        for (auto& nd : log.nodes) {
            cudaLaunchAttributeValue v;
            memset(&v, 0, sizeof(v));
            v.priority = nd.second;
            if (cudaGraphKernelNodeSetAttribute(nd.first, cudaLaunchAttributePriority, &v) != cudaSuccess) cudaGetLastError();
        }
        ce = cudaGraphInstantiate(&g->exec, graph, cudaGraphInstantiateFlagUseNodePriority);
    }
    if (graph) cudaGraphDestroy(graph);
    if (rc != GPK_OK || ce != cudaSuccess || !g->exec) {
        cudaGetLastError();
        g->exec = nullptr;
        g->failed = 1;
        if (getenv("GPK_GRAPH_DEBUG")) fprintf(stderr, "[gpk] %s: graph capture refused (rc %d, %s): staying eager\n", what, rc, cudaGetErrorString(ce));
        return body(ctx);
    }
    g->kernels = kernels;
    if (getenv("GPK_GRAPH_DEBUG")) {
        int least = 0, greatest = 0;
        cudaDeviceGetStreamPriorityRange(&least, &greatest);
        fprintf(stderr, "[gpk] %s captured: %d kernel nodes (%zu with a priority; handle priorities main %d side %d bulk %d, device "
                "range %d..%d)\n", what, kernels, log.nodes.size(), h->prio_main, h->prio_side, h->prio_pipe, greatest, least);
    }
    GPK_CUDA(h, cudaGraphLaunch(g->exec, h->stream));
    h->launches += g->kernels;
    return GPK_OK;
}
