// hrp_graph.cu -- a captured CUDA graph behind a device-side gate (CUDA 12.4+ conditional IF nodes).
//
// hrp_graph_if_create wraps an already-captured graph G as   [gate kernel] -> IF { child graph G }   and instantiates
// it.  The gate reads a 32-bit stop word when the exec runs: the body runs iff *stop == 0, and every opening adds one to
// a device counter.  PPOAgent's target_kl early stopping launches one such exec per replayed minibatch step in place of
// the bare graph, so the steps after the one that raised the word cost one one-thread kernel each instead of a whole
// forward / backward / Adam chain.  The decision is taken on the device: nothing synchronises with the host.
#include "hrp_internal.cuh"

struct hrp_graph_if {
    cudaGraph_t graph;
    cudaGraphExec_t exec;
};

namespace {

__global__ void if_gate_kernel(cudaGraphConditionalHandle handle, const unsigned *__restrict__ stop,
                               unsigned *__restrict__ opened)
{
    const bool open = *stop == 0u;
    cudaGraphSetConditional(handle, open ? 1u : 0u);
    if (open) *opened += 1u;
}

}  // namespace

// a CUDA refusal is reported like a bad argument (-1), with the CUDA error text
#define HRP_GRAPH_OK(expr, what)                                                                  \
    do {                                                                                          \
        cudaError_t _e = (expr);                                                                  \
        if (_e != cudaSuccess) {                                                                  \
            hrp_set_error("hrp_graph_if_create: %s refused: %s", what, cudaGetErrorString(_e));   \
            if (exec) cudaGraphExecDestroy(exec);                                                 \
            if (g) cudaGraphDestroy(g);                                                           \
            return -1;                                                                            \
        }                                                                                         \
    } while (0)

extern "C" {

int hrp_graph_if_create(void *body_graph, const uint32_t *stop_dev, uint32_t *opened_dev, hrp_graph_if **out)
{
    const char *bad = !body_graph ? "body_graph" : !stop_dev ? "stop_dev" : !opened_dev ? "opened_dev" : !out ? "out"
                    : nullptr;
    if (bad) { hrp_set_error("hrp_graph_if_create: bad argument %s", bad); return -1; }
    *out = nullptr;
    cudaGraph_t g = nullptr;
    cudaGraphExec_t exec = nullptr;
    HRP_GRAPH_OK(cudaGraphCreate(&g, 0), "cudaGraphCreate");
    cudaGraphConditionalHandle handle;
    HRP_GRAPH_OK(cudaGraphConditionalHandleCreate(&handle, g, 0u, 0u), "cudaGraphConditionalHandleCreate");
    cudaKernelNodeParams kp = {};
    const unsigned *stop = stop_dev;
    unsigned *opened = opened_dev;
    void *args[] = {&handle, &stop, &opened};
    kp.func = (void *)if_gate_kernel;
    kp.gridDim = dim3(1);
    kp.blockDim = dim3(1);
    kp.kernelParams = args;
    cudaGraphNode_t gate;
    HRP_GRAPH_OK(cudaGraphAddKernelNode(&gate, g, nullptr, 0, &kp), "the gate kernel node");
    cudaGraphNodeParams cp = {};
    cp.type = cudaGraphNodeTypeConditional;
    cp.conditional.handle = handle;
    cp.conditional.type = cudaGraphCondTypeIf;
    cp.conditional.size = 1;
    cudaGraphNode_t cond;
    HRP_GRAPH_OK(cudaGraphAddNode(&cond, g, &gate, 1, &cp), "the IF node");
    cudaGraphNode_t child;
    HRP_GRAPH_OK(cudaGraphAddChildGraphNode(&child, cp.conditional.phGraph_out[0], nullptr, 0, (cudaGraph_t)body_graph),
                 "the body graph inside the IF node");
    HRP_GRAPH_OK(cudaGraphInstantiate(&exec, g, 0), "cudaGraphInstantiate");
    *out = new hrp_graph_if{g, exec};
    return 0;
}

int hrp_graph_if_launch(hrp_graph_if *w, void *stream)
{
    if (!w) { hrp_set_error("hrp_graph_if_launch: bad argument wrapped"); return -1; }
    HRP_CUDA_OK(cudaGraphLaunch(w->exec, (cudaStream_t)stream));
    return 0;
}

int hrp_graph_if_destroy(hrp_graph_if *w)
{
    if (!w) return 0;
    cudaGraphExecDestroy(w->exec);
    cudaGraphDestroy(w->graph);
    delete w;
    return 0;
}

}  // extern "C"
