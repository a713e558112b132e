// graph.cu — CUDA-graph capture / replay of a gradient step, and the per-step scalar block a replay reads.
//
// The reference runs a learn step as a few hundred eager ATen launches (dqn_rainbow.py:369-490); this library
// runs it as ~40 kernels whose dependency chain is what bounds a lone agent's step (DESIGN.md section 5).  Capturing the
// chain once and replaying it removes the per-launch host cost and the inter-kernel launch gaps.  Everything that
// varies between steps lives in one b2rl_step_state on the device, rewritten by the graph's first node.
#include <vector>

#include "common.cuh"

namespace b2rl {

__global__ void step_state_write_kernel(b2rl_step_state v, b2rl_step_state *dst) { *dst = v; }

}  // namespace b2rl

using namespace b2rl;

struct b2rl_graph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    cudaGraphNode_t state_node = nullptr;
    cudaKernelNodeParams state_params{};
    b2rl_step_state *state_dev = nullptr;
    // every step_state_write_kernel node with its destination (the first of them is state_node above)
    std::vector<cudaGraphNode_t> state_nodes;
    std::vector<cudaKernelNodeParams> state_node_params;
    std::vector<b2rl_step_state *> state_dsts;
    int kernels = 0;
};

extern "C" {

int b2rl_step_state_write(const b2rl_step_state *state_host, b2rl_step_state *state_dev, void *stream) {
    B2RL_CHECK_ARG(state_host && state_dev, "NULL step state");
    step_state_write_kernel<<<1, 1, 0, as_stream(stream)>>>(*state_host, state_dev);
    B2RL_LAUNCH_CHECK();
    return B2RL_OK;
}

int b2rl_copy_d2h(void *dst_pinned_host, const void *src, size_t bytes, void *stream) {
    B2RL_CHECK_ARG(dst_pinned_host && src, "NULL argument");
    B2RL_CUDA(cudaMemcpyAsync(dst_pinned_host, src, bytes, cudaMemcpyDeviceToHost, as_stream(stream)));
    return B2RL_OK;
}

int b2rl_graph_begin(void *stream) {
    B2RL_CHECK_ARG(stream != nullptr, "graph capture needs a non-default stream");
    B2RL_CUDA(cudaStreamBeginCapture(as_stream(stream), cudaStreamCaptureModeRelaxed));
    return B2RL_OK;
}

int b2rl_graph_end(void *stream, b2rl_graph **out_host) {
    B2RL_CHECK_ARG(out_host != nullptr, "out_host is NULL");
    cudaGraph_t graph = nullptr;
    B2RL_CUDA(cudaStreamEndCapture(as_stream(stream), &graph));
    B2RL_CHECK_ARG(graph != nullptr, "stream capture was invalidated");
    b2rl_graph *g = new b2rl_graph();
    g->graph = graph;
    size_t n = 0;
    B2RL_CUDA(cudaGraphGetNodes(graph, nullptr, &n));
    std::vector<cudaGraphNode_t> nodes(n);
    if (n) B2RL_CUDA(cudaGraphGetNodes(graph, nodes.data(), &n));
    for (size_t i = 0; i < n; ++i) {
        cudaGraphNodeType t;
        B2RL_CUDA(cudaGraphNodeGetType(nodes[i], &t));
        if (t != cudaGraphNodeTypeKernel) continue;
        ++g->kernels;
        cudaKernelNodeParams p{};
        B2RL_CUDA(cudaGraphKernelNodeGetParams(nodes[i], &p));
        if (p.func != (void *)step_state_write_kernel) continue;
        b2rl_step_state *dst = *reinterpret_cast<b2rl_step_state **>(p.kernelParams[1]);
        g->state_nodes.push_back(nodes[i]);
        g->state_node_params.push_back(p);
        g->state_dsts.push_back(dst);
        if (g->state_node == nullptr) {
            g->state_node = nodes[i];
            g->state_params = p;
            g->state_dev = dst;
        }
    }
    B2RL_CUDA(cudaGraphInstantiate(&g->exec, graph, 0));
    *out_host = g;
    return B2RL_OK;
}

int b2rl_graph_launch(b2rl_graph *g, const b2rl_step_state *state_host, void *stream) {
    B2RL_CHECK_ARG(g && g->exec, "NULL graph");
    if (g->state_node) {
        B2RL_CHECK_ARG(state_host != nullptr, "this graph starts with a step-state write: state_host is required");
        b2rl_step_state v = *state_host;
        b2rl_step_state *dst = g->state_dev;
        void *args[2] = {&v, &dst};
        cudaKernelNodeParams p = g->state_params;
        p.kernelParams = args;
        p.extra = nullptr;
        B2RL_CUDA(cudaGraphExecKernelNodeSetParams(g->exec, g->state_node, &p));
    }
    B2RL_CUDA(cudaGraphLaunch(g->exec, as_stream(stream)));
    g_launches += (unsigned long long)g->kernels;
    return B2RL_OK;
}

int b2rl_graph_launch_states(b2rl_graph *g, const b2rl_step_state *const *states_host, b2rl_step_state *const *states_dev, int n,
                             void *stream) {
    B2RL_CHECK_ARG(g && g->exec, "NULL graph");
    B2RL_CHECK_ARG(n >= 0 && (n == 0 || (states_host && states_dev)), "bad step-state arguments");
    for (int k = 0; k < n; ++k) {
        B2RL_CHECK_ARG(states_host[k] != nullptr, "NULL host step state %d", k);
        size_t j = 0;
        while (j < g->state_dsts.size() && g->state_dsts[j] != states_dev[k]) ++j;
        B2RL_CHECK_ARG(j < g->state_dsts.size(), "no step-state write node of this graph writes state %d", k);
        b2rl_step_state v = *states_host[k];
        b2rl_step_state *dst = g->state_dsts[j];
        void *args[2] = {&v, &dst};
        cudaKernelNodeParams p = g->state_node_params[j];
        p.kernelParams = args;
        p.extra = nullptr;
        B2RL_CUDA(cudaGraphExecKernelNodeSetParams(g->exec, g->state_nodes[j], &p));
    }
    B2RL_CUDA(cudaGraphLaunch(g->exec, as_stream(stream)));
    g_launches += (unsigned long long)g->kernels;
    return B2RL_OK;
}

int b2rl_graph_kernel_count(const b2rl_graph *g, int *out_host) {
    B2RL_CHECK_ARG(g && out_host, "NULL argument");
    *out_host = g->kernels;
    return B2RL_OK;
}

int b2rl_graph_destroy(b2rl_graph *g) {
    if (!g) return B2RL_OK;
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->graph) cudaGraphDestroy(g->graph);
    delete g;
    return B2RL_OK;
}

}  // extern "C"
