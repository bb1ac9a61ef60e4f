// Context plumbing shared by the CRN (crn.cu) and FullSubNet (fsn.cu) contexts: device allocation, the create-time
// device check, the per-B graph cache and the packed-weight arena (se_internal.h).
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include "se_internal.h"

namespace se {

int dev_alloc_bytes(std::vector<void*>& allocs, void** out, size_t bytes) {
    void* p = nullptr;
    SE_CUDA_OK(cudaMalloc(&p, bytes));
    SE_CUDA_OK(cudaMemset(p, 0, bytes));
    allocs.push_back(p);
    *out = p;
    return 0;
}

int check_create_device(int device, const char* fn) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        set_error(std::string(fn) + ": no CUDA device (this library has no CPU fallback)");
        return 3;
    }
    SE_REQUIRE(device >= 0 && device < n, std::string(fn) + ": bad device index");
    SE_CUDA_OK(cudaSetDevice(device));
    cudaDeviceProp prop;
    SE_CUDA_OK(cudaGetDeviceProperties(&prop, device));
    SE_REQUIRE(prop.major == 10, std::string(fn) + ": kernels are built for sm_100a (Blackwell B200) only");
    return 0;
}

int replay_graph(std::map<int, cudaGraphExec_t>& graphs, cudaStream_t* own, int B,
                 const std::function<int(cudaStream_t)>& enq, cudaStream_t st) {
    auto it = graphs.find(B);
    if (it == graphs.end()) {
        if (!*own) SE_CUDA_OK(cudaStreamCreateWithFlags(own, cudaStreamNonBlocking));
        cudaGraph_t graph = nullptr;
        SE_CUDA_OK(cudaStreamBeginCapture(*own, cudaStreamCaptureModeThreadLocal));
        const int rc = enq(*own);
        cudaError_t e = cudaStreamEndCapture(*own, &graph);
        if (rc) {
            if (graph) cudaGraphDestroy(graph);
            return 1;
        }
        SE_CUDA_OK(e);
        cudaGraphExec_t exec = nullptr;
        SE_CUDA_OK(cudaGraphInstantiate(&exec, graph, 0));
        SE_CUDA_OK(cudaGraphDestroy(graph));
        it = graphs.emplace(B, exec).first;
    }
    SE_CUDA_OK(cudaGraphLaunch(it->second, st));
    return 0;
}

std::vector<float> WeightArena::pack(const HostParams& hp) const {
    std::vector<float> arena(floats, 0.f);
    for (const PackFn& f : packers) f(hp, arena.data());
    return arena;
}

int WeightArena::allocate(std::vector<void*>& allocs) {
    if (dev_alloc_bytes(allocs, reinterpret_cast<void**>(&w), floats * sizeof(float))) return 1;
    if (half && dev_alloc_bytes(allocs, reinterpret_cast<void**>(&wh), floats * sizeof(__half))) return 1;
    if (dev_alloc_bytes(allocs, reinterpret_cast<void**>(&k), khost.size() * sizeof(int))) return 1;
    SE_CUDA_OK(cudaMemcpy(k, khost.data(), khost.size() * sizeof(int), cudaMemcpyHostToDevice));
    for (const auto& bind : binds)
        if (bind()) return 1;
    return 0;
}

int WeightArena::upload(const float* const* ptrs, int n, cudaStream_t st, const char* fn) {
    SE_REQUIRE(n == (int)params.size(), std::string(fn) + ": wrong number of tensors");
    SE_CUDA_OK(cudaStreamSynchronize(st));
    HostParams hp;
    for (int i = 0; i < n; ++i) {
        SE_REQUIRE(ptrs[i] != nullptr, std::string(fn) + ": null tensor " + params[i].name);
        std::vector<float> v((size_t)params[i].numel());
        SE_CUDA_OK(cudaMemcpy(v.data(), ptrs[i], v.size() * sizeof(float), cudaMemcpyDefault));
        hp.emplace(params[i].name, std::move(v));
    }
    const std::vector<float> arena = pack(hp);
    SE_CUDA_OK(cudaDeviceSynchronize());  // no step may still read the old weights
    SE_CUDA_OK(cudaMemcpy(w, arena.data(), arena.size() * sizeof(float), cudaMemcpyHostToDevice));
    if (half) {  // fp16 copy of the whole arena (same indexing): the fp16 weight operands are read from it
        std::vector<__half> ah(arena.size());
        for (size_t i = 0; i < arena.size(); ++i) ah[i] = __float2half_rn(arena[i]);
        SE_CUDA_OK(cudaMemcpy(wh, ah.data(), ah.size() * sizeof(__half), cudaMemcpyHostToDevice));
    }
    bound = true;
    return 0;
}

}  // namespace se
