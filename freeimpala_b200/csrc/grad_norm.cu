// Global L2 norm of the flat gradient arena and the clip coefficient of torch.nn.utils.clip_grad_norm_:
//   norm = ||g||_2, coef = min(1, max_norm / (norm + 1e-6)),
// both left in device memory for the optimiser kernel (OptExtras::coef) and the loss read-back (the norm is the fifth
// device loss slot of the learner). One launch, no host synchronisation, no copy-engine operation, so it sits inside the
// step's CUDA graph between the gradient all-reduce and the optimiser.
//
// Squares and sums are formed in double: an fp32 gradient up to 3.4e38 squares to 1.2e77 and 2^26 of those sum far below
// the double range, and values down to 1e-20 keep their squares as normal doubles.
//
// Deterministic: the grid depends on n only, every thread walks its elements in a fixed order, the block reduction has
// a fixed shape, and the last block to finish (a ticket counter) adds the block partials in index order. That block
// also puts the ticket back to zero, so the same launch replays in a graph without a reset in between.
// Algorithmic traffic: 4 B per parameter.
#include <cmath>
#include <map>
#include <mutex>
#include <utility>

#include "fi_internal.cuh"

namespace fi {

constexpr int kNormThreads = 256;
constexpr int kNormMaxBlocks = kNumSMs * 8;   // 8 resident CTAs of 256 threads per SM

struct NormScratch {
    double partial[kNormMaxBlocks];
    unsigned int ticket;
};

__device__ __forceinline__ double block_sum(double v, double* sh) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum(v);
    if (lane == 0) sh[warp] = v;
    __syncthreads();
    v = 0.0;
    if (warp == 0) {
        v = lane < kNormThreads / 32 ? sh[lane] : 0.0;
        v = warp_sum(v);
    }
    return v;   // valid in thread 0
}

__device__ __forceinline__ double sq4(double acc, float4 v) {
    acc = fma((double)v.x, (double)v.x, acc);
    acc = fma((double)v.y, (double)v.y, acc);
    acc = fma((double)v.z, (double)v.z, acc);
    return fma((double)v.w, (double)v.w, acc);
}

__global__ void __launch_bounds__(kNormThreads)
grad_norm_clip_kernel(const float* __restrict__ g, size_t n, double max_norm, double* __restrict__ norm,
                      float* __restrict__ coef, NormScratch* __restrict__ ws) {
    __shared__ double sh[kNormThreads / 32];
    __shared__ bool last;
    const size_t n4 = n / 4, stride = (size_t)gridDim.x * kNormThreads;
    const float4* g4 = reinterpret_cast<const float4*>(g);
    double acc = 0.0;
    size_t i = (size_t)blockIdx.x * kNormThreads + threadIdx.x;
    for (; i + 3 * stride < n4; i += 4 * stride) {   // four 16-byte loads in flight per thread
        const float4 a = __ldg(g4 + i), b = __ldg(g4 + i + stride), c = __ldg(g4 + i + 2 * stride), d = __ldg(g4 + i + 3 * stride);
        acc = sq4(sq4(sq4(sq4(acc, a), b), c), d);
    }
    for (; i < n4; i += stride) acc = sq4(acc, __ldg(g4 + i));
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {   // tail (n % 4 values)
        const double x = g[n4 * 4 + threadIdx.x];
        acc = fma(x, x, acc);
    }
    acc = block_sum(acc, sh);
    if (threadIdx.x == 0) {
        ws->partial[blockIdx.x] = acc;
        __threadfence();
        last = atomicAdd(&ws->ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    double t = 0.0;
    for (unsigned b = threadIdx.x; b < gridDim.x; b += kNormThreads) t += __ldcg(ws->partial + b);   // L2: written by other SMs
    __syncthreads();   // sh is reused
    t = block_sum(t, sh);
    if (threadIdx.x == 0) {
        const double nr = sqrt(t);
        const double c = max_norm / (nr + 1e-6);
        *norm = nr;
        *coef = (float)(c < 1.0 ? c : 1.0);
        ws->ticket = 0u;   // ready for the next launch (graph replay)
    }
}

size_t grad_norm_scratch_bytes() { return sizeof(NormScratch); }

int launch_grad_norm_clip(size_t n, const float* g, double max_norm, double* norm, float* coef, void* scratch, cudaStream_t stream) {
    if (!g || !norm || !coef || !scratch || n == 0) return set_error(FI_ERR_ARG, "grad_norm_clip: null argument or n = 0");
    if ((uintptr_t)g & 15) return set_error(FI_ERR_ARG, "grad_norm_clip: the gradient must be 16-byte aligned");
    if (!(max_norm > 0.0) || !std::isfinite(max_norm)) return set_error(FI_ERR_ARG, "grad_norm_clip: max_norm must be positive and finite");
    const size_t n4 = n / 4 ? n / 4 : 1;
    size_t blocks = (n4 + kNormThreads - 1) / kNormThreads;
    if (blocks > (size_t)kNormMaxBlocks) blocks = kNormMaxBlocks;
    LaunchScope ls("grad_norm_clip_kernel", stream, 4.0 * (double)n, kWorkBytes);
    grad_norm_clip_kernel<<<(unsigned)blocks, kNormThreads, 0, stream>>>(g, n, max_norm, norm, coef, (NormScratch*)scratch);
    return ls.done();
}

}  // namespace fi

namespace {
// Scratch of the operator-layer entry point: one per (device, stream), allocated and zeroed on the first call on that stream and
// kept. Launches on one stream are serialised, and the kernel hands the ticket back at zero, so no call needs a memset;
// concurrent streams never share a ticket.
int op_scratch(cudaStream_t st, void** out) {
    static std::mutex mu;
    static std::map<std::pair<int, cudaStream_t>, void*> cache;
    int dev = 0;
    FI_CUDA_OK(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> g(mu);
    auto it = cache.find({dev, st});
    if (it != cache.end()) {
        *out = it->second;
        return FI_OK;
    }
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    FI_CUDA_OK(cudaStreamIsCapturing(st, &cs));
    if (cs != cudaStreamCaptureStatusNone)
        return fi::set_error(FI_ERR_STATE, "fi_op_grad_norm_clip: the first call on a stream allocates its scratch and cannot be captured");
    void* ws = nullptr;
    FI_CUDA_OK(cudaMalloc(&ws, fi::grad_norm_scratch_bytes()));
    FI_CUDA_OK(cudaMemset(ws, 0, fi::grad_norm_scratch_bytes()));
    FI_CUDA_OK(cudaDeviceSynchronize());
    cache[{dev, st}] = ws;
    *out = ws;
    return FI_OK;
}
}  // namespace

extern "C" int fi_op_grad_norm_clip(size_t n, const float* g, double max_norm, double* norm, float* coef, void* stream) {
    void* ws = nullptr;
    FI_TRY(op_scratch((cudaStream_t)stream, &ws));
    return fi::launch_grad_norm_clip(n, g, max_norm, norm, coef, ws, (cudaStream_t)stream);
}
