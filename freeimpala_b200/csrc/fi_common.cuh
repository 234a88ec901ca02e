// Shared helpers for the freeimpala-b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/fi_learner.h"

namespace fi {

// ---- thread-local error message (fi_last_error) -------------------------------------------
inline std::string& last_error_ref() {
    static thread_local std::string msg;
    return msg;
}
inline int set_error(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    last_error_ref() = buf;
    fprintf(stderr, "[freeimpala_b200][error] %s\n", buf);  // reference style: log and continue
    return code;
}

#define FI_CUDA_OK(expr)                                                                       \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess)                                                                 \
            return ::fi::set_error(FI_ERR_CUDA, "%s failed: %s (%s:%d)", #expr,                \
                                   cudaGetErrorString(_e), __FILE__, __LINE__);                \
    } while (0)

#define FI_CUDA_OK_NULL(expr)                                                                  \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            ::fi::set_error(FI_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                            __FILE__, __LINE__);                                               \
            return nullptr;                                                                    \
        }                                                                                      \
    } while (0)

#define FI_TRY(expr)                  \
    do {                              \
        int _s = (expr);              \
        if (_s < 0) return _s;        \
    } while (0)

// ---- kernel launch accounting (fi_kernel_launch_count) ------------------------------------
inline std::atomic<uint64_t>& launch_counter() {
    static std::atomic<uint64_t> n{0};
    return n;
}
inline void count_launch(uint64_t k = 1) { launch_counter().fetch_add(k, std::memory_order_relaxed); }

inline int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return set_error(FI_ERR_CUDA, "launch of %s failed: %s", what, cudaGetErrorString(e));
    count_launch();
    return FI_OK;
}

// ---- per-kernel device timing (fi_prof_enable / fi_prof_collect) --------------------------
// When enabled, launches are bracketed by two CUDA events on the launching stream and tagged with their algorithmic work
// (bytes or flops), so bench.py can report achieved GB/s / TFLOP/s per kernel from the same steps the headline number comes
// from. CONSECUTIVE launches of the same kernel on the same stream share ONE bracket (its time is divided by the launches in
// it): anything between two kernels -- an event record as much as a one-thread marker kernel -- exposes the launch set-up of
// the next one, which back-to-back launches hide behind the running kernel. Measured on the 213 KB-shared-memory cluster
// GEMMs: 147-158 us in a bracket of their own against 120 us in the ncu launch list (profiles/r2_launches.md) and ~125 us
// implied by the un-instrumented step; inside a bracket of four, three of the four launches run as they do in the real step.
// The bracket is closed lazily, by the next launch that does not extend it (or by fi_prof_collect). Disabled: one relaxed load.
enum WorkUnit { kWorkBytes = 0, kWorkFlops = 1 };
struct ProfRec {
    const char* name;
    double work;
    int unit;
    cudaEvent_t a, b;
    int launches;
};
struct ProfState {
    std::atomic<bool> on{false};
    std::mutex mu;
    std::vector<ProfRec> recs;
    std::vector<cudaEvent_t> pool;
    size_t used = 0;
    // the open bracket (valid while open_bracket)
    bool open_bracket = false;
    cudaStream_t open_stream = nullptr;
    ProfRec open_rec{};
    void close_locked() {   // caller holds mu
        if (!open_bracket) return;
        cudaEventRecord(open_rec.b, open_stream);
        if (open_rec.launches > 0) recs.push_back(open_rec);
        open_bracket = false;
    }
};
inline ProfState& prof() {
    static ProfState s;
    return s;
}
class LaunchScope {
public:
    LaunchScope(const char* name, cudaStream_t st, double work, int unit) : name_(name), st_(st) {
        // A non-sticky error left behind by an earlier runtime call of this thread (seen: "invalid device function" after
        // NCCL's communicator set-up in a 2-GPU process) must not be blamed on the launch that follows: take it out of the
        // last-error slot first, and say so once. Sticky errors (a faulted kernel) survive this and are still reported.
        const cudaError_t stale = cudaGetLastError();
        if (stale != cudaSuccess) {
            static std::atomic<bool> said{false};
            if (!said.exchange(true))
                fprintf(stderr, "[freeimpala_b200] note: cleared a stale CUDA error before launching %s: %s\n", name, cudaGetErrorString(stale));
        }
        ProfState& p = prof();
        if (!p.on.load(std::memory_order_relaxed)) return;
        std::lock_guard<std::mutex> g(p.mu);
        if (p.open_bracket && p.open_stream == st && p.open_rec.unit == unit && strcmp(p.open_rec.name, name) == 0) {
            work_ = work;   // extends the open bracket
            active_ = true;
            return;
        }
        p.close_locked();
        while (p.pool.size() < p.used + 2) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) return;
            p.pool.push_back(e);
        }
        ProfRec r{};
        r.name = name;
        r.work = 0.0;
        r.unit = unit;
        r.a = p.pool[p.used++];
        r.b = p.pool[p.used++];
        r.launches = 0;
        if (cudaEventRecord(r.a, st) != cudaSuccess) return;
        p.open_rec = r;
        p.open_stream = st;
        p.open_bracket = true;
        work_ = work;
        active_ = true;
    }
    void done_external() {  // a scope around work that is not one of this library's kernels (NCCL): timed, not counted
        if (active_) note_launch();
    }
    int done() {  // call right after the <<<>>> launch
        const int rc = check_launch(name_);
        if (active_) note_launch();
        return rc;
    }

private:
    void note_launch() {
        ProfState& p = prof();
        std::lock_guard<std::mutex> g(p.mu);
        if (p.open_bracket) {   // (the bracket this scope opened or extended)
            p.open_rec.launches++;
            p.open_rec.work += work_;
        }
    }
    const char* name_;
    cudaStream_t st_;
    double work_ = 0.0;
    bool active_ = false;
};

// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device property of a kernel: set it once per (kernel, device), safe
// against several player threads (or learners on different devices) reaching the first launch together.
inline int ensure_dynamic_smem(std::atomic<uint64_t>& done_devices, const void* kernel, int bytes) {
    int dev = 0;
    cudaGetDevice(&dev);
    const uint64_t bit = 1ull << (dev & 63);
    if (done_devices.load(std::memory_order_acquire) & bit) return FI_OK;
    static std::mutex mu;
    std::lock_guard<std::mutex> g(mu);
    if (done_devices.load(std::memory_order_relaxed) & bit) return FI_OK;
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) return set_error(FI_ERR_CUDA, "cudaFuncSetAttribute(%d B of shared memory) failed: %s", bytes, cudaGetErrorString(e));
    done_devices.fetch_or(bit, std::memory_order_release);
    return FI_OK;
}

constexpr int kNumSMs = 148;  // B200: 2 dies x 74 SMs; grids are sized in multiples of this

inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// ---- record layout of one 1024-byte trajectory element (DESIGN.md "Record layout") --------
constexpr int kRecWords = 256;
constexpr int kZDim = 162;
constexpr int kXDim = 484;
constexpr int kNumActions = 16;
constexpr int kWMu = 162;
constexpr int kWAction = 178;
constexpr int kWReward = 179;
constexpr int kWDiscount = 180;
constexpr int kWAux = 181;
constexpr int kWLegal = 182;   // uint32 legal-action word (bit j = action j legal); read only with legal_action_mask on
constexpr int kWLength = 183;  // uint32 trajectory length, record 0 only; read only with variable_length on
// L = (W == 0 || W > t) ? t : W for the length word W of a t-record trajectory (fi_learner.h, FI_REC_WORD_LENGTH)
__host__ __device__ __forceinline__ int traj_length(uint32_t w, int t) { return (w == 0u || w > (uint32_t)t) ? t : (int)w; }
constexpr int kWX = 192;
constexpr int kXPerRec = 64;
constexpr int kFarmerMinEntry = (kXDim + kXPerRec - 1) / kXPerRec;   // 8 records carry x: the shortest FarmerLstm trajectory
constexpr int kHid = 512;                    // trunk width (reference main.cpp:17-21)
constexpr int kHead = kNumActions + 1;       // fused policy/value head rows
constexpr int kLstmH = 128;                  // reference main.cpp:16

// ---- programmatic dependent launch -------------------------------------------------------------------------------
// A kernel launched with launch_pdl may become resident while the previous kernel of the stream is still draining; it must
// call pdl_wait() before it reads or writes global memory (the wait returns when that kernel has completed and its memory
// operations are visible). Takes the launch latency of the short kernels between the GEMMs off the step's critical path.
// FI_PDL=0: plain stream serialisation (pdl_wait is then a no-op).
inline bool pdl_enabled() {
    static const bool on = [] { const char* e = getenv("FI_PDL"); return !(e && e[0] == '0'); }();
    return on;
}
#ifdef __CUDACC__
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1u : 0u;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#endif

#ifdef __CUDACC__
// ---- streaming 16-byte global accesses (no L1 allocation: every byte is touched once) ------
__device__ __forceinline__ int4 ld_stream16(const int4* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream16(int4* p, const int4& v) {
    asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
#endif

}  // namespace fi
