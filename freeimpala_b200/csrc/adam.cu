// Fused optimiser update over the flat fp32 parameter arena.
//
// Replaces torch::optim::Adam/SGD/AdamW::step as configured by the reference's make_optimizer
// (cmd/libtorch_bench/main.cpp:94-103; defaults torch optim/adam.h:20-25: betas (0.9, 0.999),
// eps 1e-8, weight_decay 0 (AdamW: 1e-2), amsgrad off). libtorch walks 16 tensors with ~8
// elementwise ops each; here one kernel reads p, g, m, v and writes p, m, v once:
// 28 B/param of algorithmic traffic (SGD: 12 B/param), HBM-bound.
// Arithmetic follows libtorch's order: m = b1*m + (1-b1)*g; v = b2*v + (1-b2)*g*g;
// denom = sqrt(v)/sqrt(1-b2^t) + eps; p -= (lr/(1-b1^t)) * m/denom, with the bias
// corrections evaluated in double on the host exactly as libtorch does.
//
// RMSProp follows torch.optim.RMSprop with centered=False and weight_decay=0 (rmsprop_elem has the order of the rounded
// operations). The square average lives in the `v` arena, the momentum buffer in `m`: 20 B/param, 28 B/param with momentum.
//
// Clipping: with a non-null OptExtras::coef (written on the device by grad_norm_clip_kernel, grad_norm.cu) every kind
// multiplies g by grad_scale * *coef before the update. The gradient arena is not written back. With a null coef the
// multiplier is grad_scale itself, so the arithmetic of the kinds that existed before clipping is unchanged bit for bit.
#include <cmath>
#include <cstring>

#include "fi_internal.cuh"

namespace fi {

struct OptScalars {
    float beta1, beta2, one_minus_beta1, one_minus_beta2;  // RMSProp: beta1 = momentum, beta2 = alpha, one_minus_beta2 = 1 - alpha
    float step_size, bc2_sqrt, eps, decay;  // decay = 1 - lr*wd (AdamW), else 1
    float lr, grad_scale;
};

// Optional by-products of the update, so that a learner step needs no copy-engine operation on its stream (copy-engine
// hand-overs jitter by 10-300 us, and with 8 data-parallel ranks every step takes the worst rank's jitter):
//  * snapshot: the updated parameters are also written here (the model store's device snapshot, +4 B/param);
//  * losses_src/dst: block 0 copies the step's four loss sums and the gradient norm (kLossWords doubles) into mapped pinned
//    host memory (zero-copy read-back);
//  * coef: the clip coefficient of grad_norm_clip_kernel, or null (no clipping).
struct OptExtras {
    float* snapshot;
    const double* losses_src;
    double* losses_dst;
    const float* coef;
};

__device__ __forceinline__ void adam_elem(float& p, float g, float& m, float& v, const OptScalars& s, float gs) {
    g *= gs;
    p *= s.decay;
    m = __fadd_rn(__fmul_rn(s.beta1, m), __fmul_rn(s.one_minus_beta1, g));
    v = __fadd_rn(__fmul_rn(s.beta2, v), __fmul_rn(__fmul_rn(s.one_minus_beta2, g), g));
    const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), s.bc2_sqrt), s.eps);
    p = __fsub_rn(p, __fmul_rn(s.step_size, __fdiv_rn(m, denom)));
}

// torch.optim.RMSprop (centered=False, weight_decay=0), every operation rounded once in this order:
//   g = g * gs; sa = alpha*sa + ((1-alpha)*g)*g; avg = sqrt(sa) + eps;
//   momentum: buf = mu*buf + g/avg; p = p - lr*buf      otherwise: p = p - lr*(g/avg)
// (tests/optim_reference.py rmsprop_f32 restates it operation for operation)
template <bool kMomentum>
__device__ __forceinline__ void rmsprop_elem(float& p, float g, float& buf, float& sa, const OptScalars& s, float gs) {
    g *= gs;
    sa = __fadd_rn(__fmul_rn(s.beta2, sa), __fmul_rn(__fmul_rn(s.one_minus_beta2, g), g));
    const float avg = __fadd_rn(__fsqrt_rn(sa), s.eps);
    if constexpr (kMomentum) {
        buf = __fadd_rn(__fmul_rn(s.beta1, buf), __fdiv_rn(g, avg));
        p = __fsub_rn(p, __fmul_rn(s.lr, buf));
    } else {
        p = __fsub_rn(p, __fmul_rn(s.lr, __fdiv_rn(g, avg)));
    }
}

constexpr int kOptThreads = 256;
enum OptKernelKind { kKernSgd = 0, kKernAdam = 1, kKernRms = 2, kKernRmsMomentum = 3 };

template <int kKind>
__device__ __forceinline__ void opt_elem(float& p, float g, float& m, float& v, const OptScalars& s, float gs) {
    if constexpr (kKind == kKernAdam) adam_elem(p, g, m, v, s, gs);
    else if constexpr (kKind == kKernRms) rmsprop_elem<false>(p, g, m, v, s, gs);
    else if constexpr (kKind == kKernRmsMomentum) rmsprop_elem<true>(p, g, m, v, s, gs);
    else p -= s.lr * (g * gs);
}

template <int kKind>
__global__ void __launch_bounds__(kOptThreads)
fused_opt_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                 float* __restrict__ v, size_t n, OptScalars s, OptExtras x) {
    constexpr bool kReadM = kKind == kKernAdam || kKind == kKernRmsMomentum;   // m: Adam's first moment / the momentum buffer
    constexpr bool kReadV = kKind != kKernSgd;                                 // v: Adam's second moment / the square average
    if (x.losses_dst && blockIdx.x == 0 && threadIdx.x < kLossWords) {
        x.losses_dst[threadIdx.x] = x.losses_src[threadIdx.x];
        __threadfence_system();
    }
    const float gs = x.coef ? s.grad_scale * *x.coef : s.grad_scale;
    float4* s4 = reinterpret_cast<float4*>(x.snapshot);
    const size_t n4 = n / 4;
    const size_t stride = (size_t)gridDim.x * kOptThreads;
    float4* p4 = reinterpret_cast<float4*>(p);
    const float4* g4 = reinterpret_cast<const float4*>(g);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);
    for (size_t i = (size_t)blockIdx.x * kOptThreads + threadIdx.x; i < n4; i += stride) {
        float4 pp = p4[i];
        const float4 gg = __ldg(g4 + i);
        float4 mm = {}, vv = {};
        if constexpr (kReadM) mm = m4[i];
        if constexpr (kReadV) vv = v4[i];
        opt_elem<kKind>(pp.x, gg.x, mm.x, vv.x, s, gs);
        opt_elem<kKind>(pp.y, gg.y, mm.y, vv.y, s, gs);
        opt_elem<kKind>(pp.z, gg.z, mm.z, vv.z, s, gs);
        opt_elem<kKind>(pp.w, gg.w, mm.w, vv.w, s, gs);
        if constexpr (kReadM) m4[i] = mm;
        if constexpr (kReadV) v4[i] = vv;
        p4[i] = pp;
        if (s4) s4[i] = pp;
    }
    // tail (n % 4 values), handled by the first threads of block 0
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const size_t i = n4 * 4 + threadIdx.x;
        float pp = p[i], mm = 0.f, vv = 0.f;
        if constexpr (kReadM) mm = m[i];
        if constexpr (kReadV) vv = v[i];
        opt_elem<kKind>(pp, g[i], mm, vv, s, gs);
        if constexpr (kReadM) m[i] = mm;
        if constexpr (kReadV) v[i] = vv;
        p[i] = pp;
        if (x.snapshot) x.snapshot[i] = pp;
    }
}

// Everything a launch of the optimiser kernel needs, by value: shared by the direct launch and by the CUDA-graph path of
// the learner step, which re-parameterises ONE captured kernel node per step (step count -> bias corrections, learning rate,
// snapshot and loss read-back slots) with cudaGraphExecKernelNodeSetParams.
int opt_launch_desc(const OptConfig& o, int64_t step, size_t n, float* p, const float* g, float* m, float* v, float grad_scale,
                    const float* coef, float* snapshot, const double* losses_src, double* losses_dst, OptLaunchDesc* d) {
    if (!p || !g) return set_error(FI_ERR_ARG, "optimiser: null p/g");
    const int opt_kind = o.kind;
    const double lr = o.lr;
    const bool adam = opt_kind == FI_OPT_ADAM || opt_kind == FI_OPT_ADAMW;
    const bool rms = opt_kind == FI_OPT_RMSPROP;
    if (!adam && !rms && opt_kind != FI_OPT_SGD) return set_error(FI_ERR_ARG, "optimiser: unknown kind %d", opt_kind);
    if (adam && (!m || !v)) return set_error(FI_ERR_ARG, "optimiser: Adam needs m and v");
    if (rms && (!v || (o.rms_momentum > 0.0 && !m))) return set_error(FI_ERR_ARG, "optimiser: RMSProp needs the square average (and a momentum buffer)");
    if (adam && step < 1) return set_error(FI_ERR_ARG, "optimiser: step counts from 1");
    if (rms && !(o.rms_alpha > 0.0 && o.rms_alpha < 1.0 && o.rms_eps > 0.0 && std::isfinite(o.rms_eps) && o.rms_momentum >= 0.0 &&
                 o.rms_momentum < 1.0))
        return set_error(FI_ERR_ARG, "optimiser: RMSProp needs 0 < alpha < 1, eps > 0 and 0 <= momentum < 1");
    if (((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v | (uintptr_t)snapshot) & 15)
        return set_error(FI_ERR_ARG, "optimiser: arenas must be 16-byte aligned");
    OptScalars s;
    int kern = kKernSgd;
    if (rms) {
        const bool mom = o.rms_momentum > 0.0;
        kern = mom ? kKernRmsMomentum : kKernRms;
        s.beta1 = (float)o.rms_momentum; s.beta2 = (float)o.rms_alpha;
        s.one_minus_beta1 = 0.f; s.one_minus_beta2 = (float)(1.0 - o.rms_alpha);
        s.step_size = 0.f; s.bc2_sqrt = 1.f;
        s.eps = (float)o.rms_eps;
        s.decay = 1.f;
    } else {
        const double b1 = 0.9, b2 = 0.999, eps = 1e-8;
        const double wd = opt_kind == FI_OPT_ADAMW ? 1e-2 : 0.0;
        if (adam) kern = kKernAdam;
        s.beta1 = (float)b1; s.beta2 = (float)b2;
        s.one_minus_beta1 = (float)(1.0 - b1); s.one_minus_beta2 = (float)(1.0 - b2);
        const double bc1 = 1.0 - std::pow(b1, (double)step), bc2 = 1.0 - std::pow(b2, (double)step);
        s.step_size = adam ? (float)(lr / bc1) : 0.f;
        s.bc2_sqrt = adam ? (float)std::sqrt(bc2) : 1.f;
        s.eps = (float)eps;
        s.decay = (float)(1.0 - lr * wd);
    }
    s.lr = (float)lr;
    s.grad_scale = grad_scale;
    const size_t n4 = n / 4 ? n / 4 : 1;
    size_t blocks = (n4 + kOptThreads - 1) / kOptThreads;
    const size_t cap = (size_t)kNumSMs * 8;  // whole waves of 8 resident CTAs per SM
    if (blocks > cap) blocks = cap;
    static_assert(sizeof(OptScalars) <= sizeof(d->scalars) && sizeof(OptExtras) <= sizeof(d->extras), "OptLaunchDesc storage");
    static const void* const kFuncs[4] = {(const void*)fused_opt_kernel<kKernSgd>, (const void*)fused_opt_kernel<kKernAdam>,
                                          (const void*)fused_opt_kernel<kKernRms>, (const void*)fused_opt_kernel<kKernRmsMomentum>};
    d->func = kFuncs[kern];
    d->grid = (unsigned)blocks;
    d->block = kOptThreads;
    d->p = p; d->g = g; d->m = m; d->v = v; d->n = n;
    memcpy(d->scalars, &s, sizeof(s));
    const OptExtras x{snapshot, losses_src, losses_src ? losses_dst : nullptr, coef};
    memcpy(d->extras, &x, sizeof(x));
    d->args[0] = &d->p; d->args[1] = &d->g; d->args[2] = &d->m; d->args[3] = &d->v; d->args[4] = &d->n;
    d->args[5] = d->scalars; d->args[6] = d->extras;
    // algorithmic traffic: Adam reads p,g,m,v + writes p,m,v = 28 B/param; SGD 12; RMSProp 20 (28 with momentum)
    const double per_param = kern == kKernAdam || kern == kKernRmsMomentum ? 28.0 : kern == kKernRms ? 20.0 : 12.0;
    d->work_bytes = (per_param + (snapshot ? 4.0 : 0.0)) * (double)n;
    return FI_OK;
}

int launch_opt(const OptConfig& o, int64_t step, size_t n, float* p, const float* g, float* m, float* v, float grad_scale,
               cudaStream_t stream, const float* coef, float* snapshot, const double* losses_src, double* losses_dst) {
    if (n == 0) return FI_OK;
    OptLaunchDesc d;
    FI_TRY(opt_launch_desc(o, step, n, p, g, m, v, grad_scale, coef, snapshot, losses_src, losses_dst, &d));
    LaunchScope ls("fused_opt_kernel", stream, d.work_bytes, kWorkBytes);
    const cudaError_t e = cudaLaunchKernel(d.func, dim3(d.grid), dim3(d.block), d.args, 0, stream);
    if (e != cudaSuccess) return set_error(FI_ERR_CUDA, "launch of fused_opt_kernel failed: %s", cudaGetErrorString(e));
    return ls.done();
}

}  // namespace fi

extern "C" int fi_op_adam(int opt_kind, double lr, int64_t step, size_t n, float* p, const float* g, float* m,
                          float* v, float grad_scale, void* stream) {
    if (opt_kind == FI_OPT_RMSPROP) return fi::set_error(FI_ERR_ARG, "fi_op_adam: use fi_op_rmsprop for RMSProp");
    fi::OptConfig o;
    o.kind = opt_kind;
    o.lr = lr;
    return fi::launch_opt(o, step, n, p, g, m, v, grad_scale, (cudaStream_t)stream);
}

extern "C" int fi_op_rmsprop(double lr, double alpha, double eps, double momentum, size_t n, float* p, const float* g,
                             float* square_avg, float* momentum_buf, const float* coef, void* stream) {
    fi::OptConfig o;
    o.kind = FI_OPT_RMSPROP;
    o.lr = lr;
    o.rms_alpha = alpha;
    o.rms_eps = eps;
    o.rms_momentum = momentum;
    return fi::launch_opt(o, 1, n, p, g, momentum > 0.0 ? momentum_buf : nullptr, square_avg, 1.0f, (cudaStream_t)stream, coef);
}
