// FarmerLstmModel learner step: the numerics the reference defines in
// cmd/libtorch_bench/main.cpp:14-42 (model), :105-114 (criterion), :117-135 (train_step):
//   lstm(z)[B,T,162 -> 128] -> h_{T-1} -> cat with x[B,484] -> 5 x (Linear + ReLU) -> Linear -> y[B,1]
//   loss = mse / l1 / smooth_l1 (mean over the batch), backward through the dense stack and BPTT.
// PyTorch LSTM conventions (SURVEY.md 8c): gate row blocks i,f,g,o of the [4H, .] weights,
// c' = f*c + i*g, h' = o*tanh(c'), h0 = c0 = 0, two bias vectors (both trainable).
//
// Layout: z is read straight out of the gathered batch (row (b,t) = record t of slot b, stride
// 256 words); the input projection of all B*T rows is ONE GEMM; the recurrence runs in a
// kernel that owns R batch rows per CTA for all T steps (rows are independent, so no inter-CTA
// synchronisation); BPTT mirrors it and leaves the pre-activation gate gradients in place of
// the gates, so dW_ih, dW_hh and the bias gradients are again single GEMMs / column sums.
#include <cuda_fp16.h>

#include "learner.cuh"

namespace fi {

constexpr int kG4 = 4 * kLstmH;          // 512 gate columns
constexpr int kFeat = kLstmH + kXDim;    // 612 = cat(h_last, x)
constexpr int kLstmRows = 8;             // batch rows per CTA in the recurrent kernels
constexpr int kLstmThreads = 256;

struct FarmerWs {
    float* gates = nullptr;   // [rows*T, 512]: x-projection -> post-activation gates -> gate gradients
    float* hprev = nullptr;   // [rows*T, 128]: h_{t-1} (0 at t = 0)
    float* cst = nullptr;     // [rows*T, 128]: c_t
    float* whh_t = nullptr;   // [128, 512]: W_hh transposed (coalesced reads in the forward recurrence)
    float* feat = nullptr;    // [rows, 612]
    float* h_last = nullptr;  // inference: [states, 612], h_{T-1} of each state in columns 0..127 (the recurrence writes kFeat-wide rows)
    float* y = nullptr;       // [rows]
    float* dy = nullptr;      // [rows]
    float* target = nullptr;  // [rows]
    void* gemm_ws = nullptr; size_t gemm_ws_bytes = 0;
    void* colsum_ws = nullptr; size_t colsum_ws_bytes = 0;
    size_t states = 0, rows = 0, t = 0;   // rows of the recurrence, rows of the dense stack (equal when training), steps
    // tensor-core path of the three [rows*T]-sized products (input projection and the two LSTM weight gradients): 3xFP16
    // operand pairs (gemm_tc.cu), each big operand split ONCE per step — the observations serve the projection and the
    // W_ih gradient, the gate gradients serve both weight gradients
    bool half = false;
    HScale* hs = nullptr;                          // [4]: observations, W_ih, gate gradients, h_prev
    void *obs_hi = nullptr, *obs_lo = nullptr;     // [rows*T, 192] fp16
    void *wih_hi = nullptr, *wih_lo = nullptr;     // [512, 192]
    void *dg_hi = nullptr, *dg_lo = nullptr;       // [rows*T, 512]
    void *hp_hi = nullptr, *hp_lo = nullptr;       // [rows*T, 128]
    void* split_ws = nullptr; size_t split_ws_bytes = 0;
    float* bias_part = nullptr;                    // [CTAs of the BPTT kernel, 512]: their column sums of dG (the LSTM bias gradient)
    float* dfeat = nullptr;                        // [rows, 128]: dL/dh_{T-1} from the split-operand dense stack (the x part of the
                                                   // feature row needs no gradient)
    // history_length (training): each slot's history is its first L records (word 183 of record 0). The plain-fp32 projection
    // and W_ih gradient read z from this zero-padded copy [rows*T, kObsLd] instead of the batch (allocated when the learner's
    // GEMM mode can take that path); the 3xFP16 path splits padding rows as zeros itself.
    bool history = false;
    float* zpad = nullptr;
};
constexpr int kFeatLdH = 640;   // 612 feature columns padded to whole 128-byte lines of fp16
enum { kLstmHsObs = 0, kLstmHsWih = 1, kLstmHsDg = 2, kLstmHsHp = 3 };   // FarmerWs::hs slots

// Branch-free gate functions for the recurrent kernels. The library expf / tanhf / IEEE division carry range checks and
// (tanhf) a data-dependent branch that a warp of 32 different pre-activations takes both ways; the element-wise part of a
// step is a chain of five of them per (row, unit) pair and was 3100 clocks of a 9500-clock step (clock64 trace).
//   e^x: ex2.approx of x * log2(e) with the rounding error of that product (and of the constant) fed back as a first-order
//        correction: ~2 ulp, the error class of expf itself;
//   sigmoid: one approximate reciprocal (1 ulp);
//   tanh: |x| >= 0.25: 1 - 2 / (e^{2|x|} + 1) (absolute error ~1e-7, i.e. <= 5e-7 relative there);
//         |x| <  0.25: odd Taylor polynomial to x^9 (next term < 1e-8 relative).
__device__ __forceinline__ float fast_exp(float x) {
    const float t = x * 1.44269502f;
    const float r = fmaf(x, 1.44269502f, -t) + x * 1.925963033e-8f;
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(t));
    return e * fmaf(r, 0.693147182f, 1.f);   // (not e + e * r ln 2: e may be +inf)
}
__device__ __forceinline__ float sigmoidf_(float x) { return __fdividef(1.f, 1.f + fast_exp(-x)); }
__device__ __forceinline__ float fast_tanh(float x) {
    const float ax = fabsf(x), x2 = ax * ax;
    const float big = 1.f - __fdividef(2.f, fast_exp(2.f * ax) + 1.f);
    const float poly = fmaf(x2, fmaf(x2, fmaf(x2, 0.0218694885f, -0.0539682540f), 0.133333333f), -0.333333333f);
    const float small = fmaf(ax * x2, poly, ax);
    return copysignf(ax < 0.25f ? small : big, x);
}

// Two fp32 FMAs in one instruction (sm_100 FFMA2; bit-identical to two fmaf's). With b = {w, w} ptxas emits the scalar-broadcast
// form (FFMA2 Rd, Ra.F32x2, Rb.F32, Rc.F32x2), so a row pair of the recurrent products costs one issue slot instead of two.
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
    float2 d;
    asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
        "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
        : "=f"(d.x), "=f"(d.y)
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
    return d;
}

__device__ __forceinline__ void lstm_trace_ev(unsigned long long* tr, int s, int point) {   // FI_LSTM_TRACE (fi_internal.cuh)
#if FI_TRACE_BUILD
    if (tr && s < 128) tr[s * 12 + point] = clock64();
#else
    (void)tr; (void)s; (void)point;
#endif
}

// out[k][j] = in[j][k] for the [512,128] recurrent weight
__global__ void transpose_whh_kernel(const float* __restrict__ w, float* __restrict__ wt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < kG4 * kLstmH) {
        const int j = i / kLstmH, k = i % kLstmH;
        wt[k * kG4 + j] = w[i];
    }
}

// feat[b, 128 + j] = x_j (64 words of x in each of the first 8 records), target[b] = aux of record 0
__global__ void farmer_assemble_kernel(const float* __restrict__ batch, int m, int t, float* __restrict__ feat,
                                       float* __restrict__ target) {
    pdl_wait();
    const int b = blockIdx.x;
    const float* slot = batch + (size_t)b * t * kRecWords;
    for (int j = threadIdx.x; j < kXDim; j += blockDim.x) {
        const int rec = j / kXPerRec, off = j % kXPerRec;
        feat[(size_t)b * kFeat + kLstmH + j] = rec < t ? __ldg(slot + (size_t)rec * kRecWords + kWX + off) : 0.f;
    }
    if (threadIdx.x == 0) target[b] = __ldg(slot + kWAux);
}
// Inference: feat[r] = h_last[state[r], 0..127] ‖ x[r] for candidate rows r < rows. A feature row is 153 float4 (32 of h, 121
// of x; every row of the three arrays starts on a 16-byte boundary), one float4 per thread.
constexpr int kFeat4 = kFeat / 4, kH4 = kLstmH / 4, kX4 = kXDim / 4;
static_assert(kFeat % 4 == 0 && kLstmH % 4 == 0 && kXDim % 4 == 0, "16-byte rows");

__global__ void farmer_assemble_grouped_kernel(const float4* __restrict__ h_last, const float4* __restrict__ x,
                                               const uint32_t* __restrict__ state, int rows, float4* __restrict__ feat) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * kFeat4) return;
    const int r = i / kFeat4, c = i - r * kFeat4;
    feat[i] = c < kH4 ? __ldg(h_last + (size_t)__ldg(state + r) * kFeat4 + c) : __ldg(x + (size_t)r * kX4 + (c - kH4));
}

// best[s] = the index within group s (rows offsets[s] .. offsets[s+1]-1 of y) of its largest value, in numpy's argmax order:
// NaN above every number, then the larger value, then the lower index. One warp per group: each lane scans every 32nd row in
// ascending order, then a butterfly reduction on (value, index); the result does not depend on the group's size or on timing.
__device__ __forceinline__ bool argmax_before(float v, int i, float bv, int bi) {
    const bool vn = v != v, bn = bv != bv;
    if (vn != bn) return vn;
    return (!vn && v > bv) || ((vn || v == bv) && i < bi);
}

__global__ void segment_argmax_kernel(const float* __restrict__ y, const uint32_t* __restrict__ offsets, int states,
                                      int32_t* __restrict__ best) {
    const int s = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32, lane = threadIdx.x & 31;
    if (s >= states) return;
    const int r0 = (int)__ldg(offsets + s), n = (int)__ldg(offsets + s + 1) - r0;
    float bv = -INFINITY;
    int bi = INT_MAX;   // a lane without rows loses to any row (every group has one)
    for (int i = lane; i < n; i += 32) {
        const float v = __ldg(y + r0 + i);
        if (argmax_before(v, i, bv, bi)) { bv = v; bi = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
        if (argmax_before(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) best[s] = bi;
}

// Forward recurrence. gates[(b,t), 512] holds W_ih z + b_ih on entry and the post-activation gates i,f,g,o on
// exit. Each CTA owns kLstmRows batch rows for all T steps (rows are independent: no inter-CTA synchronisation).
// Per step the [8 x 128] x [128 x 512] product is register-tiled: thread t owns gate columns 2t, 2t+1 for all 8
// rows (16 accumulators), reads h_{s-1} as two broadcast 16-byte shared-memory loads per k and the two weights as
// one 8-byte load; the whole of W_hh^T stays on chip for all T steps: k-rows 0..63 (128 KB) in shared memory,
// k-rows 64..127 in registers (2 columns x 64 k = 128 registers per thread). The x-projection of the step is
// loaded before the product and added after it, so its global-memory latency hides behind the FMAs. (The first version gave one column to each of 512 threads and re-read h with 1024
// scalar broadcast loads per thread and step: shared-memory-issue bound at 10 us per step.)
constexpr int kLstmSmemK = 64;  // k-rows of W_hh^T kept in shared memory
constexpr float kHprevScale = 8192.f;   // hscale_from_bound(1)
constexpr size_t kLstmFwdSmem = ((size_t)kLstmSmemK * kG4 + kLstmRows * kG4 + kLstmH * kLstmRows + kLstmRows * kLstmH) * sizeof(float);

//
// kLength (history_length, and inference with per-state lengths): row b's history is its first L_b = traj_length(len[b *
// len_stride], t) steps. The CTA runs the steps below the largest L of its rows; a row at s >= L keeps h and c by select (no
// arithmetic on a padding gate reaches them), takes feat from h_{L-1}, and gets a zero h_prev row (fp32 or fp16 pair) at every
// s >= L, the steps past the CTA's loop included: the W_hh gradient product reads all m*T rows. Its gate and c rows are not
// written (the backward pass does not read them).
template <bool kLength>
__global__ void __launch_bounds__(kLstmThreads, 1)
lstm_forward_kernel(float* __restrict__ gates, const float* __restrict__ whh_t, const float* __restrict__ b_hh,
                    int m, int t, float* __restrict__ hprev, float* __restrict__ cst, float* __restrict__ feat,
                    __half* __restrict__ hp_hi, __half* __restrict__ hp_lo, HScale* __restrict__ hp_hs, unsigned long long* trace,
                    const uint32_t* __restrict__ len, int len_stride) {
    extern __shared__ __align__(16) float lstm_smem[];
    float* Ws = lstm_smem;                          // [64][512]   W_hh^T rows k < 64
    float* ps = Ws + kLstmSmemK * kG4;              // [8][512]    pre-activations of this step
    float* hs = ps + kLstmRows * kG4;               // [128][8]    h_{s-1}, k-major
    float* cs = hs + kLstmH * kLstmRows;            // [8][128]    c_{s-1}
    const int tid = threadIdx.x;
    const int j0 = 2 * tid;
    const int b0 = blockIdx.x * kLstmRows;
    const int nrows = min(kLstmRows, m - b0);
    for (int i = tid; i < kLstmSmemK * kG4 / 4; i += kLstmThreads)
        reinterpret_cast<float4*>(Ws)[i] = __ldg(reinterpret_cast<const float4*>(whh_t) + i);
    for (int i = tid; i < kLstmRows * kLstmH; i += kLstmThreads) { hs[i] = 0.f; cs[i] = 0.f; }
    const float2 bias = __ldg(reinterpret_cast<const float2*>(b_hh + j0));
    float2 wreg[kLstmH - kLstmSmemK];
#pragma unroll
    for (int k = 0; k < kLstmH - kLstmSmemK; k++)
        wreg[k] = __ldg(reinterpret_cast<const float2*>(whh_t + (size_t)(kLstmSmemK + k) * kG4 + j0));
    __syncthreads();
    // Programmatic dependent launch: W_hh^T and b_hh were written at least two kernels back, so staging them (128 KB of
    // shared memory + 128 registers per thread) overlaps the tail of the input projection; the gates it writes are touched
    // only after this wait.
    pdl_wait();
    if (hp_hs && blockIdx.x == 0 && tid == 0) {   // |h| <= 1: the fp16 pairs of h_prev use the constant scale 2^13, no max|x| pass
        hp_hs->scale = kHprevScale;
        hp_hs->inv = 1.f / kHprevScale;
        hp_hs->amax = 1.f;
        hp_hs->bound = 1.f;
    }
    constexpr int kPairs = kLstmRows * kLstmH / kLstmThreads;
    const int u = tid & (kLstmH - 1), r4 = (tid >> 7) * kPairs;   // this thread's unit and first row in the element-wise part
    int steps = t;            // steps this CTA runs
    int lrow[kPairs];         // kLength: the lengths of this thread's rows (0 past the batch)
    if constexpr (kLength) {
        steps = 0;
#pragma unroll
        for (int r = 0; r < kLstmRows; r++)
            if (r < nrows) steps = max(steps, traj_length(__ldg(len + (size_t)(b0 + r) * len_stride), t));
#pragma unroll
        for (int k = 0; k < kPairs; k++)
            lrow[k] = r4 + k < nrows ? traj_length(__ldg(len + (size_t)(b0 + r4 + k) * len_stride), t) : 0;
    }
    unsigned long long* tr = (blockIdx.x == 0 && tid == 0) ? trace : nullptr;
    for (int s = 0; s < steps; s++) {
        lstm_trace_ev(tr, s, 0);
        float2 acc2[kLstmRows / 2][2];   // [row pair][column]: .x = row 2 rp, .y = row 2 rp + 1
        float2 gx[kLstmRows];
#pragma unroll
        for (int r = 0; r < kLstmRows; r++) {
            gx[r] = make_float2(0.f, 0.f);
            if (r < nrows) gx[r] = *reinterpret_cast<const float2*>(gates + ((size_t)(b0 + r) * t + s) * kG4 + j0);
        }
#pragma unroll
        for (int rp = 0; rp < kLstmRows / 2; rp++) {
            acc2[rp][0] = make_float2(bias.x, bias.x);
            acc2[rp][1] = make_float2(bias.y, bias.y);
        }
        auto fma_k = [&](int k, float2 w) {
            const float4 h0 = *reinterpret_cast<const float4*>(hs + k * kLstmRows);
            const float4 h1 = *reinterpret_cast<const float4*>(hs + k * kLstmRows + 4);
            const float2 hp[4] = {make_float2(h0.x, h0.y), make_float2(h0.z, h0.w), make_float2(h1.x, h1.y), make_float2(h1.z, h1.w)};
            const float2 wx = make_float2(w.x, w.x), wy = make_float2(w.y, w.y);
#pragma unroll
            for (int rp = 0; rp < kLstmRows / 2; rp++) {   // 8 FFMA2 = the 16 FMAs of this k
                acc2[rp][0] = ffma2(hp[rp], wx, acc2[rp][0]);
                acc2[rp][1] = ffma2(hp[rp], wy, acc2[rp][1]);
            }
        };
        lstm_trace_ev(tr, s, 1);
#pragma unroll 8
        for (int k = 0; k < kLstmSmemK; k++) fma_k(k, *reinterpret_cast<const float2*>(Ws + k * kG4 + j0));
        lstm_trace_ev(tr, s, 2);
#pragma unroll
        for (int k = kLstmSmemK; k < kLstmH; k++) fma_k(k, wreg[k - kLstmSmemK]);
#pragma unroll
        for (int r = 0; r < kLstmRows; r++) {
            const float a0 = (r & 1) ? acc2[r >> 1][0].y : acc2[r >> 1][0].x, a1 = (r & 1) ? acc2[r >> 1][1].y : acc2[r >> 1][1].x;
            *reinterpret_cast<float2*>(ps + r * kG4 + j0) = make_float2(a0 + gx[r].x, a1 + gx[r].y);
        }
        lstm_trace_ev(tr, s, 3);
        __syncthreads();
        lstm_trace_ev(tr, s, 4);
        // (row, unit) pairs: 8 * 128 = 1024 over 256 threads = 4 per thread: unit tid % 128, rows 4 (tid / 128) + k, so that a
        // thread's entries of the k-major hs array ([unit][8 rows]) are one 16-byte vector (scalar accesses, 32 bytes apart from
        // lane to lane, were 8-way bank conflicts). All loads
        // first, then the four gate chains side by side, then the stores: written pair by pair the shared-memory stores of one
        // pair ordered the loads of the next behind them and the phase took 3200 clocks of exposed latency per step. A pair's
        // h_{s-1} entry in hs is read by its own thread only (the product is done), so h_s goes straight back into it.
        float pin[kPairs][4], cin[kPairs], hin[kPairs];
#pragma unroll
        for (int k = 0; k < kPairs; k++) {
            const int r = r4 + k;
#pragma unroll
            for (int g = 0; g < 4; g++) pin[k][g] = ps[r * kG4 + g * kLstmH + u];
            cin[k] = cs[r * kLstmH + u];
        }
        {
            const float4 h4 = *reinterpret_cast<const float4*>(hs + u * kLstmRows + r4);
            hin[0] = h4.x; hin[1] = h4.y; hin[2] = h4.z; hin[3] = h4.w;
        }
        float gv[kPairs][4], cv[kPairs], hv[kPairs];
#pragma unroll
        for (int k = 0; k < kPairs; k++) {
            gv[k][0] = sigmoidf_(pin[k][0]);
            gv[k][1] = sigmoidf_(pin[k][1]);
            gv[k][2] = fast_tanh(pin[k][2]);
            gv[k][3] = sigmoidf_(pin[k][3]);
            cv[k] = fmaf(gv[k][1], cin[k], gv[k][0] * gv[k][2]);
            hv[k] = gv[k][3] * fast_tanh(cv[k]);
        }
        if constexpr (kLength) {
#pragma unroll
            for (int k = 0; k < kPairs; k++) {   // past its length a row keeps h and c (selects: the gates there may be anything)
                cv[k] = s < lrow[k] ? cv[k] : cin[k];
                hv[k] = s < lrow[k] ? hv[k] : hin[k];
            }
        }
#pragma unroll
        for (int k = 0; k < kPairs; k++) {
            const int r = r4 + k;
            if constexpr (kLength) {
                if (r < nrows && s >= lrow[k]) {   // a padding step: only its zero h_prev row
                    const size_t row = (size_t)(b0 + r) * t + s;
                    if (hprev) hprev[row * kLstmH + u] = 0.f;
                    if (hp_hi) {
                        hp_hi[row * kLstmH + u] = __float2half_rn(0.f);
                        hp_lo[row * kLstmH + u] = __float2half_rn(0.f);
                    }
                }
            }
            if (r < nrows && (!kLength || s < lrow[k])) {
                const size_t row = (size_t)(b0 + r) * t + s;
                float* g = gates + row * kG4;
                g[u] = gv[k][0]; g[kLstmH + u] = gv[k][1]; g[2 * kLstmH + u] = gv[k][2]; g[3 * kLstmH + u] = gv[k][3];
                if (cst) cst[row * kLstmH + u] = cv[k];
                if (hprev) hprev[row * kLstmH + u] = hin[k];   // h_{s-1}
                if (hp_hi) {   // ... or directly as the fp16 pair the W_hh gradient product reads
                    const float x = hin[k] * kHprevScale;
                    const __half hh = __float2half_rn(x);
                    hp_hi[row * kLstmH + u] = hh;
                    hp_lo[row * kLstmH + u] = __float2half_rn((x - __half2float(hh)) * 2048.f);
                }
                if (s == (kLength ? lrow[k] : t) - 1) feat[(size_t)(b0 + r) * kFeat + u] = hv[k];
            }
            cs[r * kLstmH + u] = r < nrows ? cv[k] : 0.f;
            if (r >= nrows) hv[k] = 0.f;
        }
        *reinterpret_cast<float4*>(hs + u * kLstmRows + r4) = make_float4(hv[0], hv[1], hv[2], hv[3]);
        lstm_trace_ev(tr, s, 5);
        __syncthreads();
        lstm_trace_ev(tr, s, 6);
        lstm_trace_ev(tr, s, 7);
    }
    if constexpr (kLength) {   // the steps past the CTA's longest row: zero h_prev rows only
        for (int s = steps; s < t; s++)
#pragma unroll
            for (int k = 0; k < kPairs; k++) {
                const size_t row = (size_t)(b0 + r4 + k) * t + s;
                if (r4 + k >= nrows) continue;
                if (hprev) hprev[row * kLstmH + u] = 0.f;
                if (hp_hi) {
                    hp_hi[row * kLstmH + u] = __float2half_rn(0.f);
                    hp_lo[row * kLstmH + u] = __float2half_rn(0.f);
                }
            }
    }
}

// BPTT. On entry gates holds post-activation i,f,g,o; on exit the pre-activation gradients dG.
// dfeat [m, ldf]: its first 128 columns are dL/dh_{T-1}. dh_{s-1} = dG_s W_hh is register-tiled like the forward
// product: thread (q, kp) owns hidden units 2kp, 2kp+1 for all 8 rows over gate rows [128q, 128q+128); the four
// partial sums are combined through shared memory. W_hh stays on chip: the first 64 gate rows of every quarter
// (128 KB) in shared memory, the other 64 in registers (128 per thread).
constexpr int kLstmSmemJ = 256;
constexpr int kLstmBwdPre = 6;   // per (row, unit) pair and step: gates i, f, g, o, c_s, c_{s-1}, prefetched one step ahead
constexpr size_t kLstmBwdSmem =
    ((size_t)kLstmSmemJ * kLstmH + kG4 * kLstmRows + 4 * kLstmRows * kLstmH + kLstmBwdPre * kLstmRows * kLstmH) * sizeof(float);

//
// kLength: the loop starts at the CTA's largest L - 1. A row at s >= L gets dG = 0 and carries dL/dh and dL/dc to s - 1
// unchanged (selects; its gate and c operands are not fetched), and every step past the loop gets zero dG rows: the weight
// gradient products and their max |dG| read all m*T rows.
template <bool kLength>
__global__ void __launch_bounds__(kLstmThreads, 1)
lstm_backward_kernel(float* __restrict__ gates, const float* __restrict__ whh, const float* __restrict__ cst,
                     const float* __restrict__ dfeat, int ldf, int m, int t, HScale* __restrict__ dg_hs, float* __restrict__ bias_part,
                     unsigned long long* trace, const uint32_t* __restrict__ len, int len_stride) {
    extern __shared__ __align__(16) float lstm_smem[];
    float* Wh = lstm_smem;                          // [4][64][128] W_hh rows 128q + jj, jj < 64
    float* dgs = Wh + kLstmSmemJ * kLstmH;          // [512][8]    dG of this step, j-major
    float* part = dgs + kG4 * kLstmRows;            // [4][8][128]   (dL/dh and dL/dc of a (row, unit) pair live in its thread's registers)
    float* pre = part + 4 * kLstmRows * kLstmH;     // [6][8][128] next step's operands of the element-wise part
    const int tid = threadIdx.x;
    const int b0 = blockIdx.x * kLstmRows;
    const int nrows = min(kLstmRows, m - b0);
    // The element-wise part of a step reads 6 values per (row, unit) pair from global memory; loaded where they are used
    // they cost 4900 clocks of exposed latency per step (41 % of the step, clock64 trace). Each thread fetches ITS pairs'
    // operands of step s-1 with cp.async while the dh product of step s runs; it is also the only reader of those entries.
    const int u = tid & (kLstmH - 1), r4 = (tid >> 7) * (kLstmRows * kLstmH / kLstmThreads);   // this thread's unit and first of its 4 rows
    int steps = t;                                               // steps this CTA runs
    int lrow[kLstmRows * kLstmH / kLstmThreads];                 // kLength: the lengths of this thread's rows (0 past the batch)
    auto prefetch = [&](int s) {
#pragma unroll
        for (int i = tid; i < kLstmRows * kLstmH; i += kLstmThreads) {   // i: the thread's private slots of `pre`
            const int r = r4 + i / kLstmThreads;
            if (r < nrows && (!kLength || s < lrow[i / kLstmThreads])) {
                const size_t row = (size_t)(b0 + r) * t + s;
                const float* g = gates + row * kG4 + u;
                const uint32_t dst = (uint32_t)__cvta_generic_to_shared(pre + i);
#pragma unroll
                for (int j = 0; j < 4; j++)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + j * kLstmRows * kLstmH * 4), "l"(g + j * kLstmH) : "memory");
                asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 4 * kLstmRows * kLstmH * 4), "l"(cst + row * kLstmH + u) : "memory");
                if (s > 0)
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst + 5 * kLstmRows * kLstmH * 4), "l"(cst + (row - 1) * kLstmH + u)
                                 : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // W_hh (a parameter: last written by the previous step's optimiser) is staged first; under a programmatic dependent
    // launch that overlaps the tail of the dgrad product whose output (dfeat) is read only after the wait below.
    for (int i = tid; i < kLstmSmemJ * kLstmH / 4; i += kLstmThreads) {
        const int row = i / (kLstmH / 4), c4 = i % (kLstmH / 4);       // smem row = 64 * quarter + jj
        const int j = (row >> 6) * kLstmH + (row & 63);
        reinterpret_cast<float4*>(Wh)[i] = __ldg(reinterpret_cast<const float4*>(whh + (size_t)j * kLstmH) + c4);
    }
    const int q = tid >> 6, k0 = (tid & 63) * 2;
    float2 wreg[64];
#pragma unroll
    for (int jj = 0; jj < 64; jj++) wreg[jj] = __ldg(reinterpret_cast<const float2*>(whh + (size_t)(q * kLstmH + 64 + jj) * kLstmH + k0));
    pdl_wait();
    if constexpr (kLength) {
        steps = 0;
#pragma unroll
        for (int r = 0; r < kLstmRows; r++)
            if (r < nrows) steps = max(steps, traj_length(__ldg(len + (size_t)(b0 + r) * len_stride), t));
#pragma unroll
        for (int k = 0; k < kLstmRows * kLstmH / kLstmThreads; k++)
            lrow[k] = r4 + k < nrows ? traj_length(__ldg(len + (size_t)(b0 + r4 + k) * len_stride), t) : 0;
    }
    prefetch(steps - 1);
    // dL/dh and dL/dc of this thread's 4 (row, unit) pairs (unit tid % 128, rows 4 (tid / 128) + k) live in registers
    constexpr int kPairs = kLstmRows * kLstmH / kLstmThreads;
    float dhr[kPairs], dcr[kPairs];
#pragma unroll
    for (int k = 0; k < kPairs; k++) {
        const int r = r4 + k;
        dhr[k] = r < nrows ? dfeat[(size_t)(b0 + r) * ldf + u] : 0.f;
        dcr[k] = 0.f;
    }
    __syncthreads();
    // max |dG| (for the fp16 split that follows) and this CTA's column sums of dG (the bias gradient): thread tid always
    // meets unit tid % 128 (rows 4 (tid / 128) + k)
    float run_max = 0.f, bs0 = 0.f, bs1 = 0.f, bs2 = 0.f, bs3 = 0.f;
    unsigned long long* tr = (blockIdx.x == 0 && tid == 0) ? trace : nullptr;
    for (int s = steps - 1; s >= 0; s--) {
        lstm_trace_ev(tr, t - 1 - s, 0);
        asm volatile("cp.async.wait_group 0;" ::: "memory");   // this thread's operands of step s have landed
        float pv[kLstmRows * kLstmH / kLstmThreads][kLstmBwdPre];
#pragma unroll
        for (int k = 0; k < kLstmRows * kLstmH / kLstmThreads; k++)
#pragma unroll
            for (int j = 0; j < kLstmBwdPre; j++) pv[k][j] = pre[j * kLstmRows * kLstmH + tid + k * kLstmThreads];
        if (s > 0) prefetch(s - 1);   // rows of step s-1: disjoint from the rows of step s written below
        float dd[kPairs][4];
#pragma unroll   // the four chains side by side: every operand is in registers
        for (int k = 0; k < kPairs; k++) {
            const float ig = pv[k][0], fg = pv[k][1], gg = pv[k][2], og = pv[k][3];
            const float tc = fast_tanh(pv[k][4]);
            const float cp = s > 0 ? pv[k][5] : 0.f;
            const float dct = dcr[k] + dhr[k] * og * (1.f - tc * tc);
            dd[k][0] = dct * gg * ig * (1.f - ig);
            dd[k][1] = dct * cp * fg * (1.f - fg);
            dd[k][2] = dct * ig * (1.f - gg * gg);
            dd[k][3] = dhr[k] * tc * og * (1.f - og);
            if constexpr (kLength) {   // past its length a row has dG = 0 and keeps dL/dc (its operands were not fetched)
                const bool live = s < lrow[k];
#pragma unroll
                for (int g = 0; g < 4; g++) dd[k][g] = live ? dd[k][g] : 0.f;
                dcr[k] = live ? dct * fg : dcr[k];
            } else {
                dcr[k] = dct * fg;
            }
        }
#pragma unroll
        for (int k = 0; k < kPairs; k++) {
            const int r = r4 + k;
            if (r < nrows) {
                float* g = gates + ((size_t)(b0 + r) * t + s) * kG4;
                g[u] = dd[k][0]; g[kLstmH + u] = dd[k][1]; g[2 * kLstmH + u] = dd[k][2]; g[3 * kLstmH + u] = dd[k][3];
                run_max = fmaxf(fmaxf(run_max, fmaxf(fabsf(dd[k][0]), fabsf(dd[k][1]))), fmaxf(fabsf(dd[k][2]), fabsf(dd[k][3])));
                bs0 += dd[k][0]; bs1 += dd[k][1]; bs2 += dd[k][2]; bs3 += dd[k][3];
            } else {
                dd[k][0] = dd[k][1] = dd[k][2] = dd[k][3] = 0.f;   // rows beyond the batch (their operands were never fetched)
                dcr[k] = 0.f;
            }
        }
#pragma unroll   // the thread's 4 rows of a gate column: one 16-byte store into the j-major dgs array
        for (int g4 = 0; g4 < 4; g4++)
            *reinterpret_cast<float4*>(dgs + (g4 * kLstmH + u) * kLstmRows + r4) = make_float4(dd[0][g4], dd[1][g4], dd[2][g4], dd[3][g4]);
        lstm_trace_ev(tr, t - 1 - s, 1);
        __syncthreads();
        lstm_trace_ev(tr, t - 1 - s, 2);
        if (s > 0) {  // dh_{s-1}[r][k] = sum_j dG[r][j] W_hh[j][k]
            float2 acc2[kLstmRows / 2][2];   // [row pair][column]
#pragma unroll
            for (int rp = 0; rp < kLstmRows / 2; rp++) acc2[rp][0] = acc2[rp][1] = make_float2(0.f, 0.f);
            auto fma_j = [&](int j, float2 w) {
                const float4 g0 = *reinterpret_cast<const float4*>(dgs + j * kLstmRows);
                const float4 g1 = *reinterpret_cast<const float4*>(dgs + j * kLstmRows + 4);
                const float2 gp[4] = {make_float2(g0.x, g0.y), make_float2(g0.z, g0.w), make_float2(g1.x, g1.y), make_float2(g1.z, g1.w)};
                const float2 wx = make_float2(w.x, w.x), wy = make_float2(w.y, w.y);
#pragma unroll
                for (int rp = 0; rp < kLstmRows / 2; rp++) {
                    acc2[rp][0] = ffma2(gp[rp], wx, acc2[rp][0]);
                    acc2[rp][1] = ffma2(gp[rp], wy, acc2[rp][1]);
                }
            };
#pragma unroll 8
            for (int jj = 0; jj < 64; jj++) fma_j(q * kLstmH + jj, *reinterpret_cast<const float2*>(Wh + (q * 64 + jj) * kLstmH + k0));
            lstm_trace_ev(tr, t - 1 - s, 3);
#pragma unroll
            for (int jj = 0; jj < 64; jj++) fma_j(q * kLstmH + 64 + jj, wreg[jj]);
            lstm_trace_ev(tr, t - 1 - s, 4);
#pragma unroll
            for (int r = 0; r < kLstmRows; r++)
                *reinterpret_cast<float2*>(part + (q * kLstmRows + r) * kLstmH + k0) =
                    make_float2((r & 1) ? acc2[r >> 1][0].y : acc2[r >> 1][0].x, (r & 1) ? acc2[r >> 1][1].y : acc2[r >> 1][1].x);
            lstm_trace_ev(tr, t - 1 - s, 5);
            __syncthreads();
            lstm_trace_ev(tr, t - 1 - s, 6);
#pragma unroll
            for (int k = 0; k < kPairs; k++) {
                const int i = (r4 + k) * kLstmH + u;
                const float dh = (part[i] + part[kLstmRows * kLstmH + i]) + (part[2 * kLstmRows * kLstmH + i] + part[3 * kLstmRows * kLstmH + i]);
                if constexpr (kLength) dhr[k] = s < lrow[k] ? dh : dhr[k];   // past its length a row keeps dL/dh
                else dhr[k] = dh;
            }
            // (no barrier here: `part` is next written after the barrier that follows the next step's element-wise part)
            lstm_trace_ev(tr, t - 1 - s, 7);
        }
    }
    if constexpr (kLength) {   // the steps past the CTA's longest row: zero dG rows only
        for (int s = steps; s < t; s++)
#pragma unroll
            for (int k = 0; k < kPairs; k++) {
                if (r4 + k >= nrows) continue;
                float* g = gates + ((size_t)(b0 + r4 + k) * t + s) * kG4;
                g[u] = 0.f; g[kLstmH + u] = 0.f; g[2 * kLstmH + u] = 0.f; g[3 * kLstmH + u] = 0.f;
            }
    }
    if (dg_hs) {
        const uint32_t wm = __reduce_max_sync(0xFFFFFFFFu, __float_as_uint(run_max));
        if ((tid & 31) == 0 && wm) atomicMax(reinterpret_cast<unsigned int*>(&dg_hs->amax), wm);
    }
    if (bias_part) {   // fixed order: the two threads of a unit, then (lstm_bias_grad_kernel) the CTAs in index order
        __syncthreads();
        float* bq = part;   // [2][4][128]
        const int half = tid >> 7, u = tid & 127;
        bq[(half * 4 + 0) * kLstmH + u] = bs0; bq[(half * 4 + 1) * kLstmH + u] = bs1;
        bq[(half * 4 + 2) * kLstmH + u] = bs2; bq[(half * 4 + 3) * kLstmH + u] = bs3;
        __syncthreads();
        for (int j = tid; j < kG4; j += kLstmThreads) bias_part[(size_t)blockIdx.x * kG4 + j] = bq[j] + bq[kG4 + j];
    }
}

// criterion (main.cpp:105-114) and the seed of backward: dy = dloss_i/dy / denom (mean over the
// GLOBAL batch). losses[0] += sum_i loss_i / denom (double).
__global__ void regression_loss_kernel(const float* __restrict__ y, const float* __restrict__ target, int m, int kind,
                                       double inv_denom, float* __restrict__ dy, double* __restrict__ losses, HScale* __restrict__ dy_hs) {
    pdl_wait();
    double local = 0.0;
    float dmax = 0.f;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < m; i += gridDim.x * blockDim.x) {
        const float d = y[i] - target[i];
        float g, l;
        if (kind == FI_LOSS_MAE) {
            g = (float)((d > 0.f) - (d < 0.f));
            l = fabsf(d);
        } else if (kind == FI_LOSS_HUBER) {  // smooth_l1_loss, beta = 1
            if (fabsf(d) < 1.f) { g = d; l = 0.5f * d * d; }
            else { g = (float)((d > 0.f) - (d < 0.f)); l = fabsf(d) - 0.5f; }
        } else {
            g = 2.f * d;
            l = d * d;
        }
        const float dv = (float)((double)g * inv_denom);
        dy[i] = dv;
        dmax = fmaxf(dmax, fabsf(dv));
        local += (double)l;
    }
    if (dy_hs) {   // max |dy| for the fp16 split of the tensor-core backward pass
        const uint32_t wm = __reduce_max_sync(0xffffffffu, __float_as_uint(dmax));
        if ((threadIdx.x & 31) == 0 && wm) atomicMax(reinterpret_cast<unsigned int*>(&dy_hs->amax), wm);
    }
    local = warp_sum(local);
    if ((threadIdx.x & 31) == 0 && local != 0.0) atomicAdd(losses, local * inv_denom);
}

// ------------------------------------------------------------------------------------------
static void ws_release(FarmerWs* w) {
    if (!w) return;
    float* f[] = {w->gates, w->hprev, w->cst, w->whh_t, w->feat, w->h_last, w->y, w->dy, w->target, w->dfeat, w->zpad};
    for (float* p : f)
        if (p) cudaFree(p);
    if (w->gemm_ws) cudaFree(w->gemm_ws);
    if (w->colsum_ws) cudaFree(w->colsum_ws);
    void* h[] = {w->hs, w->obs_hi, w->obs_lo, w->wih_hi, w->wih_lo, w->dg_hi, w->dg_lo, w->hp_hi, w->hp_lo, w->split_ws, w->bias_part};
    for (void* p : h)
        if (p) cudaFree(p);
    delete w;
}

// The workspaces of a step (training: states == rows) or of batched inference (the recurrence runs on `states` rows, the
// dense stack on `rows` candidate rows), and the dense stack `ds` they run with.
static int ws_create(fi_learner* l, size_t states, size_t rows, size_t t, bool training, FarmerWs** out, DenseStack* ds) {
    FarmerWs* w = new FarmerWs();
    *out = w;
    w->states = states;
    w->rows = rows;
    w->t = t;
    const size_t rt = states * t;
    // the tensor-core recurrence keeps gates and c in 64-row blocks (fi_internal.cuh): room for the padded rows, zeroed once so
    // that what the padding rows carry stays finite
    const size_t rt_pad = ((states + kStepBlockRows - 1) / kStepBlockRows) * kStepBlockRows * t;
    FI_CUDA_OK(cudaMalloc((void**)&w->gates, rt_pad * kG4 * sizeof(float)));
    FI_CUDA_OK(cudaMemset(w->gates, 0, rt_pad * kG4 * sizeof(float)));
    FI_CUDA_OK(cudaMalloc((void**)&w->whh_t, (size_t)kG4 * kLstmH * sizeof(float)));
    FI_CUDA_OK(cudaMalloc((void**)&w->feat, rows * kFeat * sizeof(float)));
    if (!training) FI_CUDA_OK(cudaMalloc((void**)&w->h_last, states * kFeat * sizeof(float)));
    if (training) {
        FI_CUDA_OK(cudaMalloc((void**)&w->y, rows * sizeof(float)));
        FI_CUDA_OK(cudaMalloc((void**)&w->hprev, rt * kLstmH * sizeof(float)));
        FI_CUDA_OK(cudaMalloc((void**)&w->cst, rt_pad * kLstmH * sizeof(float)));
        FI_CUDA_OK(cudaMemset(w->cst, 0, rt_pad * kLstmH * sizeof(float)));
        FI_CUDA_OK(cudaMalloc((void**)&w->dy, rows * sizeof(float)));
        FI_CUDA_OK(cudaMalloc((void**)&w->bias_part, ((rows + kLstmRows - 1) / kLstmRows) * kG4 * sizeof(float)));   // one row per CTA of the BPTT kernel
        FI_CUDA_OK(cudaMalloc((void**)&w->target, rows * sizeof(float)));
        const int mode = l->cfg.gemm_mode;
        size_t ws = 0;
        auto upd = [&](size_t b) { if (b > ws) ws = b; };
        upd(gemm_workspace_bytes(mode, 2, kG4, kZDim, (int)rt));
        upd(gemm_workspace_bytes(mode, 2, kG4, kLstmH, (int)rt));
        upd(gemm_workspace_bytes(mode, 2, kHid, kFeat, (int)rows));
        upd(gemm_workspace_bytes(mode, 2, kHid, kHid, (int)rows));
        upd(gemm_workspace_bytes(mode, 2, 1, kHid, (int)rows));
        // forward (NT) and dgrad (NN) shapes: the 3xFP16 operand copies are laid out per operand shape
        upd(gemm_workspace_bytes(mode, 0, (int)rt, kG4, kZDim));
        upd(gemm_workspace_bytes(mode, 0, (int)rows, kHid, kFeat));
        upd(gemm_workspace_bytes(mode, 0, (int)rows, kHid, kHid));
        upd(gemm_workspace_bytes(mode, 0, (int)rows, 1, kHid));
        upd(gemm_workspace_bytes(mode, 1, (int)rows, kHid, 1));
        upd(gemm_workspace_bytes(mode, 1, (int)rows, kFeat, kHid));
        upd(gemm_workspace_bytes(mode, 1, (int)rows, kHid, kHid));
        w->gemm_ws_bytes = ws;
        if (ws) FI_CUDA_OK(cudaMalloc(&w->gemm_ws, ws));
        w->colsum_ws_bytes = colsum_workspace_bytes((int)rt, kG4);
        FI_CUDA_OK(cudaMalloc(&w->colsum_ws, w->colsum_ws_bytes));
        w->half = (mode == FI_GEMM_AUTO || mode == FI_GEMM_TCGEN05_F16) && gemm_tc_available();
        if (w->half) {
            FI_CUDA_OK(cudaMalloc((void**)&w->hs, 4 * sizeof(HScale)));
            FI_CUDA_OK(cudaMalloc(&w->obs_hi, rt * kObsLdH * 2));
            FI_CUDA_OK(cudaMalloc(&w->obs_lo, rt * kObsLdH * 2));
            FI_CUDA_OK(cudaMalloc(&w->wih_hi, (size_t)kG4 * kObsLdH * 2));
            FI_CUDA_OK(cudaMalloc(&w->wih_lo, (size_t)kG4 * kObsLdH * 2));
            FI_CUDA_OK(cudaMalloc(&w->dg_hi, rt * kG4 * 2));
            FI_CUDA_OK(cudaMalloc(&w->dg_lo, rt * kG4 * 2));
            FI_CUDA_OK(cudaMalloc(&w->hp_hi, rt * kLstmH * 2));
            FI_CUDA_OK(cudaMalloc(&w->hp_lo, rt * kLstmH * 2));

            size_t sw = gemm_tc_split_workspace_bytes(2, kG4, kZDim, (int)rt);
            const size_t sw2 = gemm_tc_split_workspace_bytes(2, kG4, kLstmH, (int)rt);
            if (sw2 > sw) sw = sw2;
            w->split_ws_bytes = sw;
            if (sw) FI_CUDA_OK(cudaMalloc(&w->split_ws, sw));
            FI_CUDA_OK(cudaMalloc((void**)&w->dfeat, rows * kLstmH * sizeof(float)));
        }
        w->history = l->cfg.history_length != 0;
        // partial batches move AUTO below farmer_use_half's threshold: every mode but a 3xFP16-only learner can take the plain path
        if (w->history && !(w->half && mode == FI_GEMM_TCGEN05_F16)) FI_CUDA_OK(cudaMalloc((void**)&w->zpad, rt * kObsLd * sizeof(float)));
    }
    // split-operand buffers wherever the 3xFP16 path is available; farmer_dense_tc picks the path per step
    return dense_alloc(ds, DenseShape{kFeat, kFeatLdH, 1, 4}, rows, l->arena_elems, w->half ? kDenseTrain : kDenseNone, true,
                       training ? kDenseTrain : kDenseForward);
}

int farmer_alloc(fi_learner* l, Player* p) {
    FarmerWs* w = nullptr;
    const int rc = ws_create(l, l->cfg.batch_size, l->cfg.batch_size, l->cfg.entry_size, true, &w, &p->dense);
    p->farmer_ws = w;
    return rc;
}

void farmer_free(Player* p) {
    ws_release(p->farmer_ws);
    ws_release(p->farmer_inf_ws);
    p->farmer_ws = p->farmer_inf_ws = nullptr;
}

// The tensor-core path pays four pre-pass launches per product: taken from ~64 MFLOP up (as launch_gemm's AUTO does), always
// when the 3xFP16 mode is required.
static bool farmer_use_half(const fi_learner* l, const FarmerWs* w, int rt) {
    return w->half && (l->cfg.gemm_mode == FI_GEMM_TCGEN05_F16 || 2.0 * rt * kG4 * kZDim >= 64e6);
}

// The dense stack runs on the tensor cores (3xFP16, fused epilogues) when that format is required, and under AUTO from 128
// batch rows up (below that the fp32 FFMA kernels win: every product is launch-latency bound).
static bool farmer_dense_tc(const fi_learner* l, const DenseStack* ds, int m) {
    return ds->split && (l->cfg.gemm_mode == FI_GEMM_TCGEN05_F16 || m >= 128);
}

// The LSTM half of the forward over m rows of z (row (b,t) at z + (b*t + s) * ldz): the input projection and the recurrence,
// leaving h_{T-1} of row b in columns 0..127 of h [m, kFeat] (and the BPTT state when training). dense_tc: the dense stack
// that follows runs on split operands; its scales are zeroed and its parameters split here, before W_ih's split that shares
// the arena's scale. len (may be null): row b's history is its first traj_length(len[b * len_stride], t) steps, and h is
// h_{L-1}; a history learner's step passes the length words of the gathered batch (z is then that batch).
static int farmer_lstm_forward(fi_learner* l, FarmerWs* w, DenseStack* ds, const float* params, const float* z, int ldz, int m, int t,
                               bool dense_tc, float* h, cudaStream_t st, const uint32_t* len, int len_stride) {
    const auto& T = l->tensors;
    // inference workspaces carry no GEMM workspace: actor batches are small and run on the fp32 FFMA kernels
    const int mode = w->gemm_ws ? l->cfg.gemm_mode : FI_GEMM_SIMT;
    const int rt = m * t;
    // the recurrence on the tensor cores (lstm_tc.cu) needs the BPTT state arrays of a training workspace, and has no lengths
    const bool lstm_tc = !len && farmer_use_half(l, w, rt) && w->hp_hi && w->cst && lstm_tc_enabled();
    if (!lstm_tc) {
        LaunchScope ls("transpose_whh_kernel", st, 2.0 * 4 * kG4 * kLstmH, kWorkBytes);
        transpose_whh_kernel<<<(kG4 * kLstmH + 255) / 256, 256, 0, st>>>(params + T[1].offset, w->whh_t);
        FI_TRY(ls.done());
    }
    const bool half_proj = farmer_use_half(l, w, rt);
    if (half_proj || dense_tc) FI_TRY(launch_zero2(w->hs, 4 * sizeof(HScale), ds->hs, ds->hs ? kHsCount * sizeof(HScale) : 0, st));
    // parameters: max |p|, the split of the whole arena and dense1.w's copy with padded rows, one launch
    if (dense_tc) FI_TRY(dense_split_params(l, ds, params, st));
    // gates = z W_ih^T + b_ih for all B*T rows at once
    if (half_proj) {
        // a history learner's padding rows leave the max out and are split as zeros
        FI_TRY(launch_amax_split_h(z, ldz, (size_t)rt, kZDim, kObsLdH, w->obs_hi, w->obs_lo, w->hs + kLstmHsObs, st, w->history ? t : 0));
        HScale* wih_hs = dense_tc ? ds->hs + kHsW : w->hs + kLstmHsWih;   // the arena's scale bounds W_ih as well
        if (!dense_tc) FI_TRY(launch_amax(params + T[0].offset, kZDim, kG4, kZDim, wih_hs, st));
        FI_TRY(launch_split_h(params + T[0].offset, kZDim, kG4, kZDim, kObsLdH, w->wih_hi, w->wih_lo, wih_hs, dense_tc ? 0 : 1, st));
        const SplitMat a{w->obs_hi, w->obs_lo, kObsLdH, w->hs + kLstmHsObs}, b{w->wih_hi, w->wih_lo, kObsLdH, wih_hs};
        TcOut out{w->gates, kG4, nullptr, nullptr, 0, 0, nullptr, nullptr, 0, nullptr};
        if (lstm_tc) {   // straight into the blocked layout the recurrent kernels move with one bulk copy per CTA and step
            out.step_t = t;
            out.step_nblk = (m + kStepBlockRows - 1) / kStepBlockRows;
        }
        FI_TRY(launch_gemm_tc_split(0, rt, kG4, kZDim, a, b, out, params + T[2].offset, 0, nullptr, 0, nullptr, 0, st));
    } else {
        if (w->history) {   // the zero-padded copy of z (also the W_ih gradient's operand)
            FI_TRY(launch_obs_length(z, rt, t, w->zpad, st));
            z = w->zpad;
            ldz = kObsLd;
        }
        FI_TRY(launch_gemm(mode, 0, rt, kG4, kZDim, z, ldz, params + T[0].offset, kZDim, w->gates, kG4, params + T[2].offset,
                           0, nullptr, 0, w->gemm_ws, w->gemm_ws_bytes, st));
    }
    if (lstm_tc) {
        // h_{s-1} leaves the kernel as the fp16 pairs the W_hh gradient product reads (scale 2^13: |h| <= 1)
        FI_TRY(launch_lstm_forward_tc(w->gates, params + T[1].offset, params + T[3].offset, m, t, w->hp_hi, w->hp_lo, w->hs + kLstmHsHp, w->cst,
                                      h, kFeat, st));
    } else {
        // recurrent flops: 2 * 128 * 512 per (row, step)
        // (with lengths: nominal flops, as if every row ran all t steps)
        LaunchScope ls(len ? "lstm_forward_kernel_length" : "lstm_forward_kernel", st, 2.0 * kLstmH * kG4 * (double)rt, kWorkFlops);
        static std::atomic<uint64_t> fwd_attr[2] = {};
        const auto kernel = len ? lstm_forward_kernel<true> : lstm_forward_kernel<false>;
        FI_TRY(ensure_dynamic_smem(fwd_attr[len ? 1 : 0], (const void*)kernel, (int)kLstmFwdSmem));
        // training on the 3xFP16 path: h_prev leaves the kernel as the fp16 pairs the W_hh gradient product reads
        const bool hp_pairs = half_proj && w->hp_hi;
        launch_pdl(kernel, dim3((m + kLstmRows - 1) / kLstmRows), dim3(kLstmThreads), kLstmFwdSmem, st, w->gates, w->whh_t,
                   params + T[3].offset, m, t, hp_pairs ? nullptr : w->hprev, w->cst, h,
                   hp_pairs ? static_cast<__half*>(w->hp_hi) : nullptr, hp_pairs ? static_cast<__half*>(w->hp_lo) : nullptr,
                   hp_pairs ? w->hs + kLstmHsHp : nullptr, lstm_trace_buffer(), len, len_stride);
        FI_TRY(ls.done());
        lstm_trace_report("forward (FFMA)", lstm_trace_buffer(), t, st);
    }
    return FI_OK;
}

// The step's forward. Leaves y[m], feat, the dense stack's activations and the BPTT state.
static int farmer_forward(fi_learner* l, FarmerWs* w, DenseStack* ds, const float* params, const float* z, int ldz, int m, int t,
                          cudaStream_t st) {
    const bool dense_tc = farmer_dense_tc(l, ds, m);
    // a history learner: each slot's length word, word 183 of its record 0
    const uint32_t* len = w->history ? reinterpret_cast<const uint32_t*>(z) + kWLength : nullptr;
    FI_TRY(farmer_lstm_forward(l, w, ds, params, z, ldz, m, t, dense_tc, w->feat, st, len, t * kRecWords));
    if (dense_tc) {
        FI_TRY(launch_amax_split_h(w->feat, kFeat, (size_t)m, kFeat, kFeatLdH, ds->in_hi, ds->in_lo, ds->hs + kHsIn, st));
        return dense_forward_split(l, ds, params, m, w->y, st);
    }
    const int mode = w->gemm_ws ? l->cfg.gemm_mode : FI_GEMM_SIMT;
    return dense_forward_plain(l, ds, mode, params, w->feat, kFeat, m, w->y, w->gemm_ws, w->gemm_ws_bytes, st);
}

int farmer_forward_backward(fi_learner* l, Player* p, const float* batch, int m, int t, int global_m) {
    FarmerWs* w = p->farmer_ws;
    if (!w) return set_error(FI_ERR_STATE, "farmer workspaces missing");
    const auto& T = l->tensors;
    const int mode = l->cfg.gemm_mode;
    DenseStack* ds = &p->dense;
    cudaStream_t st = p->stream;
    float* g = p->grads;
    {
        LaunchScope ls("farmer_assemble_kernel", st, 2.0 * 4 * kXDim * (double)m, kWorkBytes);
        launch_pdl(farmer_assemble_kernel, dim3(m), dim3(128), 0, st, batch, m, t, w->feat, w->target);
        FI_TRY(ls.done());
    }
    FI_TRY(farmer_forward(l, w, ds, p->params, batch, kRecWords, m, t, st));
    FI_TRY(launch_zero2(p->d_losses, 4 * sizeof(double), nullptr, 0, st));
    const bool dense_tc = farmer_dense_tc(l, ds, m);
    {
        LaunchScope ls("regression_loss_kernel", st, 12.0 * m, kWorkBytes);
        launch_pdl(regression_loss_kernel, dim3((m + 255) / 256), dim3(256), 0, st, w->y, w->target, m, l->cfg.loss, 1.0 / (double)global_m,
                   w->dy, p->d_losses, dense_tc ? ds->hs + kHsDout : nullptr);
        FI_TRY(ls.done());
    }
    const float* d;   // dL/dfeat [m, ldd]
    int ldd;
    if (dense_tc) {
        FI_TRY(launch_split_h(w->dy, 1, (size_t)m, 1, kDoutLd, ds->dout_hi, ds->dout_lo, ds->hs + kHsDout, 1, st));   // max |dy| came with the loss
        // dL/dh_{T-1} = the first 128 columns of dL/dfeat (the x part of the feature row takes no gradient)
        FI_TRY(dense_backward_split(l, ds, w->dy, m, g, w->dfeat, kLstmH, nullptr, 0, st));
        d = w->dfeat;
        ldd = kLstmH;
    } else {
        FI_TRY(dense_backward_plain(l, ds, mode, p->params, w->feat, kFeat, w->dy, m, g, &d, w->gemm_ws, w->gemm_ws_bytes, w->colsum_ws,
                                    w->colsum_ws_bytes, st));
        ldd = kFeat;
    }
    // d = dfeat [m, ldd]: its first 128 columns are dL/dh_{T-1}; BPTT turns the stored gates into pre-activation gate gradients
    const int rt = m * t;
    const bool lstm_tc = !w->history && farmer_use_half(l, w, rt) && lstm_tc_enabled();
    if (lstm_tc) {
        // also leaves db_ih = db_hh (the column sums of dG) and max |dG|
        FI_TRY(launch_lstm_backward_tc(w->gates, p->params + T[1].offset, w->cst, d, ldd, m, t, w->hs + kLstmHsDg, w->bias_part,
                                       g + T[2].offset, g + T[3].offset, st));
    } else {
        const bool hist = w->history;
        LaunchScope ls(hist ? "lstm_backward_kernel_length" : "lstm_backward_kernel", st, 2.0 * kLstmH * kG4 * (double)m * t, kWorkFlops);
        static std::atomic<uint64_t> bwd_attr[2] = {};
        const auto kernel = hist ? lstm_backward_kernel<true> : lstm_backward_kernel<false>;
        FI_TRY(ensure_dynamic_smem(bwd_attr[hist ? 1 : 0], (const void*)kernel, (int)kLstmBwdSmem));
        const int ctas = (m + kLstmRows - 1) / kLstmRows;
        launch_pdl(kernel, dim3(ctas), dim3(kLstmThreads), kLstmBwdSmem, st, w->gates, p->params + T[1].offset, w->cst, d, ldd, m,
                   t, farmer_use_half(l, w, rt) ? w->hs + kLstmHsDg : nullptr, w->bias_part, lstm_trace_buffer(),
                   hist ? reinterpret_cast<const uint32_t*>(batch) + kWLength : nullptr, t * kRecWords);
        FI_TRY(ls.done());
        lstm_trace_report("backward (FFMA)", lstm_trace_buffer(), t, st);
        // db_ih = db_hh = the CTAs' column sums of dG, added in CTA order
        FI_TRY(launch_lstm_bias_grad(w->bias_part, ctas, g + T[2].offset, g + T[3].offset, st));
    }
    if (farmer_use_half(l, w, rt)) {
        // dW_ih = dgates^T z, dW_hh = dgates^T h_prev: the gate gradients are split once and read MN-major by both. The
        // tensor-core recurrence has already left max |dG| and h_prev as fp16 pairs.
        // (both recurrent kernels have left max |dG| and h_prev as fp16 pairs)
        if (lstm_tc) FI_TRY(launch_lstm_split_gates(w->gates, m, t, w->dg_hi, w->dg_lo, w->hs + kLstmHsDg, st));
        else FI_TRY(launch_split_h(w->gates, kG4, (size_t)rt, kG4, kG4, w->dg_hi, w->dg_lo, w->hs + kLstmHsDg, 1, st));
        const SplitMat dg{w->dg_hi, w->dg_lo, kG4, w->hs + kLstmHsDg};
        const SplitMat obs{w->obs_hi, w->obs_lo, kObsLdH, w->hs + kLstmHsObs}, hp{w->hp_hi, w->hp_lo, kLstmH, w->hs + kLstmHsHp};
        FI_TRY(launch_gemm_tc_split(2, kG4, kZDim, rt, dg, obs, TcOut{g + T[0].offset, kZDim, nullptr, nullptr, 0, 0, nullptr, nullptr, 0, nullptr},
                                    nullptr, 0, nullptr, 0, w->split_ws, w->split_ws_bytes, st));
        FI_TRY(launch_gemm_tc_split(2, kG4, kLstmH, rt, dg, hp, TcOut{g + T[1].offset, kLstmH, nullptr, nullptr, 0, 0, nullptr, nullptr, 0, nullptr},
                                    nullptr, 0, nullptr, 0, w->split_ws, w->split_ws_bytes, st));
    } else {
        // a history learner's z is the zero-padded copy the projection read
        FI_TRY(launch_gemm(mode, 2, kG4, kZDim, rt, w->gates, kG4, w->history ? w->zpad : batch, w->history ? kObsLd : kRecWords,
                           g + T[0].offset, kZDim, nullptr, 0, nullptr,
                           0, w->gemm_ws, w->gemm_ws_bytes, st));
        FI_TRY(launch_gemm(mode, 2, kG4, kLstmH, rt, w->gates, kG4, w->hprev, kLstmH, g + T[1].offset, kLstmH, nullptr, 0,
                           nullptr, 0, w->gemm_ws, w->gemm_ws_bytes, st));
    }
    return FI_OK;
}

int farmer_infer_alloc(fi_learner* l, Player* p, size_t states, size_t rows, size_t t) {
    ws_release(p->farmer_inf_ws);
    dense_free(&p->inf_dense);
    FarmerWs* w = nullptr;
    const int rc = ws_create(l, states, rows, t, false, &w, &p->inf_dense);
    p->farmer_inf_ws = w;
    return rc;
}

int farmer_infer(fi_learner* l, Player* p, const float* params, const float* z_dev, const float* x_dev, const uint32_t* offsets_dev,
                 const uint32_t* state_dev, const uint32_t* lengths_dev, size_t states, size_t rows, size_t t, float* values_dev,
                 int32_t* best_dev, cudaStream_t stream) {
    FarmerWs* w = p->farmer_inf_ws;
    if (!w || states > w->states || rows > w->rows || t > w->t) return set_error(FI_ERR_STATE, "farmer inference workspaces too small");
    // inference runs every product on the fp32 FFMA kernels: each row's value is then independent of the batch around it
    FI_TRY(farmer_lstm_forward(l, w, &p->inf_dense, params, z_dev, kZDim, (int)states, (int)t, false, w->h_last, stream, lengths_dev, 1));
    {
        const int n4 = (int)rows * kFeat4;
        LaunchScope ls("farmer_assemble_grouped_kernel", stream, 2.0 * 4 * kFeat * (double)rows, kWorkBytes);
        farmer_assemble_grouped_kernel<<<(n4 + 255) / 256, 256, 0, stream>>>(reinterpret_cast<const float4*>(w->h_last),
                                                                            reinterpret_cast<const float4*>(x_dev), state_dev, (int)rows,
                                                                            reinterpret_cast<float4*>(w->feat));
        FI_TRY(ls.done());
    }
    FI_TRY(dense_forward_plain(l, &p->inf_dense, FI_GEMM_SIMT, params, w->feat, kFeat, (int)rows, values_dev, nullptr, 0, stream));
    if (best_dev) {
        constexpr int kWarps = 8;
        LaunchScope ls("segment_argmax_kernel", stream, 4.0 * (double)rows + 12.0 * (double)states, kWorkBytes);
        segment_argmax_kernel<<<(unsigned)((states + kWarps - 1) / kWarps), kWarps * 32, 0, stream>>>(values_dev, offsets_dev, (int)states,
                                                                                                        best_dev);
        FI_TRY(ls.done());
    }
    return FI_OK;
}

}  // namespace fi
