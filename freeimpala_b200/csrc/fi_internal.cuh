// Internal (non-ABI) entry points shared between the translation units of the library.
#pragma once
#include "fi_common.cuh"

namespace fi {

int launch_gather(const void* ring_base, size_t capacity, size_t slot_bytes, size_t first, size_t m, void* dst,
                  cudaStream_t stream);
// ring.cu: the consumer of a gathered batch tells the owning ring (looked up by the batch pointer; no-op for other pointers)
// that every read of it has been enqueued on `consumer`, so that the ring's next gather is ordered behind them
int ring_note_consumed(const void* dev_ptr, cudaStream_t consumer);
// The learner's device loss slots: {total, pg, baseline, entropy} of the step, then the pre-clip gradient norm that
// grad_norm_clip_kernel writes. The optimiser kernel copies all of them into the pinned read-back ring.
constexpr int kLossWords = 5;
struct OptConfig {       // what the fused optimiser kernel computes (adam.cu)
    int kind = FI_OPT_ADAM;  // fi_opt_kind
    double lr = 0.0;
    double rms_alpha = 0.99, rms_eps = 1e-8, rms_momentum = 0.0;   // FI_OPT_RMSPROP only
};
// coef: device float, the clip coefficient grad_norm_clip_kernel wrote (null = no clipping)
int launch_opt(const OptConfig& o, int64_t step, size_t n, float* p, const float* g, float* m, float* v, float grad_scale,
               cudaStream_t stream, const float* coef = nullptr, float* snapshot = nullptr, const double* losses_src = nullptr,
               double* losses_dst = nullptr);
struct OptLaunchDesc {   // a launch of the fused optimiser kernel, by value (adam.cu)
    const void* func;
    unsigned grid, block;
    float* p; const float* g; float* m; float* v; size_t n;
    alignas(8) unsigned char scalars[48];
    alignas(8) unsigned char extras[32];
    void* args[7];
    double work_bytes;
};
int opt_launch_desc(const OptConfig& o, int64_t step, size_t n, float* p, const float* g, float* m, float* v, float grad_scale,
                    const float* coef, float* snapshot, const double* losses_src, double* losses_dst, OptLaunchDesc* d);
// grad_norm.cu: *norm = ||g||_2 (squares and sums in double, deterministic order), *coef = min(1, max_norm / (*norm + 1e-6)).
// `scratch` holds grad_norm_scratch_bytes() of device memory, zeroed once; the kernel leaves it ready for the next launch,
// so a captured launch can be replayed.
size_t grad_norm_scratch_bytes();
int launch_grad_norm_clip(size_t n, const float* g, double max_norm, double* norm, float* coef, void* scratch, cudaStream_t stream);
int launch_vtrace_scan(int m, int t, const float* log_rho, const float* discount, const float* reward,
                       const float* value, const float* bootstrap, float rho_bar, float c_bar, float pg_rho_bar,
                       float lambda_, float* vs, float* pg_adv, cudaStream_t stream);
int launch_vtrace_loss_head(const void* batch, int m, int t, const float* head, int ldh, float rho_bar, float c_bar,
                            float pg_rho_bar, float lambda_, float baseline_cost, float entropy_cost, bool legal, float* dhead,
                            float* vs, float* pg_adv, double* losses, cudaStream_t stream,
                            float* dhead_hi = nullptr, float* dhead_lo = nullptr, int ld_split = 0, struct HScale* dhead_hs = nullptr);

// trans: 0 "NT" C = A[m,k] B[n,k]^T; 1 "NN" C = A[m,k] B[k,n]; 2 "TN" C = A[k,m]^T B[k,n].
int launch_gemm_simt(int trans, int m, int n, int k, const float* a, int lda, const float* b, int ldb, float* c,
                     int ldc, const float* bias, int relu, const float* mask, int ldmask, void* workspace,
                     size_t workspace_bytes, cudaStream_t stream);
size_t gemm_simt_workspace_bytes(int trans, int m, int n, int k);
int launch_colsum(const float* x, int ldx, int m, int n, float* out, void* workspace, size_t workspace_bytes,
                  cudaStream_t stream);
int launch_colsum2(const float* x, const float* x2, int ldx, int m, int n, float* out, void* workspace, size_t workspace_bytes,
                   cudaStream_t stream);
size_t colsum_workspace_bytes(int m, int n);

int launch_zero2(void* a, size_t a_bytes, void* b, size_t b_bytes, cudaStream_t stream);  // zero two small buffers, one kernel
int launch_copy_words(float* dst, const float* src, int n, cudaStream_t stream);            // small device copy as a kernel

// grad_reduce.cu: every split-K slab sum and bias column sum of a step in two launches (deterministic order).
constexpr int kGradSegMax = 16;
struct GradSeg {
    const float* src;   // kind 0: [splits][stride] partial slabs; kind 1: [rows = splits][ld = stride] matrix
    float* dst;         // n outputs in the gradient arena
    float* scratch;     // kind 1: [rb][n] row-block partials
    size_t stride;
    int n, splits, kind, rb, rows_per_block;
};
struct GradSegTable {
    GradSeg seg[kGradSegMax];
    int first_block[kGradSegMax + 1];    // pass 2: first block of every segment
    int first_block1[kGradSegMax + 1];   // pass 1: first block of every column-sum segment
    int colsum_index[kGradSegMax];
    int count = 0, num_colsum = 0;
};
int grad_table_add_slabs(GradSegTable* t, const float* slabs, int splits, size_t stride, int n, float* dst);
int grad_table_add_colsum(GradSegTable* t, const float* x, int ld, int rows, int n, float* dst, float* scratch);
size_t grad_colsum_scratch_bytes(int rows, int n);
int launch_grad_finalize(GradSegTable* t, cudaStream_t st);

// out[i] = sum_s partial[s * stride + i] in fixed order (deterministic split-K reduction).
int launch_reduce_splits(const float* partial, int splits, size_t stride, size_t n, float* out, cudaStream_t stream);

// ---- tcgen05 split-operand paths (gemm_tc.cu) ---------------------------------------------------
// Two operand formats, one kernel:
//  * 3xTF32: an fp32 matrix carried as the exact pair x = hi + lo (hi: low 13 mantissa bits cleared), both fp32 arrays;
//  * 3xFP16 (hs != nullptr): x * scale = hi + lo' / 2048 with hi, lo' fp16 arrays and `scale` a power of two kept in a
//    device-resident HScale next to the tensor's measured max |x|. kind::f16 MMAs run at twice the kind::tf32 rate on
//    half the shared-memory bytes per reduction element, and fp16 carries the same 11 significant bits as TF32.
struct HScale {    // device memory, one per split tensor
    float scale;   // power of two applied before the fp16 split
    float inv;     // 1 / scale
    float amax;    // max |x| in true units (atomicMax over the bit pattern; zero it before the producer runs)
    float bound;   // the a-priori bound the scale was derived from (diagnostics)
};
struct SplitMat {
    const void* hi;  // float (3xTF32) or __half (3xFP16)
    const void* lo;
    int ld;          // row stride in elements
    const HScale* hs = nullptr;  // non-null selects the fp16 format
};
struct TcOut {
    float* c; int ldc;                       // plain fp32 output (may be null)
    void* c_hi; void* c_lo; int ld_split;    // hi/lo output for the next GEMM (may be null); element type as the operands
    int transpose;                           // plain output written as c[col * ldc + row]
    const uint32_t* mask_bits_in;            // bit-packed ReLU decisions applied to the output (backward), or null
    uint32_t* mask_bits_out;                 // bit-packed (output > 0) written by a ReLU epilogue (forward), or null
    int mask_ldw;                            // words per mask row (a multiple of 4)
    float* colsum_out;                       // [4 * ceil(m/128), n] per-32-row column sums of the output (split-output path), or null
    HScale* out_hs = nullptr;                // fp16 format with a split output: receives the output's scale and max |x|
    const HScale* bias_hs = nullptr;         // fp16 format: a tensor whose amax bounds |bias| (the parameter arena)
    int* deferred_splits = nullptr;          // non-null: leave the split-K slabs in the workspace ([splits][m*n], the output's
                                             // layout) and report their number here (1: the product wrote `c` itself)
    int step_t = 0, step_nblk = 0;           // step_t > 0: c is the blocked gate array of the recurrent kernels (step_block_offset)
};

// ---- blocked per-step arrays of the recurrent kernels (lstm_tc.cu) ----------------------------------------------------------
// gates [(b, s), 512] and c [(b, s), 128] are kept so that what ONE CTA touches per step is contiguous: blocks of
// [4 gates][64 batch rows][16 units] fp32 (16 KB) / [64 batch rows][16 units] (4 KB), ordered [step][64-row block][unit block].
// Inside a block a row is 64 bytes and its four 16-byte chunks are XOR-swizzled with bits 1..2 of the row, so that threads
// that own one batch row each (a TMEM lane) read and write shared-memory copies of the block without bank conflicts.
constexpr int kStepBlockRows = 64, kStepBlockUnits = 16;
constexpr int kStepGateBlock = 4 * kStepBlockRows * kStepBlockUnits;   // floats per gate block
constexpr int kStepCellBlock = kStepBlockRows * kStepBlockUnits;       // floats per c block
__host__ __device__ __forceinline__ size_t step_block_index(int s, int b, int unit, int nblk) {
    return ((size_t)s * nblk + (b >> 6)) * 8 + (unit >> 4);
}
__host__ __device__ __forceinline__ int step_row_offset(int b, int unit) {   // floats, inside a [64 rows][16 units] tile
    const int r = b & 63, uu = unit & 15;
    return r * 16 + (((uu >> 2) ^ ((r >> 1) & 3)) << 2) + (uu & 3);
}
// gate column col = gate * 128 + unit of batch row b at step s
__host__ __device__ __forceinline__ size_t step_block_offset(int s, int b, int col, int nblk) {
    const int gate = col >> 7, unit = col & 127;
    return step_block_index(s, b, unit, nblk) * kStepGateBlock + gate * kStepCellBlock + step_row_offset(b, unit);
}
__host__ __device__ __forceinline__ size_t step_cell_offset(int s, int b, int unit, int nblk) {
    return step_block_index(s, b, unit, nblk) * kStepCellBlock + step_row_offset(b, unit);
}
int launch_split_tf32(const float* x, int ld_in, size_t rows, int cols, int ld_out, float* hi, float* lo, cudaStream_t st);
// fp16 format pre-passes: amax accumulates max |x| into hs->amax; split derives the scale from hs->amax (which must
// bound the matrix) and writes hi / lo' with columns [cols, ld_out) zero-filled. write_scale: publish scale/inv in *hs.
int launch_amax(const float* x, int ld_in, size_t rows, int cols, HScale* hs, cudaStream_t st);
int launch_split_h(const float* x, int ld_in, size_t rows, int cols, int ld_out, void* hi, void* lo, HScale* hs, int write_scale,
                   cudaStream_t st);
// amax + split in one cooperative launch (row matrices; hs->amax must be zero on entry; publishes scale / inv / bound)
int launch_amax_split_h(const float* x, int ld_in, size_t rows, int cols, int ld_out, void* hi, void* lo, HScale* hs, cudaStream_t st);
// lstm_tc.cu: the FarmerLstm recurrence on tcgen05 (clusters of 8 CTAs per 128 batch rows, exchange through DSMEM)
bool lstm_tc_enabled();   // FI_LSTM_TC=0 keeps the fp32 FFMA kernels of model_farmer.cu
int launch_lstm_forward_tc(float* gates, const float* whh, const float* b_hh, int m, int t, void* hp_hi, void* hp_lo, HScale* hp_hs,
                           float* cst, float* feat, int ldfeat, cudaStream_t st);
// gates / cst: blocked arrays (step_block_offset below), rows padded to 64. bias_part: [ceil(m / 64), 512] scratch.
int launch_lstm_backward_tc(float* gates, const float* whh, const float* cst, const float* dfeat, int ldf, int m, int t, HScale* dg_hs,
                            float* bias_part, float* g_bih, float* g_bhh, cudaStream_t st);
// db_ih = db_hh = sum over the BPTT kernel's CTAs (or clusters) of their column sums of dG, in index order
int launch_lstm_bias_grad(const float* part, int nparts, float* g_bih, float* g_bhh, cudaStream_t st);
// Trace hooks (the clock64 stamps behind FI_TC_TRACE / FI_LSTM_TRACE) are COMPILED OUT of the product build: a disabled hook
// is still a handful of predicated instructions per event, and in the tcgen05 GEMM those were 8.9 % of all warp instructions
// executed (ncu source page of the final round-2 build, profiles/r2_gemm.md). `FI_TRACE_BUILD=1 python -m freeimpala_b200.build
// --force` compiles them in for tools/gemm_trace.py and the LSTM phase trace; the environment switches then work as before.
#ifndef FI_TRACE_BUILD
#define FI_TRACE_BUILD 0
#endif
// true when this library carries the trace hooks; the host side warns once when a trace is requested without them
inline bool trace_hooks_built(const char* what) {
#if FI_TRACE_BUILD
    (void)what;
    return true;
#else
    static bool warned = false;
    if (!warned) {
        warned = true;
        fprintf(stderr, "[freeimpala_b200] %s is set but this library was built without the trace hooks: rebuild with "
                        "FI_TRACE_BUILD=1 python -m freeimpala_b200.build --force\n", what);
    }
    return false;
#endif
}
// FI_LSTM_TRACE=1 (diagnostics): a device buffer of [128 steps][12 points] clock64 stamps written by the first thread (points
// 0..7) and a second role (8..11) of CTA 0 of a recurrent kernel; the report prints median clocks between consecutive points
unsigned long long* lstm_trace_buffer();
void lstm_trace_report(const char* name, unsigned long long* dev, int steps, cudaStream_t st);
int launch_lstm_split_gates(const float* gates, int m, int t, void* hi, void* lo, HScale* hs, cudaStream_t st);
int launch_amax_split_params(const float* p, int n, int ld_flat, void* hi, void* lo, const float* w, int w_rows, int w_cols, int ld2,
                             void* hi2, void* lo2, HScale* hs, cudaStream_t st);
int launch_gemm_tc_split(int trans, int m, int n, int k, SplitMat a, SplitMat b, TcOut out, const float* bias, int relu,
                         const float* mask, int ldmask, void* workspace, size_t workspace_bytes, cudaStream_t st);
size_t gemm_tc_split_workspace_bytes(int trans, int m, int n, int k);
bool gemm_tc_available();

// Dispatching GEMM (gemm.cu): picks the tcgen05 3xTF32 kernel or the SIMT kernel per fi_gemm_mode.
int launch_gemm(int mode, int trans, int m, int n, int k, const float* a, int lda, const float* b, int ldb, float* c,
                int ldc, const float* bias, int relu, const float* mask, int ldmask, void* workspace,
                size_t workspace_bytes, cudaStream_t stream);
size_t gemm_workspace_bytes(int mode, int trans, int m, int n, int k);

}  // namespace fi
