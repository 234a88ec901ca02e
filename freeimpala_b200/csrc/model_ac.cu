// MLP actor-critic V-trace learner step (BASELINE.json north_star; configs[1], configs[3]).
// Trunk = the reference's dense1..5 shapes (cmd/libtorch_bench/main.cpp:17-21) applied per
// transition to the 162-feature observation; one fused head [17, 512]: 16 policy logits + value.
// Parameter order: dense1.w [512,162], dense1.b, dense2..5 .w [512,512], .b, head.w [17,512], head.b.
//
// The trunk and head are the dense stack (dense_stack.cu), on one of its two paths:
//  * split operands (gemm_mode auto / tcgen05 / tcgen05_f16): the tcgen05 kernel (gemm_tc.cu) in the 3xFP16 format, or in
//    3xTF32 for gemm_mode tcgen05 (and auto with FI_AC_FORMAT=tf32). The observations are split out of the gathered batch
//    (row stride 256 words) by a pre-pass here.
//  * plain fp32 (gemm_mode simt): FFMA GEMMs (gemm_simt.cu); the first GEMM reads the observations straight out of the
//    gathered batch.
#include "learner.cuh"

namespace fi {

constexpr int kObsLd = 164;     // 162 observation words padded to a 16-byte multiple (TMA row stride), 3xTF32 format

static bool use_tc(const fi_learner* l) { return l->cfg.gemm_mode != FI_GEMM_SIMT && gemm_tc_available(); }

int ac_alloc(fi_learner* l, Player* p) {
    const size_t rows = l->cfg.batch_size * l->cfg.entry_size;
    if ((l->cfg.gemm_mode == FI_GEMM_TCGEN05 || l->cfg.gemm_mode == FI_GEMM_TCGEN05_F16) && !gemm_tc_available())
        return set_error(FI_ERR_STATE, "gemm_mode tcgen05 requested but cuTensorMapEncodeTiled is unavailable");
    FI_CUDA_OK(cudaMalloc((void**)&p->head, rows * kHead * sizeof(float)));
    p->colsum_ws_bytes = colsum_workspace_bytes((int)rows, kHid);
    FI_CUDA_OK(cudaMalloc(&p->colsum_ws, p->colsum_ws_bytes));
    if (use_tc(l)) {
        // AUTO picks the 3xFP16 format (twice the tensor-core rate of 3xTF32 at the same 22 significant bits);
        // FI_AC_FORMAT=tf32 keeps AUTO on 3xTF32 (A/B experiments)
        const char* fmt = getenv("FI_AC_FORMAT");
        const bool half = l->cfg.gemm_mode == FI_GEMM_TCGEN05_F16 || (l->cfg.gemm_mode == FI_GEMM_AUTO && !(fmt && fmt[0] == 't'));
        FI_TRY(dense_alloc(&p->dense, DenseShape{kZDim, half ? kObsLdH : kObsLd, kHead, 0}, rows, l->arena_elems, kDenseTrain, half,
                           kDenseNone));
        // 3xFP16: the loss head writes plain fp32 rows (and their max |x|), split afterwards; 3xTF32: it writes the pair itself
        if (half) FI_CUDA_OK(cudaMalloc((void**)&p->dhead, rows * kHead * sizeof(float)));
        return FI_OK;
    }
    FI_TRY(dense_alloc(&p->dense, DenseShape{kZDim, 0, kHead, 0}, rows, l->arena_elems, kDenseNone, false, kDenseTrain));
    FI_CUDA_OK(cudaMalloc((void**)&p->dhead, rows * kHead * sizeof(float)));
    p->gemm_ws_bytes = gemm_simt_workspace_bytes(2, kHid, kHid, (int)rows);
    if (p->gemm_ws_bytes) FI_CUDA_OK(cudaMalloc(&p->gemm_ws, p->gemm_ws_bytes));
    return FI_OK;
}

int ac_forward_backward(fi_learner* l, Player* p, const float* batch, int m, int t, int /*global_m*/) {
    const auto& c = l->cfg;
    DenseStack* s = &p->dense;
    const int rows = m * t;
    cudaStream_t st = p->stream;
    if (!s->split) {
        FI_TRY(dense_forward_plain(l, s, FI_GEMM_SIMT, p->params, batch, kRecWords, rows, p->head, p->gemm_ws, p->gemm_ws_bytes, st));
        FI_TRY(launch_zero2(p->d_losses, 4 * sizeof(double), nullptr, 0, st));
        FI_TRY(launch_vtrace_loss_head(batch, m, t, p->head, kHead, c.rho_bar, c.c_bar, c.pg_rho_bar, c.lambda_,
                                       c.baseline_cost, c.entropy_cost, c.legal_action_mask != 0, p->dhead, nullptr, nullptr,
                                       p->d_losses, st));
        return dense_backward_plain(l, s, FI_GEMM_SIMT, p->params, batch, kRecWords, p->dhead, rows, p->grads, nullptr, p->gemm_ws,
                                    p->gemm_ws_bytes, p->colsum_ws, p->colsum_ws_bytes, st);
    }
    // pre-passes: weights (4.6 MB) and observations -> hi/lo pairs
    if (s->half) {
        // one scale for the whole parameter arena (weights and biases), one for the observations; every activation and
        // back-propagated gradient gets its scale from the producing GEMM (bound k * amax_a * amax_b, gemm_tc.cu)
        FI_TRY(launch_zero2(s->hs, kHsCount * sizeof(HScale), p->d_losses, 4 * sizeof(double), st));
        FI_TRY(dense_split_params(l, s, p->params, st));
        // observations: max |x| and the split in one cooperative launch (the second pass reads the batch out of L2)
        FI_TRY(launch_amax_split_h(batch, kRecWords, (size_t)rows, kZDim, kObsLdH, s->in_hi, s->in_lo, s->hs + kHsIn, st));
    } else {
        FI_TRY(dense_split_params(l, s, p->params, st));
        FI_TRY(launch_split_tf32(batch, kRecWords, (size_t)rows, kZDim, kObsLd, (float*)s->in_hi, (float*)s->in_lo, st));
    }
    FI_TRY(dense_forward_split(l, s, p->params, rows, p->head, st));
    if (s->half) {  // the loss head writes plain fp32 rows and their max |x|; the fp16 split follows (13 MB)
        FI_TRY(launch_vtrace_loss_head(batch, m, t, p->head, kHead, c.rho_bar, c.c_bar, c.pg_rho_bar, c.lambda_,
                                       c.baseline_cost, c.entropy_cost, c.legal_action_mask != 0, p->dhead, nullptr, nullptr,
                                       p->d_losses, st, nullptr, nullptr, 0, s->hs + kHsDout));
        FI_TRY(launch_split_h(p->dhead, kHead, (size_t)rows, kHead, kDoutLd, s->dout_hi, s->dout_lo, s->hs + kHsDout, 1, st));
    } else {
        FI_TRY(launch_zero2(p->d_losses, 4 * sizeof(double), nullptr, 0, st));
        FI_TRY(launch_vtrace_loss_head(batch, m, t, p->head, kHead, c.rho_bar, c.c_bar, c.pg_rho_bar, c.lambda_,
                                       c.baseline_cost, c.entropy_cost, c.legal_action_mask != 0, nullptr, nullptr, nullptr,
                                       p->d_losses, st, (float*)s->dout_hi, (float*)s->dout_lo, kDoutLd));
    }
    return dense_backward_split(l, s, p->dhead, rows, p->grads, nullptr, 0, p->colsum_ws, p->colsum_ws_bytes, st);
}

// ---------------------------------------------------------------- batched actor inference -----
// (SURVEY.md 8f rank 2) the forward kernels of the learner step on the published device snapshot of the weights:
// obs_dev [rows,162] -> out_dev [rows,17]. Small batches (a few actors x a few rows) run the fp32 FFMA kernels; from
// kInferTcRows rows on, the tensor-core forward of the step: 3xFP16 operand pairs, the same tcgen05 kernel and epilogue,
// with two alternating activation buffers instead of five (nothing is kept for a backward pass).
constexpr size_t kInferTcRows = 256;

int ac_infer_alloc(fi_learner* l, Player* p, size_t rows) {
    dense_free(&p->inf_dense);
    const DenseUse split = use_tc(l) && l->cfg.gemm_mode != FI_GEMM_TCGEN05 && rows >= kInferTcRows ? kDenseForward : kDenseNone;
    return dense_alloc(&p->inf_dense, DenseShape{kZDim, kObsLdH, kHead, 0}, rows, l->arena_elems, split, true, kDenseForward);
}

int ac_infer(fi_learner* l, Player* p, const float* params, const float* obs_dev, size_t rows, float* out_dev,
             cudaStream_t stream) {
    DenseStack* s = &p->inf_dense;
    if (!s->split || rows < kInferTcRows || rows > s->rows)
        return dense_forward_plain(l, s, FI_GEMM_SIMT, params, obs_dev, kZDim, (int)rows, out_dev, nullptr, 0, stream);
    const int n = (int)l->arena_elems;
    FI_TRY(launch_zero2(s->hs, kHsCount * sizeof(HScale), nullptr, 0, stream));
    FI_TRY(launch_amax(params, n, 1, n, s->hs + kHsW, stream));
    FI_TRY(launch_amax(obs_dev, kZDim, rows, kZDim, s->hs + kHsIn, stream));
    FI_TRY(launch_split_h(params, n, 1, n, (int)((l->arena_elems + 7) & ~(size_t)7), s->w_hi, s->w_lo, s->hs + kHsW, 1, stream));
    FI_TRY(launch_split_h(params + l->tensors[0].offset, kZDim, kHid, kZDim, kObsLdH, s->w1_hi, s->w1_lo, s->hs + kHsW, 0, stream));
    FI_TRY(launch_split_h(obs_dev, kZDim, rows, kZDim, kObsLdH, s->in_hi, s->in_lo, s->hs + kHsIn, 1, stream));
    return dense_forward_split(l, s, params, (int)rows, out_dev, stream);
}

}  // namespace fi
