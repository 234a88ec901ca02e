// The dense stack both learner steps end in: x_l = relu(x_{l-1} W_l^T + b_l) for five layers of width 512, then y = x_5 W_h^T + b_h.
// The actor-critic runs it as its whole trunk on the observations (162 -> 17), FarmerLstm on the feature row cat(h_{T-1}, x)
// (612 -> 1); DenseShape carries the difference. Two execution paths, same math:
//  * split operands (tcgen05, gemm_tc.cu): 3xFP16 (fp16 pairs, per-tensor HScales) or 3xTF32. Every activation and
//    back-propagated gradient is written as a hi/lo pair by the GEMM that produces it, with the ReLU bit mask (forward) or the
//    per-32-row column sums of the next bias gradient (dgrad), so no product re-splits its big operand; only the input, the
//    parameter arena and the loss gradient are split by pre-passes.
//  * plain fp32 operands through launch_gemm (gemm.cu), with column-sum launches for the bias gradients.
#include "learner.cuh"

namespace fi {

int dense_alloc(DenseStack* s, const DenseShape& sh, size_t rows, size_t arena_elems, DenseUse split, bool half, DenseUse plain) {
    s->sh = sh;
    s->rows = rows;
    if (split != kDenseNone) {
        const bool train = split == kDenseTrain;
        s->split = true;
        s->half = half;
        const size_t esz = s->esz = half ? 2 : 4;
        const size_t ab = ((arena_elems + 7) & ~(size_t)7) * esz, rb = rows * kHid * esz;
        if (half) FI_CUDA_OK(cudaMalloc((void**)&s->hs, kHsCount * sizeof(HScale)));
        FI_CUDA_OK(cudaMalloc(&s->w_hi, ab));
        FI_CUDA_OK(cudaMalloc(&s->w_lo, ab));
        FI_CUDA_OK(cudaMalloc(&s->w1_hi, (size_t)kHid * sh.in_ld * esz));
        FI_CUDA_OK(cudaMalloc(&s->w1_lo, (size_t)kHid * sh.in_ld * esz));
        FI_CUDA_OK(cudaMalloc(&s->in_hi, rows * sh.in_ld * esz));
        FI_CUDA_OK(cudaMalloc(&s->in_lo, rows * sh.in_ld * esz));
        for (int i = 0; i < 5; i++) {
            if (train || i < 2) {
                FI_CUDA_OK(cudaMalloc(&s->act_hi[i], rb));
                FI_CUDA_OK(cudaMalloc(&s->act_lo[i], rb));
            } else {   // nothing is kept for a backward pass
                s->act_hi[i] = s->act_hi[i & 1];
                s->act_lo[i] = s->act_lo[i & 1];
            }
            if (train) FI_CUDA_OK(cudaMalloc((void**)&s->relu_bits[i], rows * (kHid / 32) * sizeof(uint32_t)));
        }
        if (train) {
            for (int i = 0; i < 2; i++) {
                FI_CUDA_OK(cudaMalloc(&s->d_hi[i], rb));
                FI_CUDA_OK(cudaMalloc(&s->d_lo[i], rb));
            }
            FI_CUDA_OK(cudaMalloc(&s->dout_hi, rows * kDoutLd * esz));
            FI_CUDA_OK(cudaMalloc(&s->dout_lo, rows * kDoutLd * esz));
            FI_CUDA_OK(cudaMemset(s->dout_hi, 0, rows * kDoutLd * esz));
            FI_CUDA_OK(cudaMemset(s->dout_lo, 0, rows * kDoutLd * esz));
            const int part_rows = 4 * (int)((rows + 127) / 128);
            for (int i = 0; i < 5; i++) {
                FI_CUDA_OK(cudaMalloc((void**)&s->colsum_part[i], (size_t)part_rows * kHid * sizeof(float)));
                FI_CUDA_OK(cudaMalloc((void**)&s->colsum_scratch[i], grad_colsum_scratch_bytes(part_rows, kHid)));
                s->slab_bytes[i] = gemm_tc_split_workspace_bytes(2, kHid, i == 0 ? sh.in : kHid, (int)rows);
            }
            FI_CUDA_OK(cudaMalloc((void**)&s->colsum_scratch[5], grad_colsum_scratch_bytes((int)rows, sh.out)));
            s->slab_bytes[5] = gemm_tc_split_workspace_bytes(2, kHid, sh.out, (int)rows);
            for (int i = 0; i < 6; i++)
                if (s->slab_bytes[i]) FI_CUDA_OK(cudaMalloc(&s->slab[i], s->slab_bytes[i]));
        }
    }
    if (plain != kDenseNone) {
        for (int i = 0; i < 5; i++) FI_CUDA_OK(cudaMalloc((void**)&s->act[i], rows * kHid * sizeof(float)));
        if (plain == kDenseTrain)
            for (int i = 0; i < 2; i++) FI_CUDA_OK(cudaMalloc((void**)&s->d[i], rows * (sh.in > kHid ? sh.in : kHid) * sizeof(float)));
    }
    return FI_OK;
}

void dense_free(DenseStack* s) {
    void* f[] = {s->hs, s->w_hi, s->w_lo, s->w1_hi, s->w1_lo, s->in_hi, s->in_lo, s->d_hi[0], s->d_hi[1], s->d_lo[0], s->d_lo[1],
                 s->dout_hi, s->dout_lo, s->d[0], s->d[1]};
    for (void* x : f) if (x) cudaFree(x);
    for (int i = 0; i < 6; i++) {
        if (s->colsum_scratch[i]) cudaFree(s->colsum_scratch[i]);
        if (s->slab[i]) cudaFree(s->slab[i]);
    }
    for (int i = 0; i < 5; i++) {
        void* g[] = {s->relu_bits[i], s->colsum_part[i], s->act[i]};
        for (void* x : g) if (x) cudaFree(x);
        if (i >= 2 && s->act_hi[i] == s->act_hi[i & 1]) continue;   // a forward-only stack's alternating buffers
        if (s->act_hi[i]) cudaFree(s->act_hi[i]);
        if (s->act_lo[i]) cudaFree(s->act_lo[i]);
    }
    *s = DenseStack();
}

int dense_split_params(const fi_learner* l, DenseStack* s, const float* params, cudaStream_t st) {
    const int n = (int)l->arena_elems;
    const float* w1 = params + l->tensors[s->sh.w0].offset;
    if (s->half)
        return launch_amax_split_params(params, n, (int)((l->arena_elems + 7) & ~(size_t)7), s->w_hi, s->w_lo, w1, kHid, s->sh.in,
                                        s->sh.in_ld, s->w1_hi, s->w1_lo, s->hs + kHsW, st);
    FI_TRY(launch_split_tf32(params, n, 1, n, n, (float*)s->w_hi, (float*)s->w_lo, st));
    return launch_split_tf32(w1, s->sh.in, kHid, s->sh.in, s->sh.in_ld, (float*)s->w1_hi, (float*)s->w1_lo, st);
}

// The split operands every product of the stack reads: parameter tensor `tensor` ([rows, 512] row-major), the input, dense1.w's
// re-laid-out copy, layer l's activations. 3xFP16 scales: one for the arena, one per activation tensor.
namespace {
struct SplitOps {
    const fi_learner* l;
    const DenseStack* s;
    HScale* hs(int slot) const { return s->half ? s->hs + slot : nullptr; }
    SplitMat w(int tensor) const {
        const size_t off = l->tensors[tensor].offset * s->esz;
        return SplitMat{static_cast<char*>(s->w_hi) + off, static_cast<char*>(s->w_lo) + off, kHid, hs(kHsW)};
    }
    SplitMat in() const { return SplitMat{s->in_hi, s->in_lo, s->sh.in_ld, hs(kHsIn)}; }
    SplitMat w1() const { return SplitMat{s->w1_hi, s->w1_lo, s->sh.in_ld, hs(kHsW)}; }
    SplitMat act(int layer) const { return SplitMat{s->act_hi[layer], s->act_lo[layer], kHid, hs(kHsAct0 + layer)}; }
};
}  // namespace

int dense_forward_split(const fi_learner* l, DenseStack* s, const float* params, int rows, float* y, cudaStream_t st) {
    const auto& T = l->tensors;
    const int w0 = s->sh.w0;
    const SplitOps op{l, s};
    s->last_split = true;
    for (int layer = 0; layer < 5; layer++) {
        const TcOut out{nullptr, 0, s->act_hi[layer], s->act_lo[layer], kHid, 0, nullptr, s->relu_bits[layer], kHid / 32, nullptr,
                        op.hs(kHsAct0 + layer), op.hs(kHsW)};
        FI_TRY(launch_gemm_tc_split(0, rows, kHid, layer == 0 ? s->sh.in : kHid, layer == 0 ? op.in() : op.act(layer - 1),
                                    layer == 0 ? op.w1() : op.w(w0 + 2 * layer), out, params + T[w0 + 2 * layer + 1].offset, 1, nullptr,
                                    0, nullptr, 0, st));
    }
    return launch_gemm_tc_split(0, rows, s->sh.out, kHid, op.act(4), op.w(w0 + 10),
                                TcOut{y, s->sh.out, nullptr, nullptr, 0, 0, nullptr, nullptr, 0, nullptr}, params + T[w0 + 11].offset, 0,
                                nullptr, 0, nullptr, 0, st);
}

int dense_backward_split(const fi_learner* l, DenseStack* s, const float* dout, int rows, float* g, float* din, int din_cols,
                         void* colsum_ws, size_t colsum_ws_bytes, cudaStream_t st) {
    const auto& T = l->tensors;
    const int w0 = s->sh.w0, out = s->sh.out;
    const SplitOps op{l, s};
    const SplitMat dy{s->dout_hi, s->dout_lo, kDoutLd, op.hs(kHsDout)};
    // Bias column sums and split-K slab sums are deferred to launch_grad_finalize at the end.
    GradSegTable segs;
    int splits = 1;
    const int part_rows = 4 * ((rows + 127) / 128);
    // dW [512, n] (stored transposed as [n, 512] for the head) = a^T b, its split-K slabs kept in slab[i]
    auto wgrad = [&](const SplitMat& a, const SplitMat& b, int n, int transpose, int i, float* dst) {
        TcOut o{dst, transpose ? kHid : n, nullptr, nullptr, 0, transpose, nullptr, nullptr, 0, nullptr};
        o.deferred_splits = &splits;
        FI_TRY(launch_gemm_tc_split(2, kHid, n, rows, a, b, o, nullptr, 0, nullptr, 0, s->slab[i], s->slab_bytes[i], st));
        return splits > 1 ? grad_table_add_slabs(&segs, (const float*)s->slab[i], splits, (size_t)kHid * n, kHid * n, dst) : FI_OK;
    };
    // d_l = (a W_tensor) * relu'(act_l) as the next pair of the ping-pong, with the column sums of d_l (layer l's bias gradient)
    auto dgrad = [&](const SplitMat& a, int k, int tensor, int layer) {
        const int j = 4 - layer;
        return launch_gemm_tc_split(1, rows, kHid, k, a, op.w(tensor),
                                    TcOut{nullptr, 0, s->d_hi[j & 1], s->d_lo[j & 1], kHid, 0, s->relu_bits[layer], nullptr, kHid / 32,
                                          s->colsum_part[layer], op.hs(kHsD0 + j), nullptr},
                                    nullptr, 0, nullptr, 0, nullptr, 0, st);
    };
    // head: db = colsum(dy); dW_h^T [512, out] = act4^T dy; d4 = (dy W_h) * relu'(act4)
    if (s->half) FI_TRY(grad_table_add_colsum(&segs, dout, out, rows, out, g + T[w0 + 11].offset, s->colsum_scratch[5]));
    else FI_TRY(launch_colsum2((float*)s->dout_hi, (float*)s->dout_lo, kDoutLd, rows, out, g + T[w0 + 11].offset, colsum_ws, colsum_ws_bytes, st));
    FI_TRY(wgrad(op.act(4), dy, out, 1, 5, g + T[w0 + 10].offset));
    FI_TRY(dgrad(dy, out, w0 + 10, 4));
    for (int layer = 4; layer >= 0; layer--) {
        const int j = 4 - layer;
        const SplitMat d{s->d_hi[j & 1], s->d_lo[j & 1], kHid, op.hs(kHsD0 + j)};
        // bias gradient: the dgrad epilogue that produced d left per-32-row column sums (6.5 MB at 1024 x 100 rows instead of
        // re-reading 420 MB)
        FI_TRY(grad_table_add_colsum(&segs, s->colsum_part[layer], kHid, part_rows, kHid, g + T[w0 + 2 * layer + 1].offset,
                                     s->colsum_scratch[layer]));
        FI_TRY(wgrad(d, layer == 0 ? op.in() : op.act(layer - 1), layer == 0 ? s->sh.in : kHid, 0, layer, g + T[w0 + 2 * layer].offset));
        if (layer > 0) FI_TRY(dgrad(d, kHid, w0 + 2 * layer, layer - 1));
        else if (din)
            FI_TRY(launch_gemm_tc_split(1, rows, din_cols, kHid, d, op.w1(), TcOut{din, din_cols, nullptr, nullptr, 0, 0, nullptr, nullptr, 0, nullptr},
                                        nullptr, 0, nullptr, 0, nullptr, 0, st));
    }
    return launch_grad_finalize(&segs, st);
}

int dense_forward_plain(const fi_learner* l, DenseStack* s, int mode, const float* params, const float* x, int ldx, int rows, float* y,
                        void* ws, size_t ws_bytes, cudaStream_t st) {
    const auto& T = l->tensors;
    const int w0 = s->sh.w0;
    s->last_split = false;
    int k = s->sh.in;
    for (int layer = 0; layer < 5; layer++) {
        FI_TRY(launch_gemm(mode, 0, rows, kHid, k, x, ldx, params + T[w0 + 2 * layer].offset, k, s->act[layer], kHid,
                           params + T[w0 + 2 * layer + 1].offset, 1, nullptr, 0, ws, ws_bytes, st));
        x = s->act[layer];
        ldx = kHid;
        k = kHid;
    }
    return launch_gemm(mode, 0, rows, s->sh.out, kHid, x, kHid, params + T[w0 + 10].offset, kHid, y, s->sh.out,
                       params + T[w0 + 11].offset, 0, nullptr, 0, ws, ws_bytes, st);
}

int dense_backward_plain(const fi_learner* l, DenseStack* s, int mode, const float* params, const float* x, int ldx, const float* dout,
                         int rows, float* g, const float** din, void* ws, size_t ws_bytes, void* colsum_ws, size_t colsum_ws_bytes,
                         cudaStream_t st) {
    const auto& T = l->tensors;
    const int w0 = s->sh.w0, out = s->sh.out;
    // head: db = colsum(dy), dW_h = dy^T act4, d4 = (dy W_h) * relu'(act4)
    FI_TRY(launch_colsum(dout, out, rows, out, g + T[w0 + 11].offset, colsum_ws, colsum_ws_bytes, st));
    FI_TRY(launch_gemm(mode, 2, out, kHid, rows, dout, out, s->act[4], kHid, g + T[w0 + 10].offset, kHid, nullptr, 0, nullptr, 0, ws,
                       ws_bytes, st));
    float* d = s->d[0];
    float* d_next = s->d[1];
    FI_TRY(launch_gemm(mode, 1, rows, kHid, out, dout, out, params + T[w0 + 10].offset, kHid, d, kHid, nullptr, 0, s->act[4], kHid, ws,
                       ws_bytes, st));
    for (int layer = 4; layer >= 0; layer--) {
        const float* in = layer == 0 ? x : s->act[layer - 1];
        const int ld_in = layer == 0 ? ldx : kHid, k = layer == 0 ? s->sh.in : kHid;
        FI_TRY(launch_colsum(d, kHid, rows, kHid, g + T[w0 + 2 * layer + 1].offset, colsum_ws, colsum_ws_bytes, st));
        FI_TRY(launch_gemm(mode, 2, kHid, k, rows, d, kHid, in, ld_in, g + T[w0 + 2 * layer].offset, k, nullptr, 0, nullptr, 0, ws,
                           ws_bytes, st));
        if (layer > 0 || din) {   // dgrad into [rows, k]: the ReLU mask of the producing layer, none for the input
            FI_TRY(launch_gemm(mode, 1, rows, k, kHid, d, kHid, params + T[w0 + 2 * layer].offset, k, d_next, k, nullptr, 0,
                               layer == 0 ? nullptr : s->act[layer - 1], kHid, ws, ws_bytes, st));
            float* tmp = d; d = d_next; d_next = tmp;
        }
    }
    if (din) *din = d;
    return FI_OK;
}

const uint32_t* dense_relu_bits(const DenseStack& s, int layer) { return s.last_split ? s.relu_bits[layer] : nullptr; }
const float* dense_activation(const DenseStack& s, int layer) { return s.last_split ? nullptr : s.act[layer]; }

}  // namespace fi
