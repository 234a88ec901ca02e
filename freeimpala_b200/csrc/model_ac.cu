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
//    gathered batch, or, with variable_length, out of a copy whose padding rows are zero (obs_length_kernel).
// variable_length: every observation pre-pass writes the rows past a trajectory's length (fi_learner.h, FI_REC_WORD_LENGTH)
// as zero rows without reading them, and the loss head gives them zero d(head) rows. The padding rows still run through the
// trunk and the head (fixed shapes: one captured graph), on zero inputs, so every later activation and gradient scale stays
// finite and independent of them (the scales are bounded from the input and weight maxima, gemm_tc.cu), and they add exact
// zeros to every weight and bias gradient.
#include "learner.cuh"

namespace fi {

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
    if (l->cfg.variable_length) FI_CUDA_OK(cudaMalloc((void**)&p->obs, rows * kObsLd * sizeof(float)));
    p->gemm_ws_bytes = gemm_simt_workspace_bytes(2, kHid, kHid, (int)rows);
    if (p->gemm_ws_bytes) FI_CUDA_OK(cudaMalloc(&p->gemm_ws, p->gemm_ws_bytes));
    return FI_OK;
}

int ac_forward_backward(fi_learner* l, Player* p, const float* batch, int m, int t, int /*global_m*/) {
    const auto& c = l->cfg;
    DenseStack* s = &p->dense;
    const int rows = m * t;
    cudaStream_t st = p->stream;
    const bool legal = c.legal_action_mask != 0, lengths = c.variable_length != 0;
    PopArtArgs pa;   // PopArt: mu and sigma from the player's device slot, per-trajectory partials reduced right after the loss head
    if (p->popart) {
        pa.ms = &p->popart->mu_f;
        pa.part = p->popart_part;
    }
    auto popart_sums = [&]() { return p->popart ? launch_popart_sums(p->popart_part, m, p->d_losses + kLossPopArt, st) : FI_OK; };
    if (!s->split) {
        const float* x = batch;   // the first GEMM's input: the batch itself (row stride 256 words) or its length-aware copy
        int ldx = kRecWords;
        if (lengths) {
            FI_TRY(launch_obs_length(batch, rows, t, p->obs, st));
            x = p->obs;
            ldx = kObsLd;
        }
        FI_TRY(dense_forward_plain(l, s, FI_GEMM_SIMT, p->params, x, ldx, rows, p->head, p->gemm_ws, p->gemm_ws_bytes, st));
        FI_TRY(launch_zero2(p->d_losses, 4 * sizeof(double), nullptr, 0, st));
        FI_TRY(launch_vtrace_loss_head(batch, m, t, p->head, kHead, c.rho_bar, c.c_bar, c.pg_rho_bar, c.lambda_,
                                       c.baseline_cost, c.entropy_cost, legal, lengths, p->dhead, nullptr, nullptr, p->d_losses, st,
                                       nullptr, nullptr, 0, nullptr, pa));
        FI_TRY(popart_sums());
        return dense_backward_plain(l, s, FI_GEMM_SIMT, p->params, x, ldx, p->dhead, rows, p->grads, nullptr, p->gemm_ws,
                                    p->gemm_ws_bytes, p->colsum_ws, p->colsum_ws_bytes, st);
    }
    // pre-passes: weights (4.6 MB) and observations -> hi/lo pairs
    if (s->half) {
        // one scale for the whole parameter arena (weights and biases), one for the observations; every activation and
        // back-propagated gradient gets its scale from the producing GEMM (bound k * amax_a * amax_b, gemm_tc.cu)
        FI_TRY(launch_zero2(s->hs, kHsCount * sizeof(HScale), p->d_losses, 4 * sizeof(double), st));
        FI_TRY(dense_split_params(l, s, p->params, st));
        // observations: max |x| and the split in one cooperative launch (the second pass reads the batch out of L2)
        FI_TRY(launch_amax_split_h(batch, kRecWords, (size_t)rows, kZDim, kObsLdH, s->in_hi, s->in_lo, s->hs + kHsIn, st,
                                   lengths ? t : 0));
    } else {
        FI_TRY(dense_split_params(l, s, p->params, st));
        FI_TRY(launch_split_tf32(batch, kRecWords, (size_t)rows, kZDim, kObsLd, (float*)s->in_hi, (float*)s->in_lo, st,
                                 lengths ? t : 0));
    }
    FI_TRY(dense_forward_split(l, s, p->params, rows, p->head, st));
    if (s->half) {  // the loss head writes plain fp32 rows and their max |x|; the fp16 split follows (13 MB)
        FI_TRY(launch_vtrace_loss_head(batch, m, t, p->head, kHead, c.rho_bar, c.c_bar, c.pg_rho_bar, c.lambda_,
                                       c.baseline_cost, c.entropy_cost, legal, lengths, p->dhead, nullptr, nullptr, p->d_losses, st,
                                       nullptr, nullptr, 0, s->hs + kHsDout, pa));
        FI_TRY(launch_split_h(p->dhead, kHead, (size_t)rows, kHead, kDoutLd, s->dout_hi, s->dout_lo, s->hs + kHsDout, 1, st));
    } else {
        FI_TRY(launch_zero2(p->d_losses, 4 * sizeof(double), nullptr, 0, st));
        FI_TRY(launch_vtrace_loss_head(batch, m, t, p->head, kHead, c.rho_bar, c.c_bar, c.pg_rho_bar, c.lambda_,
                                       c.baseline_cost, c.entropy_cost, legal, lengths, nullptr, nullptr, nullptr, p->d_losses, st,
                                       (float*)s->dout_hi, (float*)s->dout_lo, kDoutLd, nullptr, pa));
    }
    FI_TRY(popart_sums());
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

// ---------------------------------------------------------------- policy sampling -----
// The actor's action drawn from the softmax of a head row over its legal set (the rule is stated in fi_learner.h, at
// fi_learner_infer_sample, and restated in float64 by tests/sampling_reference.py). One thread per row. The uniform comes from
// Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011), counter (r, 0, 0, 0), key = the
// seed: stateless, so a row's draw depends only on (seed, r) and a call can be replayed.
__device__ __forceinline__ uint32_t philox4x32_10_word0(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
#pragma unroll
    for (int round = 0; round < 10; round++) {
        if (round) {
            k0 += 0x9E3779B9u;
            k1 += 0xBB67AE85u;
        }
        const uint32_t lo0 = 0xD2511F53u * c0, hi0 = __umulhi(0xD2511F53u, c0);
        const uint32_t lo1 = 0xCD9E8D57u * c2, hi1 = __umulhi(0xCD9E8D57u, c2);
        c0 = hi1 ^ c1 ^ k0;
        c1 = lo1;
        c2 = hi0 ^ c3 ^ k1;
        c3 = lo0;
    }
    return c0;
}

// desc (learner path, may be null): per row {support | greedy << 31, row index within its call, seed low, seed high}.
// Without desc (operator path) every row uses `legal` (null = all 16 legal), `seed`, `greedy` and its own row number.
// Head rows are staged through shared memory: a row of 17 floats is not 16-byte aligned, and with ldh == 17 the block's rows
// are one contiguous span, read with coalesced loads and read back one row per thread (odd stride: no bank conflict).
constexpr int kSampleThreads = 128;
__global__ void __launch_bounds__(kSampleThreads)
policy_sample_kernel(const float* __restrict__ head, int ldh, size_t rows, const uint4* __restrict__ desc,
                     const uint32_t* __restrict__ legal, uint32_t seed_lo, uint32_t seed_hi, int greedy_all,
                     int32_t* __restrict__ actions) {
    __shared__ float s_z[kSampleThreads * kNumActions];
    const size_t r0 = (size_t)blockIdx.x * kSampleThreads;
    const int n = (int)min((size_t)kSampleThreads, rows - r0);
    for (int i = threadIdx.x; i < n * kNumActions; i += kSampleThreads)
        s_z[i] = __ldg(head + (r0 + i / kNumActions) * ldh + i % kNumActions);
    __syncthreads();
    if ((int)threadIdx.x >= n) return;
    const size_t row = r0 + threadIdx.x;
    uint32_t sup, ctr, k0 = seed_lo, k1 = seed_hi;
    bool greedy = greedy_all != 0;
    if (desc) {
        const uint4 d = __ldg(desc + row);
        sup = d.x;
        greedy = (d.x >> 31) != 0;
        ctr = d.y;
        k0 = d.z;
        k1 = d.w;
    } else {
        sup = legal ? __ldg(legal + row) : 0xFFFFu;
        ctr = (uint32_t)row;
    }
    sup &= 0xFFFFu;
    const float* z = s_z + threadIdx.x * kNumActions;
    // greedy action: the largest logit in the support, NaN counting as largest, the lowest index on ties (numpy's argmax)
    int g = -1;
    float zg = 0.f;
#pragma unroll
    for (int j = 0; j < kNumActions; j++) {
        const float zj = z[j];
        if (((sup >> j) & 1u) && (g < 0 || (!isnan(zg) && (isnan(zj) || zj > zg)))) {
            g = j;
            zg = zj;
        }
    }
    int a = g;
    if (g >= 0 && !greedy && isfinite(zg)) {
        const uint32_t x0 = philox4x32_10_word0(ctr, 0u, 0u, 0u, k0, k1);
        const float u = (float)(x0 >> 8) * 0x1p-24f;
        float w[kNumActions], p[kNumActions], acc = 0.f;
#pragma unroll
        for (int j = 0; j < kNumActions; j++) {
            w[j] = ((sup >> j) & 1u) ? expf(z[j] - zg) : 0.f;
            acc += w[j];
            p[j] = acc;
        }
        const float thr = u * acc;
        int pick = -1, last = -1;
#pragma unroll
        for (int j = kNumActions - 1; j >= 0; j--) {   // the smallest j with P_j > u W (w_j = 0 outside the support)
            if (p[j] > thr && w[j] > 0.f) pick = j;
            if (last < 0 && w[j] > 0.f) last = j;
        }
        a = pick >= 0 ? pick : last;   // rounding left no P_j above u W: the largest j with a positive weight
    }
    actions[row] = a;
}

int launch_policy_sample(const float* head, int ldh, size_t rows, const uint4* desc, const uint32_t* legal, uint64_t seed,
                         int greedy, int32_t* actions, cudaStream_t stream) {
    if (ldh < kNumActions || (greedy != 0 && greedy != 1)) return set_error(FI_ERR_ARG, "policy sample: ldh >= 16 and greedy 0 or 1");
    if (rows == 0) return FI_OK;
    if (!head || !actions) return set_error(FI_ERR_ARG, "policy sample: null head or actions");
    if (rows > 0xFFFFFFFFull) return set_error(FI_ERR_ARG, "policy sample: the row counter is 32 bits, %zu rows", rows);
    // algorithmic traffic per row: 16 logits in, the legal word or the 16-byte descriptor in, the action out
    LaunchScope ls("policy_sample_kernel", stream, (64.0 + (desc ? 16.0 : legal ? 4.0 : 0.0) + 4.0) * (double)rows, kWorkBytes);
    policy_sample_kernel<<<(unsigned)((rows + kSampleThreads - 1) / kSampleThreads), kSampleThreads, 0, stream>>>(
        head, ldh, rows, desc, legal, (uint32_t)seed, (uint32_t)(seed >> 32), greedy, actions);
    return ls.done();
}

}  // namespace fi

extern "C" int fi_op_policy_sample(const float* head, int ldh, size_t rows, const uint32_t* legal, uint64_t seed, int greedy,
                                   int32_t* actions, void* stream) {
    return fi::launch_policy_sample(head, ldh, rows, nullptr, legal, seed, greedy, actions, (cudaStream_t)stream);
}
