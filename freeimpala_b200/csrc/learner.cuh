// Internal learner structures shared by learner.cu (host orchestration, model store, DP),
// model_ac.cu (MLP actor-critic V-trace step), model_farmer.cu (FarmerLstm step) and
// dense_stack.cu (the 5 x Linear(512) + ReLU stack and linear head both steps end in).
#pragma once
#include <atomic>
#include <condition_variable>
#include <mutex>
#include <shared_mutex>
#include <string>
#include <vector>

#include "fi_internal.cuh"

namespace fi {

struct TensorSpec {
    size_t offset, numel, rows, cols;
    int fan_in;
};

// Versioned weight publication: replaces Model / ModelManager::{getModel,updateModel,
// getLatestVersion,waitForModelUpdate} (reference data_structures.h:43-157, 433-480).
// After each optimiser update the learner stream snapshots the parameter arena into one of two
// HBM snapshots (D2D, ~1.5 us); the publication stream copies that snapshot into one of three
// pinned host blobs and a host callback flips `published` (the reference's shared_ptr swap,
// :441-451). Actors read the published blob under a shared lock: many readers, no copy under
// an exclusive mutex (the reference's getData() copies 1 MiB under model_mutex, :135-138).
struct ModelStore {
    size_t bytes = 0;                       // blob size = param_count * 4
    // Device snapshots of the weights, taken by the learner stream and drained (D2H) by the publication stream. The
    // publication stream also runs the host callback that flips the host blob, and a host callback runs when the OS
    // schedules CUDA's callback thread: with 8 ranks on 16 cores that lags by milliseconds. The learner stream only
    // ever waits for the snapshot it is about to overwrite, so kSnaps - 1 publications may be in flight before host
    // latency reaches the learner (2 snapshots cost 24 % of the 8-GPU step: profiles/r1_scaling.md).
    static constexpr int kSnaps = 8;
    float* dev_snap[kSnaps] = {};
    cudaEvent_t snap_ready[kSnaps] = {};  // D2D into the snapshot finished (learner stream)
    cudaEvent_t snap_free[kSnaps] = {};   // D2H out of the snapshot finished (pub stream)
    cudaEvent_t infer_done[kSnaps] = {};  // last inference reading the snapshot finished
    bool snap_free_recorded[kSnaps] = {}, infer_recorded[kSnaps] = {};
    unsigned char* host_buf[3] = {nullptr, nullptr, nullptr};
    uint64_t buf_version[3] = {0, 0, 0};
    int published = 0;                      // index into host_buf, guarded by rw
    std::shared_mutex rw;                   // readers: shared; flip: exclusive
    std::atomic<uint64_t> latest_version{0};
    std::mutex mu;                          // snapshot / host-buffer rotation bookkeeping
    std::mutex cv_mu;                       // waitForModelUpdate (:454-472)
    std::condition_variable cv;
    cudaStream_t pub_stream = nullptr;
    int next_host = 1, next_snap = 1;
    int newest_snap = 0;                    // snapshot holding the newest weights (inference)
};

struct PublishTicket {                      // argument of the publication host callback
    ModelStore* store;
    int host_index;
    uint64_t version;
};

// fp16 elements of a split observation row: 162 padded to 192 = three whole 128-byte lines per row, so that every TMA box row
// (one 64-element k-block of one observation) is ONE aligned line; with the minimal 168 (336-byte rows) each box row straddled
// two lines and layer 1's operand loads took 5800 clocks (profiles/r2_gemm_trace.md)
constexpr int kObsLdH = 192;

// The dense stack (dense_stack.cu): five Linear(512) + ReLU layers and a linear head. The actor-critic runs it as its whole
// trunk (162 -> 512 x 5 -> 17), FarmerLstm after the LSTM (612 -> 512 x 5 -> 1); the shape is data, the code is one.
struct DenseShape {
    int in;       // input width
    int in_ld;    // row stride of the split input pair and of dense1.w's re-laid-out copy (split-operand path)
    int out;      // head width
    int w0;       // tensor index of dense1.w: layer l's weight / bias are w0 + 2l / w0 + 2l + 1, the head's w0 + 10 / w0 + 11
};
// HScale slots of the split-operand path's 3xFP16 format (one per split tensor)
enum { kHsW = 0, kHsIn = 1, kHsDout = 2, kHsAct0 = 3, kHsD0 = 8, kHsCount = 14 };
constexpr int kDoutLd = 32;   // the output gradient pair [rows, 32]: `out` columns padded to one k-block, the rest stay zero
enum DenseUse { kDenseNone = 0, kDenseForward = 1, kDenseTrain = 2 };   // which buffers dense_alloc provides for a path

struct DenseStack {
    DenseShape sh{};
    size_t rows = 0;
    bool last_split = false;                       // the last forward ran on split operands: relu_bits hold its ReLU decisions
    // Split-operand path: every wgrad keeps its split-K slabs and every dgrad its column sums until the end of the backward
    // pass, where two launches (grad_reduce.cu) sum them all into the gradient arena.
    bool split = false, half = false;              // split buffers exist; 3xFP16 (fp16 pairs + HScales) instead of 3xTF32
    size_t esz = 0;                                // bytes per element of the hi / lo arrays
    HScale* hs = nullptr;                          // [kHsCount], 3xFP16 only
    void *w_hi = nullptr, *w_lo = nullptr;         // split parameter arena (same element offsets as params)
    void *w1_hi = nullptr, *w1_lo = nullptr;       // dense1.w re-laid out as [512, in_ld]
    void *in_hi = nullptr, *in_lo = nullptr;       // [rows, in_ld]
    // per-layer outputs [rows, 512]; forward-only stacks hold two buffers and alternate them (layer l writes buffer l % 2)
    void* act_hi[5] = {};
    void* act_lo[5] = {};
    uint32_t* relu_bits[5] = {};                   // [rows, 16] words: act_l > 0, bit-packed (training only)
    void* d_hi[2] = {};
    void* d_lo[2] = {};                            // back-propagated gradient ping-pong [rows, 512]
    void *dout_hi = nullptr, *dout_lo = nullptr;   // the loss gradient dL/dy [rows, kDoutLd]
    float* colsum_part[5] = {};                    // [4 * ceil(rows/128), 512] left by the dgrad that produced d_l
    float* colsum_scratch[6] = {};                 // row-block partials of the 5 layer biases + the head bias
    void* slab[6] = {};                            // split-K slabs of the 5 layer wgrads + the head wgrad
    size_t slab_bytes[6] = {};
    // plain fp32 path
    float* act[5] = {};                            // [rows, 512]
    float* d[2] = {};                              // [rows, max(in, 512)]: the layer-0 dgrad writes all `in` columns
};

struct FarmerWs;   // model_farmer.cu

// One caller of fi_learner_infer / fi_learner_infer_grouped / fi_learner_infer_sample waiting for its rows. A FarmerLstm
// request is `states` histories z [states, t, 162] and `rows` candidate rows x [rows, 484], rows offsets[s] .. offsets[s+1]-1
// belonging to state s; a plain fi_learner_infer request is `rows` states of one candidate each (offsets null). An
// actor-critic request with `actions` set also has each row's action drawn on the device (fi_learner_infer_sample).
struct InferReq {
    const float* obs;   // actor-critic: observations [rows, 162]; FarmerLstm: z
    const float* x;
    size_t rows, t, states;
    const uint32_t* offsets;   // [states + 1], or null: candidate r belongs to state r
    float* logits;
    float* values;
    int32_t* best;             // FarmerLstm, may be null: [states], each state's argmax within its group
    int status;
    bool done;
    int32_t* actions = nullptr;         // actor-critic sampling request: [rows]; null for every other request
    const uint32_t* legal = nullptr;    // [rows] legal words, or null = all 16 legal
    uint64_t seed = 0;
    int greedy = 0;
    const uint32_t* lengths = nullptr;  // FarmerLstm, may be null (= t): [states], the history length of each state
};

struct Player {
    int index = 0;
    std::mutex step_mu;         // serialises enqueueing on `stream` against checkpoint / arena access
    cudaStream_t stream = nullptr;
    float *params = nullptr, *grads = nullptr, *adam_m = nullptr, *adam_v = nullptr;  // RMSProp: m = momentum buffer, v = square average
    int64_t opt_step = 0;
    double lr = 0.0;            // learning rate of the next optimiser step (fi_learner_set_lr), written under step_mu
    float* clip_coef = nullptr; // device float: the clip coefficient of this step (max_grad_norm > 0 only)
    void* norm_ws = nullptr;    // grad_norm_clip_kernel's block partials and ticket
    std::atomic<uint64_t> steps_done{0};  // written under step_mu (release), read without it by fi_learner_losses_at / steps_done
    uint64_t version = 1;       // version of the weights in `params` (Model ctor -> 1, :55-58,127)
    double* d_losses = nullptr; // device double[kLossAlloc]: the four loss sums, the step's pre-clip gradient norm, PopArt's S1, S2, N
    // loss read-back ring: step s (1-based) lands in slot s % kLossRing of the pinned array, so that a host loop can read
    // step s-1's losses while step s runs (fi_learner_losses_at) without stalling the stream
    static constexpr int kLossRing = 8;
    double* h_losses = nullptr; // pinned double[kLossRing + 1][kLossWords]
    double* h_losses_dev = nullptr;  // the same memory as the device sees it (the optimiser kernel writes the losses there)
    cudaEvent_t loss_ev[kLossRing] = {};
    cudaEvent_t batch_ready = nullptr;
    size_t last_rows = 0;
    bool grads_valid = false;
    // step workspaces (sized for the step's rows: batch_size x entry_size for the actor-critic, batch_size for FarmerLstm)
    DenseStack dense;               // the step's dense stack
    float *head = nullptr, *dhead = nullptr;   // actor-critic: head output [rows, 17] and the loss head's fp32 gradient of it
    float* obs = nullptr;       // actor-critic, simt path with variable_length: the observations [rows, 164], padding rows zero
    void* gemm_ws = nullptr; size_t gemm_ws_bytes = 0;       // actor-critic FFMA path
    void* colsum_ws = nullptr; size_t colsum_ws_bytes = 0;   // actor-critic
    FarmerWs* farmer_ws = nullptr;      // FarmerLstm training workspaces
    FarmerWs* farmer_inf_ws = nullptr;  // FarmerLstm workspaces for batched inference
    unsigned char* stage_dev = nullptr;  // staged batch (fi_learner_stage_batch)
    unsigned char* stage_host = nullptr; // pinned bounce buffer for pageable sources
    size_t stage_bytes = 0;
    // inference: concurrent callers are combined into one forward per batch (fi_learner_infer)
    std::mutex infer_mu;
    std::condition_variable infer_cv;
    std::vector<InferReq*> infer_pending;
    bool infer_busy = false;
    uint64_t infer_calls = 0, infer_batches = 0, infer_rows = 0;
    cudaStream_t infer_stream = nullptr;
    // FarmerLstm: inf_in holds z per state, inf_x the candidate rows, inf_idx the batch's offsets [states + 1] followed by the
    // state of each candidate row [rows] and, in a batch with a fi_learner_infer_grouped_lengths request, each state's history
    // length [states]; inf_out the values [rows] followed by best [states] (int32).
    // Actor-critic: inf_in holds the observations, inf_out the head rows [rows, 17] followed by the actions [rows] (int32) of
    // a batch with a sampling request, inf_idx that batch's sampling descriptors [rows] x 4 words (policy_sample_kernel)
    float *inf_in = nullptr, *inf_x = nullptr, *inf_out = nullptr;
    uint32_t* inf_idx = nullptr;
    float *inf_host_in = nullptr, *inf_host_x = nullptr, *inf_host_out = nullptr;  // pinned
    uint32_t* inf_host_idx = nullptr;                                              // pinned
    DenseStack inf_dense;       // the dense stack of batched inference (forward only)
    size_t inf_rows_cap = 0, inf_states_cap = 0, inf_t_cap = 0;
    // the step as one CUDA graph (learner.cu step_with_graph)
    void* graph_exec = nullptr;       // cudaGraphExec_t
    void* graph = nullptr;            // cudaGraph_t it was instantiated from
    void* graph_opt_node = nullptr;   // cudaGraphNode_t of the optimiser kernel, re-parameterised every step
    const void* graph_batch_ptr = nullptr;
    size_t graph_batch_m = 0;
    uint64_t graph_kernels = 0;       // launches inside the graph (fi_kernel_launch_count)
    bool graph_failed = false;
    // PopArt (popart_beta > 0): the statistics, the loss head's per-trajectory partials [batch_size][3] and the update kernel's
    // node in the step graph (re-parameterised every step with the snapshot it publishes into, like the optimiser's)
    PopArtState* popart = nullptr;
    double* popart_part = nullptr;
    int popart_w_off = 0, popart_b_off = 0;   // head.w row 16 and head.b[16] in the arena
    void* graph_popart_node = nullptr;
    ModelStore store;
    uint64_t checkpoint_counter = 0;
    std::mutex save_mu;         // one fi_model_save per player at a time
    void* nccl_comm = nullptr;  // one communicator per player: players step concurrently
};

}  // namespace fi

struct fi_learner {
    fi_learner_config cfg;
    std::string ckpt_dir;
    std::vector<fi::TensorSpec> tensors;
    size_t param_count = 0, arena_elems = 0;
    std::vector<fi_ring*> rings;
    std::vector<fi::Player*> players;
    int dp_rank = 0, dp_world = 1;
    size_t dp_global_batch = 0;  // sum of the ranks' batch sizes (fi_learner_dp_init)
};

namespace fi {
// dense_stack.cu. `rows` of a forward / backward call may be fewer than the stack was allocated for.
// split / plain: the buffers of each path; a forward-only split stack keeps two activation pairs and no masks.
int dense_alloc(DenseStack* s, const DenseShape& sh, size_t rows, size_t arena_elems, DenseUse split, bool half, DenseUse plain);
void dense_free(DenseStack* s);   // frees every buffer and leaves an empty stack
// Split-operand path. The parameter arena and dense1.w's re-laid-out copy as hi/lo pairs (3xFP16: hs[kHsW] must be zero; one
// cooperative launch measures max |p| and writes both). The caller splits the input into in_hi / in_lo itself (scale
// hs[kHsIn]) and, for the backward pass, the loss gradient into dout_hi / dout_lo (scale hs[kHsDout]).
int dense_split_params(const fi_learner* l, DenseStack* s, const float* params, cudaStream_t st);
int dense_forward_split(const fi_learner* l, DenseStack* s, const float* params, int rows, float* y, cudaStream_t st);
// dout: the loss gradient in fp32 [rows, out] (3xFP16: the head bias gradient is its column sum; 3xTF32 sums the pair with
// colsum_ws instead). din (may be null): the first din_cols columns of dL/d(input), [rows, din_cols].
int dense_backward_split(const fi_learner* l, DenseStack* s, const float* dout, int rows, float* g, float* din, int din_cols,
                         void* colsum_ws, size_t colsum_ws_bytes, cudaStream_t st);
// Plain fp32 path through launch_gemm(mode): x [rows, in] with row stride ldx. din (may be null) receives dL/d(input)
// [rows, in] (row stride in), which is one of the stack's d buffers.
int dense_forward_plain(const fi_learner* l, DenseStack* s, int mode, const float* params, const float* x, int ldx, int rows, float* y,
                        void* ws, size_t ws_bytes, cudaStream_t st);
int dense_backward_plain(const fi_learner* l, DenseStack* s, int mode, const float* params, const float* x, int ldx, const float* dout,
                         int rows, float* g, const float** din, void* ws, size_t ws_bytes, void* colsum_ws, size_t colsum_ws_bytes,
                         cudaStream_t st);
// ReLU decisions of hidden layer `layer` of the last forward: bit-packed [rows, 16] words when it ran on split operands, else
// the fp32 activations [rows, 512]; the other accessor returns null
const uint32_t* dense_relu_bits(const DenseStack& s, int layer);
const float* dense_activation(const DenseStack& s, int layer);
// model_ac.cu
int ac_alloc(fi_learner* l, Player* p);
int ac_forward_backward(fi_learner* l, Player* p, const float* batch, int m, int t, int global_m);
int ac_infer_alloc(fi_learner* l, Player* p, size_t rows);
int ac_infer(fi_learner* l, Player* p, const float* params, const float* obs_dev, size_t rows, float* out_dev,
             cudaStream_t stream);
// actions[r] drawn from head row r (columns 0..15, row stride ldh) over its legal set (the rule: fi_learner.h). desc (may be
// null): per row {legal word | greedy << 31, RNG counter, seed low, seed high}; without it every row uses legal[r] (null = all
// 16 legal), seed, greedy and counter r.
int launch_policy_sample(const float* head, int ldh, size_t rows, const uint4* desc, const uint32_t* legal, uint64_t seed,
                         int greedy, int32_t* actions, cudaStream_t stream);
// model_farmer.cu
int farmer_alloc(fi_learner* l, Player* p);
void farmer_free(Player* p);
int farmer_forward_backward(fi_learner* l, Player* p, const float* batch, int m, int t, int global_m);
int farmer_infer_alloc(fi_learner* l, Player* p, size_t states, size_t rows, size_t t);
// The recurrence once per state, the dense stack once per candidate row: values_dev [rows]; best_dev (may be null) [states], the
// index within each group of its largest value (lowest on ties). offsets_dev [states + 1], state_dev [rows]: the groups.
// lengths_dev (may be null = every history t steps): [states], state s's history is z[s, 0..lengths[s]-1], 1 <= lengths[s] <= t.
int farmer_infer(fi_learner* l, Player* p, const float* params, const float* z_dev, const float* x_dev, const uint32_t* offsets_dev,
                 const uint32_t* state_dev, const uint32_t* lengths_dev, size_t states, size_t rows, size_t t, float* values_dev,
                 int32_t* best_dev, cudaStream_t stream);
}  // namespace fi
