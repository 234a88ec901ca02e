// Internal learner structures shared by learner.cu (host orchestration, model store, DP),
// model_ac.cu (MLP actor-critic V-trace step) and model_farmer.cu (FarmerLstm step).
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

struct InferReq {   // one caller of fi_learner_infer waiting for its rows
    const float* obs;
    const float* x;
    size_t rows, t;
    float* logits;
    float* values;
    int status;
    bool done;
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
    double* d_losses = nullptr; // device double[kLossWords]: the four loss sums, then the step's pre-clip gradient norm
    // loss read-back ring: step s (1-based) lands in slot s % kLossRing of the pinned array, so that a host loop can read
    // step s-1's losses while step s runs (fi_learner_losses_at) without stalling the stream
    static constexpr int kLossRing = 8;
    double* h_losses = nullptr; // pinned double[kLossRing + 1][kLossWords]
    double* h_losses_dev = nullptr;  // the same memory as the device sees it (the optimiser kernel writes the losses there)
    cudaEvent_t loss_ev[kLossRing] = {};
    cudaEvent_t batch_ready = nullptr;
    size_t last_rows = 0;
    bool grads_valid = false;
    // step workspaces (model specific, sized for batch_size x entry_size rows)
    std::vector<float*> act;    // activations
    float *d_a = nullptr, *d_b = nullptr, *head = nullptr, *dhead = nullptr;
    void* gemm_ws = nullptr; size_t gemm_ws_bytes = 0;
    void* colsum_ws = nullptr; size_t colsum_ws_bytes = 0;
    void* model_ws = nullptr;
    void* ac_tc = nullptr;          // AcTc (model_ac.cu): hi/lo activation pairs of the tensor-core path
    void* farmer_ws = nullptr;      // FarmerWs (model_farmer.cu): training workspaces
    void* farmer_inf_ws = nullptr;  // FarmerWs for batched inference
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
    float *inf_in = nullptr, *inf_x = nullptr, *inf_out = nullptr;
    float *inf_host_in = nullptr, *inf_host_x = nullptr, *inf_host_out = nullptr;  // pinned
    std::vector<float*> inf_act;
    void* inf_model_ws = nullptr;
    size_t inf_rows_cap = 0, inf_t_cap = 0;
    // the step as one CUDA graph (learner.cu step_with_graph)
    void* graph_exec = nullptr;       // cudaGraphExec_t
    void* graph = nullptr;            // cudaGraph_t it was instantiated from
    void* graph_opt_node = nullptr;   // cudaGraphNode_t of the optimiser kernel, re-parameterised every step
    const void* graph_batch_ptr = nullptr;
    size_t graph_batch_m = 0;
    uint64_t graph_kernels = 0;       // launches inside the graph (fi_kernel_launch_count)
    bool graph_failed = false;
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
// model_ac.cu
int ac_alloc(fi_learner* l, Player* p);
void ac_free(Player* p);
int ac_forward_backward(fi_learner* l, Player* p, const float* batch, int m, int t, int global_m);
int ac_infer_alloc(fi_learner* l, Player* p, size_t rows);
void ac_infer_free(Player* p);
int ac_infer(fi_learner* l, Player* p, const float* params, const float* obs_dev, size_t rows, float* out_dev,
             cudaStream_t stream);
// ReLU outputs of hidden layer `layer` of the last forward: *a (+ *lo when stored as a hi/lo pair)
const uint32_t* ac_relu_bits(Player* p, int layer);
int ac_activation(Player* p, int layer, const float** a, const float** lo);
int farmer_activation(Player* p, int layer, const float** a, const float** lo);
const uint32_t* farmer_relu_bits(Player* p, int layer);
// model_farmer.cu
int farmer_alloc(fi_learner* l, Player* p);
void farmer_free(Player* p);
int farmer_forward_backward(fi_learner* l, Player* p, const float* batch, int m, int t, int global_m);
int farmer_infer_alloc(fi_learner* l, Player* p, size_t rows, size_t t);
int farmer_infer(fi_learner* l, Player* p, const float* params, const float* z_dev, const float* x_dev, size_t rows,
                 size_t t, float* out_dev, cudaStream_t stream);
}  // namespace fi
