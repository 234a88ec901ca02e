// Learner host orchestration behind the C ABI: replaces the body of Learner::trainModel
// (reference include/freeimpala/learner.h:32-49), the Learner ctor's ring/model set-up
// (:100-140) and Model / ModelManager (data_structures.h:43-157, 310-481).
//
// One CUDA stream per player (p worker threads step concurrently on distinct players,
// learner.h:160-162), one flat fp32 arena each for parameters, gradients and the two Adam
// moments (reference parameters() order, so the published blob is the raw parameter arena),
// a publication stream that moves each new version to pinned host memory off the critical
// path, and one NCCL communicator per player for the data-parallel gradient all-reduce.
// There is no libtorch and no CPU fallback anywhere in this file.
#include "learner.cuh"

#include <dirent.h>
#include <dlfcn.h>
#include <nccl.h>
#include <sys/stat.h>

#include <cerrno>
#include <chrono>
#include <cmath>
#include <cstdlib>

using fi::ModelStore;
using fi::Player;
using fi::PublishTicket;
using fi::set_error;
using fi::TensorSpec;

// ------------------------------------------------------------------------------------------
// NCCL is bound at run time (dlopen): the library has no link-time dependency on it, and a
// process that already loaded a libnccl (e.g. through torch) shares that copy.
namespace {
struct NcclApi {
    void* handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId*) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
NcclApi& nccl() {
    static NcclApi api;
    static std::once_flag once;
    std::call_once(once, [] {
        const char* env = getenv("FI_NCCL_LIB");
        const char* names[] = {env, "libnccl.so.2", "libnccl.so"};
        for (const char* n : names) {
            if (!n) continue;
            api.handle = dlopen(n, RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);  // already in the process?
            if (!api.handle) api.handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
            if (api.handle) break;
        }
        if (!api.handle) return;
#define FI_SYM(field, name) api.field = reinterpret_cast<decltype(api.field)>(dlsym(api.handle, name))
        FI_SYM(GetUniqueId, "ncclGetUniqueId");
        FI_SYM(CommInitRank, "ncclCommInitRank");
        FI_SYM(CommDestroy, "ncclCommDestroy");
        FI_SYM(AllReduce, "ncclAllReduce");
        FI_SYM(GroupStart, "ncclGroupStart");
        FI_SYM(GroupEnd, "ncclGroupEnd");
        FI_SYM(GetErrorString, "ncclGetErrorString");
#undef FI_SYM
        api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllReduce && api.GroupStart &&
                 api.GroupEnd && api.GetErrorString;
    });
    return api;
}
#define FI_NCCL_OK(expr)                                                                          \
    do {                                                                                          \
        ncclResult_t _r = (expr);                                                                 \
        if (_r != ncclSuccess)                                                                    \
            return set_error(FI_ERR_NCCL, "%s failed: %s", #expr, nccl().GetErrorString(_r));     \
    } while (0)

// splitmix64: deterministic weight init, U(+-1/sqrt(fan_in)) like torch::nn's defaults
// (SURVEY.md 8c: the init need not be reproduced; parity tests load exported weights).
struct SplitMix {
    uint64_t s;
    uint64_t next() {
        uint64_t z = (s += 0x9E3779B97F4A7C15ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    double uniform() { return (double)(next() >> 11) * (1.0 / 9007199254740992.0); }
};

void build_tensor_table(fi_learner* l) {
    auto add = [&](size_t rows, size_t cols, int fan_in) {
        TensorSpec t;
        t.offset = l->param_count;
        t.rows = rows;
        t.cols = cols;
        t.numel = rows * (cols ? cols : 1);
        t.fan_in = fan_in;
        l->tensors.push_back(t);
        l->param_count += t.numel;
    };
    using namespace fi;
    if (l->cfg.model == FI_MODEL_FARMER_LSTM) {
        // FarmerLstmModel parameters() order (reference cmd/libtorch_bench/main.cpp:16-22):
        // lstm.weight_ih_l0, weight_hh_l0, bias_ih_l0, bias_hh_l0, dense1..6 weight, bias
        add(4 * kLstmH, kZDim, kLstmH);
        add(4 * kLstmH, kLstmH, kLstmH);
        add(4 * kLstmH, 0, kLstmH);
        add(4 * kLstmH, 0, kLstmH);
        add(kHid, kLstmH + kXDim, kLstmH + kXDim);
        add(kHid, 0, kLstmH + kXDim);
        for (int i = 0; i < 4; i++) {
            add(kHid, kHid, kHid);
            add(kHid, 0, kHid);
        }
        add(1, kHid, kHid);
        add(1, 0, kHid);
    } else {
        add(kHid, kZDim, kZDim);
        add(kHid, 0, kZDim);
        for (int i = 0; i < 4; i++) {
            add(kHid, kHid, kHid);
            add(kHid, 0, kHid);
        }
        add(kHead, kHid, kHid);
        add(kHead, 0, kHid);
    }
    l->arena_elems = (l->param_count + 3) & ~(size_t)3;
}

void CUDART_CB publish_cb(void* arg) {
    PublishTicket* t = static_cast<PublishTicket*>(arg);
    ModelStore* s = t->store;
    {
        std::unique_lock<std::shared_mutex> w(s->rw);  // the reference's shared_ptr swap (:441-451)
        s->published = t->host_index;
        s->buf_version[t->host_index] = t->version;
        s->latest_version.store(t->version);
    }
    {
        std::lock_guard<std::mutex> g(s->cv_mu);
    }
    s->cv.notify_all();
    delete t;
}

// Publication = (1) a device snapshot of the weights taken on the learner stream, (2) its D2H copy and the host-blob
// flip on the publication stream. publish_begin makes the learner stream wait until the next snapshot slot is free and
// returns it; the caller fills dev_snap[slot] on the learner stream (the fused optimiser writes it as a by-product, so the
// step has no copy-engine operation; other callers copy) and calls publish_end.
int publish_begin(Player* p, int* slot) {
    ModelStore& s = p->store;
    std::lock_guard<std::mutex> g(s.mu);
    const int sn = s.next_snap;
    if (s.snap_free_recorded[sn]) FI_CUDA_OK(cudaStreamWaitEvent(p->stream, s.snap_free[sn], 0));
    if (s.infer_recorded[sn]) FI_CUDA_OK(cudaStreamWaitEvent(p->stream, s.infer_done[sn], 0));
    *slot = sn;
    return FI_OK;
}

int publish_end(Player* p, uint64_t version, int sn) {
    ModelStore& s = p->store;
    std::lock_guard<std::mutex> g(s.mu);
    FI_CUDA_OK(cudaEventRecord(s.snap_ready[sn], p->stream));
    s.newest_snap = sn;
    s.next_snap = (sn + 1) % ModelStore::kSnaps;
    FI_CUDA_OK(cudaStreamWaitEvent(s.pub_stream, s.snap_ready[sn], 0));
    const int h = s.next_host;
    s.next_host = (h + 1) % 3;
    FI_CUDA_OK(cudaMemcpyAsync(s.host_buf[h], s.dev_snap[sn], s.bytes, cudaMemcpyDeviceToHost, s.pub_stream));
    FI_CUDA_OK(cudaEventRecord(s.snap_free[sn], s.pub_stream));
    s.snap_free_recorded[sn] = true;
    PublishTicket* t = new PublishTicket{&s, h, version};
    cudaError_t e = cudaLaunchHostFunc(s.pub_stream, publish_cb, t);
    if (e != cudaSuccess) {
        delete t;
        return set_error(FI_ERR_CUDA, "cudaLaunchHostFunc failed: %s", cudaGetErrorString(e));
    }
    return FI_OK;
}

// Enqueue the publication of the weights currently in p->params as `version` (snapshot by a device-to-device copy).
int publish_async(Player* p, uint64_t version) {
    int sn = 0;
    FI_TRY(publish_begin(p, &sn));
    FI_CUDA_OK(cudaMemcpyAsync(p->store.dev_snap[sn], p->params, p->store.bytes, cudaMemcpyDeviceToDevice, p->stream));
    return publish_end(p, version, sn);
}

// Synchronous publication (create / set_params / load): everything idle on return.
int publish_sync(Player* p, uint64_t version) {
    FI_TRY(publish_async(p, version));
    FI_CUDA_OK(cudaStreamSynchronize(p->stream));
    FI_CUDA_OK(cudaStreamSynchronize(p->store.pub_stream));
    return FI_OK;
}

Player* get_player(fi_learner* l, int player) {
    if (!l || player < 0 || player >= (int)l->players.size()) {
        set_error(FI_ERR_ARG, "invalid learner or player index %d", player);
        return nullptr;
    }
    return l->players[player];
}

void free_player(fi_learner* l, Player* p) {
    if (!p) return;
    if (p->stream) cudaStreamSynchronize(p->stream);
    if (p->store.pub_stream) cudaStreamSynchronize(p->store.pub_stream);
    if (p->infer_stream) cudaStreamSynchronize(p->infer_stream);
    if (p->graph_exec) cudaGraphExecDestroy((cudaGraphExec_t)p->graph_exec);
    if (p->graph) cudaGraphDestroy((cudaGraph_t)p->graph);
    p->graph_exec = p->graph = nullptr;
    if (p->nccl_comm && nccl().ok) nccl().CommDestroy((ncclComm_t)p->nccl_comm);
    if (l->cfg.model == FI_MODEL_FARMER_LSTM) fi::farmer_free(p);
    fi::dense_free(&p->dense);
    fi::dense_free(&p->inf_dense);
    float* dev[] = {p->params, p->grads, p->adam_m, p->adam_v, p->head, p->dhead, p->inf_in, p->inf_x, p->inf_out};
    for (float* d : dev)
        if (d) cudaFree(d);
    for (float* d : p->store.dev_snap)
        if (d) cudaFree(d);
    void* devv[] = {p->d_losses, p->gemm_ws, p->colsum_ws, p->stage_dev, p->clip_coef, p->norm_ws, p->inf_idx};
    for (void* d : devv)
        if (d) cudaFree(d);
    void* pinned[] = {p->h_losses, p->stage_host, p->inf_host_in, p->inf_host_x, p->inf_host_out, p->inf_host_idx,
                      p->store.host_buf[0], p->store.host_buf[1], p->store.host_buf[2]};
    for (void* h : pinned)
        if (h) cudaFreeHost(h);
    for (cudaEvent_t e : p->loss_ev) if (e) cudaEventDestroy(e);
    if (p->batch_ready) cudaEventDestroy(p->batch_ready);
    for (int i = 0; i < ModelStore::kSnaps; i++) {
        cudaEvent_t evs[] = {p->store.snap_ready[i], p->store.snap_free[i], p->store.infer_done[i]};
        for (cudaEvent_t e : evs)
            if (e) cudaEventDestroy(e);
    }
    if (p->stream) cudaStreamDestroy(p->stream);
    if (p->store.pub_stream) cudaStreamDestroy(p->store.pub_stream);
    if (p->infer_stream) cudaStreamDestroy(p->infer_stream);
    delete p;
}

int create_player(fi_learner* l, int index) {
    Player* p = new Player();
    p->index = index;
    l->players.push_back(p);  // owned by the learner from here on (freed by fi_learner_destroy)
    const size_t abytes = l->arena_elems * sizeof(float);
    FI_CUDA_OK(cudaStreamCreateWithFlags(&p->stream, cudaStreamNonBlocking));
    FI_CUDA_OK(cudaStreamCreateWithFlags(&p->store.pub_stream, cudaStreamNonBlocking));
    FI_CUDA_OK(cudaStreamCreateWithFlags(&p->infer_stream, cudaStreamNonBlocking));
    float** arenas[] = {&p->params, &p->grads, &p->adam_m, &p->adam_v};
    for (float** a : arenas) {
        FI_CUDA_OK(cudaMalloc((void**)a, abytes));
        FI_CUDA_OK(cudaMemset(*a, 0, abytes));
    }
    FI_CUDA_OK(cudaMalloc((void**)&p->d_losses, fi::kLossWords * sizeof(double)));
    FI_CUDA_OK(cudaMemset(p->d_losses, 0, fi::kLossWords * sizeof(double)));
    const size_t ring_bytes = (Player::kLossRing + 1) * fi::kLossWords * sizeof(double);
    FI_CUDA_OK(cudaHostAlloc((void**)&p->h_losses, ring_bytes, cudaHostAllocPortable | cudaHostAllocMapped));
    memset(p->h_losses, 0, ring_bytes);
    if (l->cfg.max_grad_norm > 0.0) {
        FI_CUDA_OK(cudaMalloc((void**)&p->clip_coef, sizeof(float)));
        FI_CUDA_OK(cudaMemset(p->clip_coef, 0, sizeof(float)));
        FI_CUDA_OK(cudaMalloc(&p->norm_ws, fi::grad_norm_scratch_bytes()));
        FI_CUDA_OK(cudaMemset(p->norm_ws, 0, fi::grad_norm_scratch_bytes()));
    }
    p->lr = l->cfg.lr;
    FI_CUDA_OK(cudaHostGetDevicePointer((void**)&p->h_losses_dev, p->h_losses, 0));
    for (cudaEvent_t& e : p->loss_ev) FI_CUDA_OK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    FI_CUDA_OK(cudaEventCreateWithFlags(&p->batch_ready, cudaEventDisableTiming));
    ModelStore& s = p->store;
    s.bytes = l->param_count * sizeof(float);
    for (int i = 0; i < ModelStore::kSnaps; i++) {
        FI_CUDA_OK(cudaMalloc((void**)&s.dev_snap[i], abytes));
        FI_CUDA_OK(cudaEventCreateWithFlags(&s.snap_ready[i], cudaEventDisableTiming));
        FI_CUDA_OK(cudaEventCreateWithFlags(&s.snap_free[i], cudaEventDisableTiming));
        FI_CUDA_OK(cudaEventCreateWithFlags(&s.infer_done[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < 3; i++) FI_CUDA_OK(cudaHostAlloc((void**)&s.host_buf[i], abytes, cudaHostAllocPortable));
    // step workspaces
    if (l->cfg.model == FI_MODEL_FARMER_LSTM) FI_TRY(fi::farmer_alloc(l, p));
    else FI_TRY(fi::ac_alloc(l, p));
    // random init, distinct per player (the reference fills each player's Model with rand(), :121-127)
    std::vector<float> init(l->arena_elems, 0.f);
    SplitMix rng{l->cfg.seed * 0x100000001B3ull + (uint64_t)index + 1};
    for (const TensorSpec& t : l->tensors) {
        const double k = 1.0 / std::sqrt((double)t.fan_in);
        for (size_t i = 0; i < t.numel; i++) init[t.offset + i] = (float)((2.0 * rng.uniform() - 1.0) * k);
    }
    FI_CUDA_OK(cudaMemcpy(p->params, init.data(), abytes, cudaMemcpyHostToDevice));
    p->version = 1;  // Model ctor: version 0, generateRandomData() -> 1 (data_structures.h:52-58,121-127)
    s.next_snap = 0;
    s.next_host = 0;
    return publish_sync(p, p->version);
}

// mkdir -p
bool make_dirs(const std::string& path) {
    if (path.empty()) return false;
    for (size_t i = 1; i <= path.size(); i++) {
        if (i != path.size() && path[i] != '/') continue;
        const std::string part = path.substr(0, i);
        if (mkdir(part.c_str(), 0777) != 0 && errno != EEXIST) return false;
    }
    struct stat st;
    return stat(path.c_str(), &st) == 0 && S_ISDIR(st.st_mode);
}

bool file_exists(const std::string& path) {
    struct stat st;
    return stat(path.c_str(), &st) == 0;
}

// optimiser-state sections of a checkpoint: Adam / AdamW / SGD (m, v = the two Adam moments) and RMSProp (m = momentum
// buffer, v = square average). The layouts are the same; the magic keeps one family's state out of the other's learner.
const char kOptMagic[8] = {'F', 'I', 'O', 'P', 'T', '0', '0', '1'};
const char kRmsMagic[8] = {'F', 'I', 'R', 'M', 'S', '0', '0', '1'};
const char* opt_magic(const fi_learner* l) { return l->cfg.optimizer == FI_OPT_RMSPROP ? kRmsMagic : kOptMagic; }

}  // namespace

extern "C" {

const char* fi_last_error(void) { return fi::last_error_ref().c_str(); }
const char* fi_version(void) { return "freeimpala-b200 0.1 (sm_100a)"; }
uint64_t fi_kernel_launch_count(void) { return fi::launch_counter().load(); }

void fi_learner_config_default(fi_learner_config* c) {
    if (!c) return;
    memset(c, 0, sizeof(*c));
    c->device = 0;
    c->num_players = 2;          // -p (reference cmd/freeimpala/main.cpp:38-120 defaults)
    c->buffer_capacity = 10;     // -B
    c->entry_size = 100;         // -S
    c->batch_size = 5;           // -M
    c->model = FI_MODEL_MLP_ACTOR_CRITIC;
    c->loss = FI_LOSS_VTRACE;
    c->optimizer = FI_OPT_ADAM;
    c->lr = 5e-4;                // README bench shape
    c->seed = 0;
    c->rho_bar = 1.f; c->c_bar = 1.f; c->pg_rho_bar = 1.f; c->lambda_ = 1.f;
    c->baseline_cost = 0.5f; c->entropy_cost = 0.01f;
    c->gemm_mode = FI_GEMM_AUTO;
    c->publish_every = 1;
    c->checkpoint_location = nullptr;
    c->max_grad_norm = 0.0;      // no clipping
    c->rmsprop_alpha = 0.99;     // torch.optim.RMSprop defaults
    c->rmsprop_eps = 1e-8;
    c->rmsprop_momentum = 0.0;
    c->legal_action_mask = 0;    // every action legal; record word 182 is not read
}

fi_learner* fi_learner_create(const fi_learner_config* cfg) {
    if (!cfg || cfg->num_players < 1 || cfg->entry_size == 0 || cfg->batch_size == 0 ||
        cfg->buffer_capacity < cfg->batch_size) {  // validateParameters: M <= B (main.cpp:160-172)
        set_error(FI_ERR_ARG, "fi_learner_create: invalid configuration (need p>=1, S>0, 0<M<=B)");
        return nullptr;
    }
    const bool farmer = cfg->model == FI_MODEL_FARMER_LSTM;
    if ((farmer && cfg->loss == FI_LOSS_VTRACE) || (!farmer && cfg->loss != FI_LOSS_VTRACE) ||
        (cfg->model != FI_MODEL_FARMER_LSTM && cfg->model != FI_MODEL_MLP_ACTOR_CRITIC)) {
        set_error(FI_ERR_ARG, "fi_learner_create: model %d does not support loss %d", cfg->model, cfg->loss);
        return nullptr;
    }
    if (cfg->optimizer < FI_OPT_ADAM || cfg->optimizer > FI_OPT_RMSPROP) {
        set_error(FI_ERR_ARG, "fi_learner_create: unknown optimizer %d", cfg->optimizer);
        return nullptr;
    }
    if (!(cfg->max_grad_norm >= 0.0) || !std::isfinite(cfg->max_grad_norm)) {
        set_error(FI_ERR_ARG, "fi_learner_create: max_grad_norm must be finite and >= 0 (0 = no clipping), got %g", cfg->max_grad_norm);
        return nullptr;
    }
    if (!(cfg->rmsprop_alpha > 0.0 && cfg->rmsprop_alpha < 1.0) || !(cfg->rmsprop_eps > 0.0) || !std::isfinite(cfg->rmsprop_eps) ||
        !(cfg->rmsprop_momentum >= 0.0 && cfg->rmsprop_momentum < 1.0)) {
        set_error(FI_ERR_ARG, "fi_learner_create: RMSProp options need 0 < rmsprop_alpha < 1, rmsprop_eps > 0 and 0 <= rmsprop_momentum < 1 "
                              "(got %g, %g, %g)", cfg->rmsprop_alpha, cfg->rmsprop_eps, cfg->rmsprop_momentum);
        return nullptr;
    }
    if (cfg->legal_action_mask != 0 && cfg->legal_action_mask != 1) {
        set_error(FI_ERR_ARG, "fi_learner_create: legal_action_mask must be 0 or 1, got %d", cfg->legal_action_mask);
        return nullptr;
    }
    if (farmer && cfg->legal_action_mask) {
        set_error(FI_ERR_ARG, "fi_learner_create: legal_action_mask needs a policy; the FarmerLstm model has none");
        return nullptr;
    }
    if (!farmer) {   // V-trace constants: a NaN or out-of-range value would otherwise surface as NaN or meaningless losses
        const struct { const char* name; float v; bool ok; const char* range; } vt[] = {
            {"rho_bar", cfg->rho_bar, cfg->rho_bar > 0.f, "> 0 (+inf = no clipping)"},
            {"c_bar", cfg->c_bar, cfg->c_bar > 0.f, "> 0 (+inf = no clipping)"},
            {"pg_rho_bar", cfg->pg_rho_bar, cfg->pg_rho_bar > 0.f, "> 0 (+inf = no clipping)"},
            {"lambda_", cfg->lambda_, cfg->lambda_ >= 0.f && cfg->lambda_ <= 1.f, "in [0, 1]"},
            {"baseline_cost", cfg->baseline_cost, cfg->baseline_cost >= 0.f && std::isfinite(cfg->baseline_cost), "finite and >= 0"},
            {"entropy_cost", cfg->entropy_cost, cfg->entropy_cost >= 0.f && std::isfinite(cfg->entropy_cost), "finite and >= 0"},
        };
        for (const auto& f : vt)
            if (!f.ok) {
                set_error(FI_ERR_ARG, "fi_learner_create: V-trace %s must be %s, got %g", f.name, f.range, (double)f.v);
                return nullptr;
            }
    }
    if (farmer && cfg->entry_size < fi::kFarmerMinEntry) {   // a shorter trajectory would train on a truncated x
        set_error(FI_ERR_ARG, "fi_learner_create: the FarmerLstm model needs entry_size >= %d (x[484] spans records 0..%d), got %zu",
                  fi::kFarmerMinEntry, fi::kFarmerMinEntry - 1, cfg->entry_size);
        return nullptr;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error(FI_ERR_CUDA, "fi_learner_create: no CUDA device (there is no CPU fallback)");
        return nullptr;
    }
    FI_CUDA_OK_NULL(cudaSetDevice(cfg->device));
    fi_learner* l = new fi_learner();
    l->cfg = *cfg;
    if (l->cfg.publish_every < 1) l->cfg.publish_every = 1;
    if (cfg->checkpoint_location) l->ckpt_dir = cfg->checkpoint_location;
    l->cfg.checkpoint_location = nullptr;
    build_tensor_table(l);
    for (int p = 0; p < cfg->num_players; p++) {
        fi_ring* r = fi_ring_create(cfg->device, cfg->entry_size, cfg->buffer_capacity);  // learner.h:135-139
        if (!r) {
            fi_learner_destroy(l);
            return nullptr;
        }
        l->rings.push_back(r);
        if (create_player(l, p) < 0) {
            fi_learner_destroy(l);
            return nullptr;
        }
    }
    return l;
}

void fi_learner_destroy(fi_learner* l) {
    if (!l) return;
    cudaSetDevice(l->cfg.device);
    for (Player* p : l->players) free_player(l, p);
    for (fi_ring* r : l->rings) fi_ring_destroy(r);
    delete l;
}

fi_ring* fi_learner_ring(fi_learner* l, int player) {
    if (!l || player < 0 || player >= (int)l->rings.size()) return nullptr;
    return l->rings[player];
}
void* fi_learner_stream(fi_learner* l, int player) {
    Player* p = get_player(l, player);
    return p ? (void*)p->stream : nullptr;
}

int fi_learner_sync(fi_learner* l, int player) {
    Player* p = get_player(l, player);
    if (!p) return FI_ERR_ARG;
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    FI_CUDA_OK(cudaStreamSynchronize(p->stream));
    FI_CUDA_OK(cudaStreamSynchronize(p->store.pub_stream));
    return FI_OK;
}

int fi_learner_stage_batch(fi_learner* l, int player, const void* host, size_t num_slots, fi_batch* out) {
    Player* p = get_player(l, player);
    if (!p || !host || !out) return set_error(FI_ERR_ARG, "fi_learner_stage_batch: null argument");
    if (num_slots == 0 || num_slots > l->cfg.batch_size)
        return set_error(FI_ERR_ARG, "fi_learner_stage_batch: num_slots %zu not in [1, batch_size=%zu]", num_slots,
                         l->cfg.batch_size);
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    const size_t slot_bytes = l->cfg.entry_size * FI_ELEMENT_SIZE, cap = l->cfg.batch_size * slot_bytes;
    const size_t n = num_slots * slot_bytes;
    if (!p->stage_dev) {
        FI_CUDA_OK(cudaMalloc((void**)&p->stage_dev, cap));
        p->stage_bytes = cap;
    }
    cudaPointerAttributes attr;
    const bool pinned = cudaPointerGetAttributes(&attr, host) == cudaSuccess && attr.type == cudaMemoryTypeHost;
    cudaGetLastError();
    const void* src = host;
    if (!pinned) {  // pageable source: bounce through a pinned buffer so the copy is a real async DMA
        if (!p->stage_host) FI_CUDA_OK(cudaHostAlloc((void**)&p->stage_host, cap, cudaHostAllocPortable));
        FI_CUDA_OK(cudaStreamSynchronize(p->stream));  // previous DMA out of the bounce buffer
        memcpy(p->stage_host, host, n);
        src = p->stage_host;
    }
    FI_CUDA_OK(cudaMemcpyAsync(p->stage_dev, src, n, cudaMemcpyHostToDevice, p->stream));
    out->dev_ptr = p->stage_dev;
    out->num_slots = num_slots;
    out->slot_bytes = slot_bytes;
    out->stream = p->stream;
    out->seq = 0;
    return FI_OK;
}

namespace {
// sum-allreduce of the flat gradient arena (+ the four loss sums) over NVLink (SURVEY.md 8e), on the player's stream
int enqueue_allreduce(fi_learner* l, Player* p) {
    if (l->dp_world <= 1) return FI_OK;
    if (!p->nccl_comm) return set_error(FI_ERR_STATE, "data parallelism configured but the communicator is missing");
    NcclApi& n = nccl();
    // timed as "nccl_allreduce_grads" (bus bytes of a ring all-reduce: 2(N-1)/N x the arena); it also absorbs the wait
    // for the slowest rank, so it reads as skew + transfer
    fi::LaunchScope ls("nccl_allreduce_grads", p->stream,
                       2.0 * (l->dp_world - 1) / l->dp_world * 4.0 * (double)l->param_count, fi::kWorkBytes);
    FI_NCCL_OK(n.GroupStart());
    FI_NCCL_OK(n.AllReduce(p->grads, p->grads, l->param_count, ncclFloat, ncclSum, (ncclComm_t)p->nccl_comm, p->stream));
    FI_NCCL_OK(n.AllReduce(p->d_losses, p->d_losses, 4, ncclDouble, ncclSum, (ncclComm_t)p->nccl_comm, p->stream));
    FI_NCCL_OK(n.GroupEnd());
    ls.done_external();
    return FI_OK;
}

struct UpdateTicket {   // the host-side bookkeeping of one optimiser step
    uint64_t steps_done;
    bool publish;
    int sn, slot;
};

// counters advance; the learner stream waits until the snapshot the optimiser kernel is about to write is free
int begin_update(fi_learner* l, Player* p, UpdateTicket* u) {
    p->opt_step++;
    u->steps_done = p->steps_done.load(std::memory_order_relaxed) + 1;
    p->version++;  // generateRandomData(): version++ (data_structures.h:121-127), then updateModel
    u->publish = u->steps_done % (uint64_t)l->cfg.publish_every == 0;
    u->sn = -1;
    if (u->publish) FI_TRY(publish_begin(p, &u->sn));
    u->slot = (int)(u->steps_done % Player::kLossRing);
    return FI_OK;
}

fi::OptConfig opt_config(const fi_learner* l, const Player* p) {
    fi::OptConfig o;
    o.kind = l->cfg.optimizer;
    o.lr = p->lr;
    o.rms_alpha = l->cfg.rmsprop_alpha;
    o.rms_eps = l->cfg.rmsprop_eps;
    o.rms_momentum = l->cfg.rmsprop_momentum;
    return o;
}

// one kernel: the update, the model store's device snapshot and the loss + gradient-norm read-back (into mapped pinned memory)
int opt_desc_for(fi_learner* l, Player* p, const UpdateTicket& u, fi::OptLaunchDesc* d) {
    return fi::opt_launch_desc(opt_config(l, p), p->opt_step, l->param_count, p->params, p->grads, p->adam_m, p->adam_v, 1.0f,
                               p->clip_coef, u.publish ? p->store.dev_snap[u.sn] : nullptr, p->d_losses,
                               p->h_losses_dev + fi::kLossWords * u.slot, d);
}

// Gradient clipping (max_grad_norm > 0): the global norm of the gradient arena and the clip coefficient, on the device, right
// before the optimiser. It runs after the all-reduce, so every data-parallel rank derives the same coefficient from the same
// reduced arena and the replicas stay identical; the optimiser applies the coefficient on the fly and leaves the arena as the
// all-reduce left it (fi_learner_get_grads returns the unclipped gradient). The norm lands in d_losses[4] and travels with the
// losses. Fixed for the learner, so the graph replays this launch unchanged.
int enqueue_clip(fi_learner* l, Player* p) {
    if (!(l->cfg.max_grad_norm > 0.0)) return FI_OK;
    return fi::launch_grad_norm_clip(l->param_count, p->grads, l->cfg.max_grad_norm, p->d_losses + 4, p->clip_coef, p->norm_ws, p->stream);
}

int finish_update(fi_learner* l, Player* p, const UpdateTicket& u) {
    (void)l;
    FI_CUDA_OK(cudaEventRecord(p->loss_ev[u.slot], p->stream));
    p->steps_done.store(u.steps_done, std::memory_order_release);   // readers (losses_at, steps_done) see the event recorded
    if (u.publish) FI_TRY(publish_end(p, p->version, u.sn));
    return FI_OK;
}

int check_batch(fi_learner* l, const fi_batch* b, const char* who) {
    if (!b) return set_error(FI_ERR_ARG, "%s: null argument", who);
    if (b->num_slots == 0 || b->num_slots > l->cfg.batch_size || b->slot_bytes != l->cfg.entry_size * FI_ELEMENT_SIZE || !b->dev_ptr)
        return set_error(FI_ERR_ARG, "%s: batch [%zu x %zu B] does not match the learner (M<=%zu, S=%zu)", who, b->num_slots, b->slot_bytes,
                         l->cfg.batch_size, l->cfg.entry_size);
    // mean losses divide by the GLOBAL batch: under data parallelism that is the sum of the ranks' configured batch sizes
    // (all-reduced once in fi_learner_dp_init; shards may differ by one trajectory), so every rank must step full batches
    if (l->dp_world > 1 && b->num_slots != l->cfg.batch_size)
        return set_error(FI_ERR_STATE, "%s: a partial batch (%zu of %zu trajectories) cannot be combined with data parallelism (the "
                                       "global batch size is fixed at fi_learner_dp_init)", who, b->num_slots, l->cfg.batch_size);
    return FI_OK;
}

// forward + loss + backward of the configured model on the player's stream (caller holds step_mu)
int enqueue_forward_backward(fi_learner* l, Player* p, const fi_batch* b) {
    const int m = (int)b->num_slots, t = (int)l->cfg.entry_size;
    const int global_m = l->dp_world > 1 ? (int)l->dp_global_batch : m;
    if (l->cfg.model == FI_MODEL_FARMER_LSTM) FI_TRY(fi::farmer_forward_backward(l, p, (const float*)b->dev_ptr, m, t, global_m));
    else FI_TRY(fi::ac_forward_backward(l, p, (const float*)b->dev_ptr, m, t, global_m));
    p->last_rows = (size_t)m * t;
    p->grads_valid = true;
    return FI_OK;
}

int wait_for_batch(Player* p, const fi_batch* b) {
    if (b->stream && (cudaStream_t)b->stream != p->stream) {  // gather ran on another stream
        FI_CUDA_OK(cudaEventRecord(p->batch_ready, (cudaStream_t)b->stream));
        FI_CUDA_OK(cudaStreamWaitEvent(p->stream, p->batch_ready, 0));
    }
    return FI_OK;
}

bool graphs_enabled() {
    static const bool on = [] { const char* e = getenv("FI_GRAPH"); return !e || atoi(e) != 0; }();
    return on;
}

void drop_graph(Player* p) {
    if (p->graph_exec) cudaGraphExecDestroy((cudaGraphExec_t)p->graph_exec);
    if (p->graph) cudaGraphDestroy((cudaGraph_t)p->graph);   // kept alive: the optimiser's node handle belongs to it
    p->graph_exec = nullptr;
    p->graph = nullptr;
    p->graph_opt_node = nullptr;
}

// The whole step -- forward, fused loss head, backward, gradient finalisation, (NCCL all-reduce,) optimiser -- as ONE CUDA
// graph launch. The launch sequence of a step is static for a given batch buffer and batch size (every workspace is allocated at
// creation, tensor maps and shapes do not change), except for the optimiser kernel's scalars: the bias corrections of the step
// count, the model-store snapshot and the loss read-back slot. That one kernel node is re-parameterised each step
// (cudaGraphExecKernelNodeSetParams); everything else replays. The step is captured the first time a (buffer, batch size) pair
// is seen after two ordinary steps (first launches set kernel attributes and fill the tensor-map cache), and again whenever
// the pair changes. Not used while per-kernel profiling is on (fi_prof_enable), or with FI_GRAPH=0.
// Why: 30 launches per step cost the host 0.2-0.5 ms of enqueue time -- more than the whole step at batch 64 x 100 (BASELINE.json
// configs[1]: 0.48 ms, launch-gap bound), and with 8 data-parallel ranks sharing 16 cores the slowest rank's enqueue jitter
// becomes everyone's step time at the all-reduce (VERDICT r1 weak #7, #9).
int step_with_graph(fi_learner* l, Player* p, const fi_batch* b, bool* used) {
    *used = false;
    if (!graphs_enabled() || p->graph_failed || fi::prof().on.load(std::memory_order_relaxed)) return FI_OK;
    if (p->steps_done.load(std::memory_order_relaxed) < 2) return FI_OK;
    const bool fresh = !p->graph_exec || p->graph_batch_ptr != b->dev_ptr || p->graph_batch_m != b->num_slots;
    FI_TRY(wait_for_batch(p, b));
    UpdateTicket u;
    FI_TRY(begin_update(l, p, &u));
    fi::OptLaunchDesc d;
    FI_TRY(opt_desc_for(l, p, u, &d));
    if (fresh) {
        drop_graph(p);
        const uint64_t n0 = fi::launch_counter().load();
        cudaGraph_t graph = nullptr;
        cudaError_t e = cudaStreamBeginCapture(p->stream, cudaStreamCaptureModeThreadLocal);
        int rc = e == cudaSuccess ? FI_OK : FI_ERR_CUDA;
        if (rc == FI_OK) rc = enqueue_forward_backward(l, p, b);
        if (rc == FI_OK) rc = enqueue_allreduce(l, p);
        if (rc == FI_OK) rc = enqueue_clip(l, p);
        if (rc == FI_OK) {
            fi::LaunchScope ls("fused_opt_kernel", p->stream, d.work_bytes, fi::kWorkBytes);
            e = cudaLaunchKernel(d.func, dim3(d.grid), dim3(d.block), d.args, 0, p->stream);
            rc = e == cudaSuccess ? ls.done() : FI_ERR_CUDA;
        }
        const cudaError_t e_end = cudaStreamEndCapture(p->stream, &graph);
        cudaGraphExec_t exec = nullptr;
        if (rc == FI_OK && e_end == cudaSuccess && graph) {
            // find the optimiser's node: the one kernel node running fused_opt_kernel
            size_t nn = 0;
            cudaGraphGetNodes(graph, nullptr, &nn);
            std::vector<cudaGraphNode_t> nodes(nn);
            cudaGraphGetNodes(graph, nodes.data(), &nn);
            cudaGraphNode_t opt_node = nullptr;
            for (cudaGraphNode_t nd : nodes) {
                cudaGraphNodeType ty;
                if (cudaGraphNodeGetType(nd, &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
                cudaKernelNodeParams kp;
                if (cudaGraphKernelNodeGetParams(nd, &kp) == cudaSuccess && kp.func == d.func) opt_node = nd;
            }
            if (opt_node && cudaGraphInstantiate(&exec, graph, 0) == cudaSuccess) {
                p->graph_exec = exec;
                p->graph = graph;
                graph = nullptr;
                p->graph_opt_node = opt_node;
                p->graph_batch_ptr = b->dev_ptr;
                p->graph_batch_m = b->num_slots;
                p->graph_kernels = fi::launch_counter().load() - n0;
                fi::launch_counter().fetch_sub(p->graph_kernels);   // counted when the graph is launched
            }
        }
        if (graph) cudaGraphDestroy(graph);
        if (!p->graph_exec) {
            // capture is not possible here (e.g. a collective that cannot be captured): run this and all later steps as
            // ordinary launches. Nothing captured has run; the host-side counters of begin_update stand.
            cudaGetLastError();
            p->graph_failed = true;
            fprintf(stderr, "[freeimpala_b200] step graph capture failed (player %d): continuing with stream launches\n", p->index);
            FI_TRY(enqueue_forward_backward(l, p, b));
            FI_TRY(enqueue_allreduce(l, p));
            FI_TRY(enqueue_clip(l, p));
            fi::LaunchScope ls("fused_opt_kernel", p->stream, d.work_bytes, fi::kWorkBytes);
            if (cudaLaunchKernel(d.func, dim3(d.grid), dim3(d.block), d.args, 0, p->stream) != cudaSuccess)
                return set_error(FI_ERR_CUDA, "launch of fused_opt_kernel failed");
            FI_TRY(ls.done());
            FI_TRY(fi::ring_note_consumed(b->dev_ptr, p->stream));
            *used = true;
            return finish_update(l, p, u);
        }
    } else {
        cudaKernelNodeParams kp = {};
        kp.func = const_cast<void*>(d.func);
        kp.gridDim = dim3(d.grid);
        kp.blockDim = dim3(d.block);
        kp.sharedMemBytes = 0;
        kp.kernelParams = d.args;
        kp.extra = nullptr;
        FI_CUDA_OK(cudaGraphExecKernelNodeSetParams((cudaGraphExec_t)p->graph_exec, (cudaGraphNode_t)p->graph_opt_node, &kp));
        p->last_rows = b->num_slots * l->cfg.entry_size;
        p->grads_valid = true;
    }
    FI_CUDA_OK(cudaGraphLaunch((cudaGraphExec_t)p->graph_exec, p->stream));
    fi::count_launch(p->graph_kernels);
    // the batch buffer may be rewritten by its ring's next gather once everything enqueued above has read it
    FI_TRY(fi::ring_note_consumed(b->dev_ptr, p->stream));
    *used = true;
    return finish_update(l, p, u);
}
}  // namespace

int fi_learner_forward_backward(fi_learner* l, int player, const fi_batch* b) {
    Player* p = get_player(l, player);
    if (!p) return FI_ERR_ARG;
    FI_TRY(check_batch(l, b, "fi_learner_forward_backward"));
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    std::lock_guard<std::mutex> step_lock(p->step_mu);
    FI_TRY(wait_for_batch(p, b));
    FI_TRY(enqueue_forward_backward(l, p, b));
    // the batch buffer may be rewritten by its ring's next gather once everything enqueued above has read it
    return fi::ring_note_consumed(b->dev_ptr, p->stream);
}

int fi_learner_apply_update(fi_learner* l, int player) {
    Player* p = get_player(l, player);
    if (!p) return FI_ERR_ARG;
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    std::lock_guard<std::mutex> step_lock(p->step_mu);
    FI_TRY(enqueue_allreduce(l, p));
    UpdateTicket u;
    FI_TRY(begin_update(l, p, &u));
    FI_TRY(enqueue_clip(l, p));
    FI_TRY(fi::launch_opt(opt_config(l, p), p->opt_step, l->param_count, p->params, p->grads, p->adam_m, p->adam_v, 1.0f,
                          p->stream, p->clip_coef, u.publish ? p->store.dev_snap[u.sn] : nullptr, p->d_losses,
                          p->h_losses_dev + fi::kLossWords * u.slot));
    return finish_update(l, p, u);
}

int fi_learner_step(fi_learner* l, int player, const fi_batch* batch) {
    Player* p = get_player(l, player);
    if (!p) return FI_ERR_ARG;
    FI_TRY(check_batch(l, batch, "fi_learner_step"));
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    {
        std::lock_guard<std::mutex> step_lock(p->step_mu);
        bool used = false;
        FI_TRY(step_with_graph(l, p, batch, &used));
        if (used) return FI_OK;
    }
    FI_TRY(fi_learner_forward_backward(l, player, batch));
    return fi_learner_apply_update(l, player);
}

int fi_learner_last_losses(fi_learner* l, int player, float losses[4]) {
    Player* p = get_player(l, player);
    if (!p || !losses) return set_error(FI_ERR_ARG, "fi_learner_last_losses: null argument");
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    const uint64_t done = p->steps_done.load(std::memory_order_acquire);
    const int slot = (int)(done % Player::kLossRing);
    if (done == 0 && p->grads_valid) {  // forward_backward only: read straight from the device
        FI_CUDA_OK(cudaMemcpyAsync(p->h_losses, p->d_losses, 4 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
        FI_CUDA_OK(cudaEventRecord(p->loss_ev[0], p->stream));
    }
    FI_CUDA_OK(cudaEventSynchronize(p->loss_ev[slot]));
    for (int i = 0; i < 4; i++) losses[i] = (float)p->h_losses[fi::kLossWords * slot + i];
    return FI_OK;
}
int fi_learner_losses_at(fi_learner* l, int player, uint64_t step, float losses[4]) {
    Player* p = get_player(l, player);
    if (!p || !losses) return set_error(FI_ERR_ARG, "fi_learner_losses_at: null argument");
    const uint64_t done = p->steps_done.load(std::memory_order_acquire);   // the worker thread increments it under step_mu
    if (step == 0 || step > done || step + Player::kLossRing <= done)
        return set_error(FI_ERR_ARG, "fi_learner_losses_at: step %llu is not among the last %d of %llu", (unsigned long long)step,
                         Player::kLossRing, (unsigned long long)done);
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    const int slot = (int)(step % Player::kLossRing);
    FI_CUDA_OK(cudaEventSynchronize(p->loss_ev[slot]));
    for (int i = 0; i < 4; i++) losses[i] = (float)p->h_losses[fi::kLossWords * slot + i];
    return FI_OK;
}
int fi_learner_last_losses_f64(fi_learner* l, int player, double losses[4]) {
    Player* p = get_player(l, player);
    if (!p || !losses) return set_error(FI_ERR_ARG, "fi_learner_last_losses_f64: null argument");
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    double* scratch = p->h_losses + fi::kLossWords * Player::kLossRing;  // scratch slot behind the ring
    FI_CUDA_OK(cudaMemcpyAsync(scratch, p->d_losses, 4 * sizeof(double), cudaMemcpyDeviceToHost, p->stream));
    FI_CUDA_OK(cudaStreamSynchronize(p->stream));
    for (int i = 0; i < 4; i++) losses[i] = scratch[i];
    return FI_OK;
}
int fi_learner_grad_norm_at(fi_learner* l, int player, uint64_t step, double* norm) {
    Player* p = get_player(l, player);
    if (!p || !norm) return set_error(FI_ERR_ARG, "fi_learner_grad_norm_at: null argument");
    if (!(l->cfg.max_grad_norm > 0.0)) return set_error(FI_ERR_STATE, "fi_learner_grad_norm_at: the learner does not clip (max_grad_norm = 0)");
    const uint64_t done = p->steps_done.load(std::memory_order_acquire);
    if (step == 0 || step > done || step + Player::kLossRing <= done)
        return set_error(FI_ERR_ARG, "fi_learner_grad_norm_at: step %llu is not among the last %d of %llu", (unsigned long long)step,
                         Player::kLossRing, (unsigned long long)done);
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    const int slot = (int)(step % Player::kLossRing);
    FI_CUDA_OK(cudaEventSynchronize(p->loss_ev[slot]));
    *norm = p->h_losses[fi::kLossWords * slot + 4];
    return FI_OK;
}
int fi_learner_set_lr(fi_learner* l, int player, double lr) {
    Player* p = get_player(l, player);
    if (!p) return FI_ERR_ARG;
    if (!(lr >= 0.0) || !std::isfinite(lr)) return set_error(FI_ERR_ARG, "fi_learner_set_lr: lr must be finite and >= 0, got %g", lr);
    std::lock_guard<std::mutex> step_lock(p->step_mu);   // the next update (graph or stream) reads it under the same lock
    p->lr = lr;
    return FI_OK;
}
uint64_t fi_learner_steps_done(fi_learner* l, int player) {
    Player* p = get_player(l, player);
    return p ? p->steps_done.load(std::memory_order_acquire) : 0;
}

size_t fi_learner_param_count(const fi_learner* l) { return l ? l->param_count : 0; }
int fi_learner_num_tensors(const fi_learner* l) { return l ? (int)l->tensors.size() : 0; }
int fi_learner_tensor_info(const fi_learner* l, int i, size_t* offset, size_t* numel, size_t* rows, size_t* cols) {
    if (!l || i < 0 || i >= (int)l->tensors.size()) return set_error(FI_ERR_ARG, "fi_learner_tensor_info: bad index");
    const TensorSpec& t = l->tensors[i];
    if (offset) *offset = t.offset;
    if (numel) *numel = t.numel;
    if (rows) *rows = t.rows;
    if (cols) *cols = t.cols;
    return FI_OK;
}

static int arena_io(fi_learner* l, int player, float* host_out, const float* host_in, size_t n, int which) {
    Player* p = get_player(l, player);
    if (!p || (!host_out && !host_in)) return set_error(FI_ERR_ARG, "arena access: null argument");
    if (n != l->param_count) return set_error(FI_ERR_ARG, "arena access: n=%zu but the model has %zu parameters", n, l->param_count);
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    std::lock_guard<std::mutex> step_lock(p->step_mu);
    float* arena = which == 0 ? p->params : which == 1 ? p->grads : which == 2 ? p->adam_m : p->adam_v;
    FI_CUDA_OK(cudaStreamSynchronize(p->stream));
    if (host_out) FI_CUDA_OK(cudaMemcpy(host_out, arena, n * sizeof(float), cudaMemcpyDeviceToHost));
    else FI_CUDA_OK(cudaMemcpy(arena, host_in, n * sizeof(float), cudaMemcpyHostToDevice));
    if (host_in && which == 0) FI_TRY(publish_sync(p, p->version));  // actors see the loaded weights
    return FI_OK;
}
int fi_learner_set_params(fi_learner* l, int player, const float* host, size_t n) { return arena_io(l, player, nullptr, host, n, 0); }
int fi_learner_get_params(fi_learner* l, int player, float* host, size_t n) { return arena_io(l, player, host, nullptr, n, 0); }
int fi_learner_get_grads(fi_learner* l, int player, float* host, size_t n) { return arena_io(l, player, host, nullptr, n, 1); }
int fi_learner_set_grads(fi_learner* l, int player, const float* host, size_t n) { return arena_io(l, player, nullptr, host, n, 1); }
int fi_learner_get_opt_state(fi_learner* l, int player, float* m, float* v, size_t n, int64_t* step) {
    Player* p = get_player(l, player);
    if (!p) return FI_ERR_ARG;
    if (m) FI_TRY(arena_io(l, player, m, nullptr, n, 2));
    if (v) FI_TRY(arena_io(l, player, v, nullptr, n, 3));
    if (step) *step = p->opt_step;
    return FI_OK;
}
void* fi_learner_grad_ptr(fi_learner* l, int player) {
    Player* p = get_player(l, player);
    return p ? p->grads : nullptr;
}
void* fi_learner_param_ptr(fi_learner* l, int player) {
    Player* p = get_player(l, player);
    return p ? p->params : nullptr;
}

// ---- batched actor policy inference (SURVEY.md 8f rank 2) --------------------------------
// The hook is the comment in Agent::simulateGame (reference include/freeimpala/agent.h:52-56): every actor asks, for its
// player, for the policy at its current observations. Concurrent callers are COMBINED: requests queue per player, the
// first caller that finds no forward in flight becomes the leader, takes everything that is pending (up to
// kInferMaxRows), packs the observations into one pinned buffer, and runs ONE host->device copy, ONE forward on the
// newest published snapshot of the weights, ONE device->host copy and one stream synchronisation for the whole batch;
// the other callers sleep on a condition variable and find their rows filled in. While a forward runs the next batch
// accumulates, so 64 actors cost about two forwards per round instead of 64 (round 1: one synchronous forward per
// caller under a mutex). Batches of kInferTcRows rows or more run the tensor-core forward of the learner step.
namespace {
constexpr size_t kInferMaxRows = 16384;

int run_infer_batch(fi_learner* l, Player* p, const std::vector<fi::InferReq*>& batch, size_t rows, size_t t) {
    const bool farmer = l->cfg.model == FI_MODEL_FARMER_LSTM;
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    size_t states = 0;
    bool want_best = false;
    for (const fi::InferReq* q : batch) {
        states += q->states;
        want_best |= q->best != nullptr;
    }
    // the farmer model uploads z once per state, the actor-critic one observation per row
    const size_t row_in = farmer ? t * fi::kZDim : fi::kZDim;
    const size_t in_elems = (farmer ? states : rows) * row_in;
    if (rows > p->inf_rows_cap || (farmer && (states > p->inf_states_cap || t > p->inf_t_cap))) {  // grow (with head-room)
        auto grow = [](size_t cap, size_t need) {
            cap = cap ? cap : 64;
            while (cap < need) cap *= 2;
            return cap;
        };
        const size_t cap = grow(p->inf_rows_cap, rows);
        const size_t scap = farmer ? grow(p->inf_states_cap, states) : 0;
        const size_t tcap = farmer ? (t > p->inf_t_cap ? t : p->inf_t_cap) : 0;
        const size_t cap_in = farmer ? scap * tcap * fi::kZDim : cap * fi::kZDim;
        const size_t cap_out = farmer ? cap + scap : cap * fi::kHead;   // farmer: values, then best
        FI_CUDA_OK(cudaStreamSynchronize(p->infer_stream));
        if (p->inf_in) cudaFree(p->inf_in);
        if (p->inf_x) cudaFree(p->inf_x);
        if (p->inf_out) cudaFree(p->inf_out);
        if (p->inf_idx) cudaFree(p->inf_idx);
        if (p->inf_host_in) cudaFreeHost(p->inf_host_in);
        if (p->inf_host_x) cudaFreeHost(p->inf_host_x);
        if (p->inf_host_out) cudaFreeHost(p->inf_host_out);
        if (p->inf_host_idx) cudaFreeHost(p->inf_host_idx);
        p->inf_in = p->inf_x = p->inf_out = p->inf_host_in = p->inf_host_x = p->inf_host_out = nullptr;
        p->inf_idx = p->inf_host_idx = nullptr;
        p->inf_rows_cap = p->inf_states_cap = 0;
        FI_CUDA_OK(cudaMalloc((void**)&p->inf_in, cap_in * sizeof(float)));
        FI_CUDA_OK(cudaHostAlloc((void**)&p->inf_host_in, cap_in * sizeof(float), cudaHostAllocPortable));
        FI_CUDA_OK(cudaMalloc((void**)&p->inf_out, cap_out * sizeof(float)));
        FI_CUDA_OK(cudaHostAlloc((void**)&p->inf_host_out, cap_out * sizeof(float), cudaHostAllocPortable));
        if (farmer) {
            const size_t cap_idx = scap + 1 + cap;
            FI_CUDA_OK(cudaMalloc((void**)&p->inf_x, cap * fi::kXDim * sizeof(float)));
            FI_CUDA_OK(cudaHostAlloc((void**)&p->inf_host_x, cap * fi::kXDim * sizeof(float), cudaHostAllocPortable));
            FI_CUDA_OK(cudaMalloc((void**)&p->inf_idx, cap_idx * sizeof(uint32_t)));
            FI_CUDA_OK(cudaHostAlloc((void**)&p->inf_host_idx, cap_idx * sizeof(uint32_t), cudaHostAllocPortable));
            FI_TRY(fi::farmer_infer_alloc(l, p, scap, cap, tcap));
        } else {
            FI_TRY(fi::ac_infer_alloc(l, p, cap));
        }
        p->inf_rows_cap = cap;
        p->inf_states_cap = scap;
        p->inf_t_cap = tcap;
    }
    cudaStream_t st = p->infer_stream;
    uint32_t* const off = p->inf_host_idx;              // farmer: the batch's offsets [states + 1] ...
    uint32_t* const row_state = off ? off + states + 1 : nullptr;   // ... then the state of each candidate row [rows]
    size_t r0 = 0, s0 = 0;
    for (const fi::InferReq* q : batch) {   // pack the callers' states and rows back to back, their offsets rebased
        memcpy(p->inf_host_in + (farmer ? s0 : r0) * row_in, q->obs, (farmer ? q->states : q->rows) * row_in * sizeof(float));
        if (farmer) {
            memcpy(p->inf_host_x + r0 * fi::kXDim, q->x, q->rows * fi::kXDim * sizeof(float));
            for (size_t s = 0; s < q->states; s++) {
                const size_t b = q->offsets ? q->offsets[s] : s, e = q->offsets ? q->offsets[s + 1] : s + 1;
                off[s0 + s] = (uint32_t)(r0 + b);
                for (size_t r = b; r < e; r++) row_state[r0 + r] = (uint32_t)(s0 + s);
            }
        }
        r0 += q->rows;
        s0 += q->states;
    }
    FI_CUDA_OK(cudaMemcpyAsync(p->inf_in, p->inf_host_in, in_elems * sizeof(float), cudaMemcpyHostToDevice, st));
    if (farmer) {
        off[states] = (uint32_t)rows;
        FI_CUDA_OK(cudaMemcpyAsync(p->inf_x, p->inf_host_x, rows * fi::kXDim * sizeof(float), cudaMemcpyHostToDevice, st));
        FI_CUDA_OK(cudaMemcpyAsync(p->inf_idx, off, (states + 1 + rows) * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    }
    int32_t* const best_dev = want_best ? reinterpret_cast<int32_t*>(p->inf_out + rows) : nullptr;
    {
        ModelStore& s = p->store;
        std::lock_guard<std::mutex> g(s.mu);  // pins the newest snapshot against the learner's next write into it
        const int sn = s.newest_snap;
        FI_CUDA_OK(cudaStreamWaitEvent(st, s.snap_ready[sn], 0));
        if (farmer)
            FI_TRY(fi::farmer_infer(l, p, s.dev_snap[sn], p->inf_in, p->inf_x, p->inf_idx, p->inf_idx + states + 1, states, rows, t,
                                    p->inf_out, best_dev, st));
        else
            FI_TRY(fi::ac_infer(l, p, s.dev_snap[sn], p->inf_in, rows, p->inf_out, st));
        FI_CUDA_OK(cudaEventRecord(s.infer_done[sn], st));
        s.infer_recorded[sn] = true;
    }
    const size_t out_elems = farmer ? rows + (want_best ? states : 0) : rows * fi::kHead;
    FI_CUDA_OK(cudaMemcpyAsync(p->inf_host_out, p->inf_out, out_elems * sizeof(float), cudaMemcpyDeviceToHost, st));
    FI_CUDA_OK(cudaStreamSynchronize(st));   // one synchronisation per BATCH: the callers need their rows on the host
    const int32_t* const best_host = reinterpret_cast<const int32_t*>(p->inf_host_out + rows);
    r0 = s0 = 0;
    for (const fi::InferReq* q : batch) {
        if (farmer) {
            if (q->values) memcpy(q->values, p->inf_host_out + r0, q->rows * sizeof(float));
            if (q->best) memcpy(q->best, best_host + s0, q->states * sizeof(int32_t));
        } else {
            for (size_t r = 0; r < q->rows; r++) {
                const float* o = p->inf_host_out + (r0 + r) * fi::kHead;
                if (q->logits) memcpy(q->logits + r * fi::kNumActions, o, fi::kNumActions * sizeof(float));
                if (q->values) q->values[r] = o[fi::kNumActions];
            }
        }
        r0 += q->rows;
        s0 += q->states;
    }
    return FI_OK;
}

// Queues `req` on its player and waits for it: the first caller that finds no forward in flight becomes the leader and runs
// everything pending that fits one forward (the farmer model batches equal sequence lengths).
int submit_infer(fi_learner* l, Player* p, fi::InferReq& req) {
    std::unique_lock<std::mutex> lk(p->infer_mu);
    p->infer_pending.push_back(&req);
    p->infer_calls++;
    while (!req.done) {
        if (p->infer_busy) {   // a forward is in flight: this request rides in the next batch
            p->infer_cv.wait(lk);
            continue;
        }
        p->infer_busy = true;
        std::vector<fi::InferReq*> batch;
        size_t total = 0;
        const size_t bt = p->infer_pending.front()->t;
        for (auto it = p->infer_pending.begin(); it != p->infer_pending.end();) {
            if ((*it)->t == bt && total + (*it)->rows <= kInferMaxRows) {
                total += (*it)->rows;
                batch.push_back(*it);
                it = p->infer_pending.erase(it);
            } else {
                ++it;
            }
        }
        lk.unlock();
        const int rc = run_infer_batch(l, p, batch, total, bt);
        lk.lock();
        for (fi::InferReq* q : batch) {
            q->status = rc;
            q->done = true;
        }
        p->infer_batches++;
        p->infer_rows += total;
        p->infer_busy = false;
        p->infer_cv.notify_all();
    }
    return req.status;
}
}  // namespace

int fi_learner_infer(fi_learner* l, int player, const float* obs_or_z, const float* x, size_t rows, size_t t,
                     float* logits, float* values) {
    Player* p = get_player(l, player);
    if (!p || !obs_or_z || rows == 0) return set_error(FI_ERR_ARG, "fi_learner_infer: null argument");
    const bool farmer = l->cfg.model == FI_MODEL_FARMER_LSTM;
    if (farmer && (!x || t == 0 || !values)) return set_error(FI_ERR_ARG, "fi_learner_infer: the farmer model needs z, x, t and values");
    if (rows > kInferMaxRows) return set_error(FI_ERR_ARG, "fi_learner_infer: at most %zu rows per call", kInferMaxRows);
    fi::InferReq req{obs_or_z, x, rows, farmer ? t : 0, rows, nullptr, logits, values, nullptr, FI_OK, false};
    return submit_infer(l, p, req);
}

int fi_learner_infer_grouped(fi_learner* l, int player, const float* z, size_t states, size_t t, const float* x,
                             const uint32_t* offsets, float* values, int32_t* best) {
    Player* p = get_player(l, player);
    if (!p) return set_error(FI_ERR_ARG, "fi_learner_infer_grouped: no player %d", player);
    if (l->cfg.model != FI_MODEL_FARMER_LSTM) return set_error(FI_ERR_ARG, "fi_learner_infer_grouped: FarmerLstm model only");
    if (!z || !x || !offsets || (!values && !best))
        return set_error(FI_ERR_ARG, "fi_learner_infer_grouped: z, x, offsets and one of values / best are required");
    if (states == 0 || t == 0) return set_error(FI_ERR_ARG, "fi_learner_infer_grouped: states and t must be positive");
    if (states > kInferMaxRows) return set_error(FI_ERR_ARG, "fi_learner_infer_grouped: at most %zu rows per call", kInferMaxRows);
    if (offsets[0] != 0) return set_error(FI_ERR_ARG, "fi_learner_infer_grouped: offsets[0] must be 0");
    for (size_t s = 0; s < states; s++)
        if (offsets[s + 1] <= offsets[s])
            return set_error(FI_ERR_ARG, "fi_learner_infer_grouped: offsets must increase strictly (state %zu has no candidate)", s);
    const size_t rows = offsets[states];
    if (rows > kInferMaxRows) return set_error(FI_ERR_ARG, "fi_learner_infer_grouped: %zu rows, at most %zu per call", rows, kInferMaxRows);
    fi::InferReq req{z, x, rows, t, states, offsets, nullptr, values, best, FI_OK, false};
    return submit_infer(l, p, req);
}

int fi_learner_infer_stats(fi_learner* l, int player, uint64_t* calls, uint64_t* batches, uint64_t* rows) {
    Player* p = get_player(l, player);
    if (!p) return FI_ERR_ARG;
    std::lock_guard<std::mutex> lk(p->infer_mu);
    if (calls) *calls = p->infer_calls;
    if (batches) *batches = p->infer_batches;
    if (rows) *rows = p->infer_rows;
    return FI_OK;
}

// ---- model store -----------------------------------------------------------------------------
size_t fi_model_bytes(const fi_learner* l) { return l ? l->param_count * sizeof(float) : 0; }

uint64_t fi_model_version(fi_learner* l, int player) {
    Player* p = get_player(l, player);
    return p ? p->store.latest_version.load() : 0;  // getLatestVersion: 0 for a bad index (:475-480)
}

int fi_model_get(fi_learner* l, int player, void* dst, size_t n, uint64_t* version) {
    Player* p = get_player(l, player);
    if (!p || !dst) return set_error(FI_ERR_ARG, "fi_model_get: null argument");
    ModelStore& s = p->store;
    if (n < s.bytes) return set_error(FI_ERR_ARG, "fi_model_get: buffer of %zu B is smaller than the %zu B blob", n, s.bytes);
    std::shared_lock<std::shared_mutex> r(s.rw);
    memcpy(dst, s.host_buf[s.published], s.bytes);
    if (version) *version = s.buf_version[s.published];
    return FI_OK;
}

int fi_model_wait_update(fi_learner* l, int player, uint64_t current_version, int timeout_ms) {
    Player* p = get_player(l, player);
    if (!p) return 0;
    ModelStore& s = p->store;
    std::unique_lock<std::mutex> lock(s.cv_mu);
    if (s.latest_version.load() > current_version) return 1;
    return s.cv.wait_for(lock, std::chrono::milliseconds(timeout_ms),
                         [&] { return s.latest_version.load() > current_version; }) ? 1 : 0;
}

int fi_model_save(fi_learner* l, int player, uint64_t iteration, int with_optimizer_state) {
    Player* p = get_player(l, player);
    if (!p) return FI_ERR_ARG;
    if (l->ckpt_dir.empty()) return set_error(FI_ERR_IO, "fi_model_save: no checkpoint location configured");
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    ModelStore& s = p->store;
    std::vector<unsigned char> blob(s.bytes);
    std::vector<float> om, ov;
    uint64_t version = 0, opt_step = 0;
    if (with_optimizer_state) {  // consistent (weights, m, v, step): quiesce the player's stream
        std::lock_guard<std::mutex> step_lock(p->step_mu);
        FI_CUDA_OK(cudaStreamSynchronize(p->stream));
        om.resize(l->param_count);
        ov.resize(l->param_count);
        FI_CUDA_OK(cudaMemcpy(blob.data(), p->params, s.bytes, cudaMemcpyDeviceToHost));
        FI_CUDA_OK(cudaMemcpy(om.data(), p->adam_m, s.bytes, cudaMemcpyDeviceToHost));
        FI_CUDA_OK(cudaMemcpy(ov.data(), p->adam_v, s.bytes, cudaMemcpyDeviceToHost));
        version = p->version;
        opt_step = (uint64_t)p->opt_step;
    } else {  // the published model, as the reference's saveModel copies models[p] (:396)
        std::shared_lock<std::shared_mutex> r(s.rw);
        memcpy(blob.data(), s.host_buf[s.published], s.bytes);
        version = s.buf_version[s.published];
    }
    uint64_t stamp = iteration;
    if (iteration == 0) {  // :405
        std::lock_guard<std::mutex> g(s.mu);
        stamp = p->checkpoint_counter++;
    }
    // create_directories (data_structures.h:94-97): every missing component of the path
    if (!make_dirs(l->ckpt_dir)) return set_error(FI_ERR_IO, "fi_model_save: cannot create directory %s", l->ckpt_dir.c_str());
    const std::string base = l->ckpt_dir + "/model_" + std::to_string(player) + "_";
    const std::string paths[2] = {base + std::to_string(stamp) + ".bin", base + "latest.bin"};
    // One save per player at a time, and every file appears under its final name only when it is complete (written to a
    // temporary name in the same directory, then rename()d): a checkpoint thread and the final save of stop() can no
    // longer interleave their writes into one latest.bin (ADVICE r1).
    std::lock_guard<std::mutex> save_lock(p->save_mu);
    for (const std::string& final_path : paths) {
        const std::string path = final_path + ".tmp";
        FILE* f = fopen(path.c_str(), "wb");
        if (!f) return set_error(FI_ERR_IO, "fi_model_save: cannot open %s", path.c_str());
        bool ok = fwrite(&version, sizeof(version), 1, f) == 1 && fwrite(blob.data(), 1, blob.size(), f) == blob.size();
        if (ok && with_optimizer_state) {
            const uint64_t n = l->param_count;
            ok = fwrite(opt_magic(l), 1, 8, f) == 8 && fwrite(&opt_step, 8, 1, f) == 1 && fwrite(&n, 8, 1, f) == 1 &&
                 fwrite(om.data(), 4, n, f) == n && fwrite(ov.data(), 4, n, f) == n;
        }
        ok = (fclose(f) == 0) && ok;
        if (!ok) {
            remove(path.c_str());
            return set_error(FI_ERR_IO, "fi_model_save: short write to %s", path.c_str());
        }
        if (rename(path.c_str(), final_path.c_str()) != 0)
            return set_error(FI_ERR_IO, "fi_model_save: cannot rename %s to %s", path.c_str(), final_path.c_str());
    }
    return FI_OK;
}

int fi_model_load(fi_learner* l, const char* dir) {
    if (!l) return FI_ERR_ARG;
    if (!dir || !*dir) return 0;  // loadModels: empty path is a no-op (:338)
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    int loaded = 0;
    for (int pi = 0; pi < (int)l->players.size(); pi++) {
        Player* p = l->players[pi];
        const std::string prefix = "model_" + std::to_string(pi) + "_";
        std::string path = std::string(dir) + "/" + prefix + "latest.bin";
        if (!file_exists(path)) {  // highest-numbered model_{p}_N.bin (:344-376)
            uint64_t best = 0;
            std::string best_file;
            if (DIR* d = opendir(dir)) {
                while (dirent* e = readdir(d)) {
                    const std::string name = e->d_name;
                    if (name.compare(0, prefix.size(), prefix) != 0) continue;
                    const size_t end = name.find(".bin");
                    if (end == std::string::npos) continue;
                    const std::string num = name.substr(prefix.size(), end - prefix.size());
                    if (num.empty() || num.find_first_not_of("0123456789") != std::string::npos) continue;
                    const uint64_t it = strtoull(num.c_str(), nullptr, 10);
                    if (it > best) {
                        best = it;
                        best_file = std::string(dir) + "/" + name;
                    }
                }
                closedir(d);
            }
            if (best_file.empty()) continue;
            path = best_file;
            p->checkpoint_counter = best + 1;  // :373
        }
        FILE* f = fopen(path.c_str(), "rb");
        if (!f) continue;
        uint64_t version = 0;
        std::vector<float> blob(l->param_count);
        bool ok = fread(&version, 8, 1, f) == 1 && fread(blob.data(), 4, l->param_count, f) == l->param_count;
        if (!ok) {  // loadFromDisk returns false on a short file and the model keeps its state (:75-84)
            fclose(f);
            continue;
        }
        char magic[8];
        uint64_t opt_step = 0, n = 0;
        std::vector<float> om, ov;
        const bool have_magic = fread(magic, 1, 8, f) == 8;
        const char* other = opt_magic(l) == kOptMagic ? kRmsMagic : kOptMagic;
        if (have_magic && memcmp(magic, other, 8) == 0)   // never read one optimiser family's state as the other's
            fprintf(stderr, "[freeimpala_b200] %s: optimiser state written by %s, this learner runs %s: loaded the weights only\n",
                    path.c_str(), other == kRmsMagic ? "RMSProp" : "Adam/AdamW/SGD", other == kRmsMagic ? "Adam/AdamW/SGD" : "RMSProp");
        bool have_opt = have_magic && memcmp(magic, opt_magic(l), 8) == 0 && fread(&opt_step, 8, 1, f) == 1 &&
                        fread(&n, 8, 1, f) == 1 && n == l->param_count;
        if (have_opt) {
            om.resize(n);
            ov.resize(n);
            have_opt = fread(om.data(), 4, n, f) == n && fread(ov.data(), 4, n, f) == n;
        }
        fclose(f);
        std::lock_guard<std::mutex> step_lock(p->step_mu);
        FI_CUDA_OK(cudaStreamSynchronize(p->stream));
        FI_CUDA_OK(cudaMemcpy(p->params, blob.data(), l->param_count * 4, cudaMemcpyHostToDevice));
        if (have_opt) {
            FI_CUDA_OK(cudaMemcpy(p->adam_m, om.data(), n * 4, cudaMemcpyHostToDevice));
            FI_CUDA_OK(cudaMemcpy(p->adam_v, ov.data(), n * 4, cudaMemcpyHostToDevice));
            p->opt_step = (int64_t)opt_step;
        }
        p->version = version;
        FI_TRY(publish_sync(p, version));
        loaded++;
    }
    return loaded;
}

// ---- data parallelism ------------------------------------------------------------------------
int fi_dp_create_id(void* id_out) {
    if (!id_out) return set_error(FI_ERR_ARG, "fi_dp_create_id: null argument");
    if (!nccl().ok) return set_error(FI_ERR_NCCL, "NCCL library not found (set FI_NCCL_LIB)");
    static_assert(sizeof(ncclUniqueId) == FI_DP_ID_BYTES, "id size");
    ncclUniqueId id;
    FI_NCCL_OK(nccl().GetUniqueId(&id));
    memcpy(id_out, &id, sizeof(id));
    return FI_OK;
}

int fi_learner_dp_init(fi_learner* l, const void* ids, int rank, int world_size) {
    if (!l || !ids || world_size < 1 || rank < 0 || rank >= world_size)
        return set_error(FI_ERR_ARG, "fi_learner_dp_init: bad arguments");
    if (l->dp_world > 1) return set_error(FI_ERR_STATE, "fi_learner_dp_init: already initialised");
    if (!nccl().ok) return set_error(FI_ERR_NCCL, "NCCL library not found (set FI_NCCL_LIB)");
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    for (size_t pi = 0; pi < l->players.size(); pi++) {
        ncclUniqueId id;
        memcpy(&id, (const char*)ids + pi * FI_DP_ID_BYTES, sizeof(id));
        ncclComm_t comm = nullptr;
        FI_NCCL_OK(nccl().CommInitRank(&comm, world_size, id, rank));
        l->players[pi]->nccl_comm = comm;
    }
    l->dp_rank = rank;
    l->dp_world = world_size;
    // the global batch = sum of the ranks' batch sizes (shards of a global batch may differ by one: dp.shard_range)
    l->dp_global_batch = l->cfg.batch_size * (size_t)world_size;
    if (world_size > 1) {
        Player* p0 = l->players[0];
        double* d = nullptr;
        FI_CUDA_OK(cudaMalloc((void**)&d, sizeof(double)));
        const double mine = (double)l->cfg.batch_size;
        FI_CUDA_OK(cudaMemcpyAsync(d, &mine, sizeof(double), cudaMemcpyHostToDevice, p0->stream));
        FI_NCCL_OK(nccl().AllReduce(d, d, 1, ncclDouble, ncclSum, (ncclComm_t)p0->nccl_comm, p0->stream));
        double total = 0.0;
        FI_CUDA_OK(cudaMemcpyAsync(&total, d, sizeof(double), cudaMemcpyDeviceToHost, p0->stream));
        FI_CUDA_OK(cudaStreamSynchronize(p0->stream));
        cudaFree(d);
        l->dp_global_batch = (size_t)(total + 0.5);
    }
    return FI_OK;
}
int fi_learner_dp_world(const fi_learner* l) { return l ? l->dp_world : 0; }

// ---- inspection (parity tests) ---------------------------------------------------------------
__global__ void relu_mask_kernel(const float* __restrict__ a, const float* __restrict__ lo, size_t n,
                                 unsigned char* __restrict__ out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = (a[i] > 0.f || (lo && lo[i] > 0.f)) ? 1 : 0;
}

__global__ void relu_bits_expand_kernel(const uint32_t* __restrict__ bits, size_t n, unsigned char* __restrict__ out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = (bits[i >> 5] >> (i & 31)) & 1u;   // rows of 512 columns = 16 words: element i lives in word i / 32
}

int fi_learner_debug_relu_masks(fi_learner* l, int player, unsigned char* host, size_t n) {
    Player* p = get_player(l, player);
    if (!p || !host) return set_error(FI_ERR_ARG, "fi_learner_debug_relu_masks: null argument");
    const bool farmer = l->cfg.model == FI_MODEL_FARMER_LSTM;
    const size_t rows = farmer ? p->last_rows / l->cfg.entry_size : p->last_rows;
    const size_t per_layer = rows * fi::kHid;
    if (rows == 0 || n != 5 * per_layer)
        return set_error(FI_ERR_ARG, "fi_learner_debug_relu_masks: need n = 5 * %zu (rows of the last step x 512)", per_layer);
    FI_CUDA_OK(cudaSetDevice(l->cfg.device));
    std::lock_guard<std::mutex> step_lock(p->step_mu);
    unsigned char* dev = nullptr;
    FI_CUDA_OK(cudaMalloc((void**)&dev, n));
    int rc = FI_OK;
    for (int layer = 0; layer < 5 && rc == FI_OK; layer++) {
        if (const uint32_t* bits = fi::dense_relu_bits(p->dense, layer)) {
            // the split-operand path keeps the decisions its backward pass used as bit masks
            fi::LaunchScope ls("relu_bits_expand_kernel", p->stream, 1.125 * per_layer, fi::kWorkBytes);
            relu_bits_expand_kernel<<<fi::kNumSMs * 4, 256, 0, p->stream>>>(bits, per_layer, dev + layer * per_layer);
            rc = ls.done();
            continue;
        }
        const float* a = fi::dense_activation(p->dense, layer);
        if (!a) {
            rc = set_error(FI_ERR_STATE, "fi_learner_debug_relu_masks: no activations of the last step to read back");
            break;
        }
        fi::LaunchScope ls("relu_mask_kernel", p->stream, 5.0 * per_layer, fi::kWorkBytes);
        relu_mask_kernel<<<fi::kNumSMs * 4, 256, 0, p->stream>>>(a, nullptr, per_layer, dev + layer * per_layer);
        rc = ls.done();
    }
    if (rc == FI_OK && cudaMemcpyAsync(host, dev, n, cudaMemcpyDeviceToHost, p->stream) != cudaSuccess) rc = FI_ERR_CUDA;
    if (cudaStreamSynchronize(p->stream) != cudaSuccess && rc == FI_OK) rc = set_error(FI_ERR_CUDA, "stream sync failed");
    cudaFree(dev);
    return rc;
}

// ---- instrumentation ------------------------------------------------------------------------
void fi_prof_enable(int on) {
    fi::ProfState& p = fi::prof();
    std::lock_guard<std::mutex> g(p.mu);
    if (!on) p.close_locked();
    p.on.store(on != 0);
}

int fi_prof_collect(fi_prof_entry* out, int max_entries) {
    fi::ProfState& p = fi::prof();
    std::vector<fi::ProfRec> recs;
    {
        std::lock_guard<std::mutex> g(p.mu);
        p.close_locked();
        recs.swap(p.recs);
    }
    std::vector<fi_prof_entry> agg;
    for (const fi::ProfRec& r : recs) {
        if (cudaEventSynchronize(r.b) != cudaSuccess) continue;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.a, r.b) != cudaSuccess) continue;
        fi_prof_entry* e = nullptr;
        for (fi_prof_entry& a : agg)
            if (strncmp(a.name, r.name, sizeof(a.name)) == 0) e = &a;
        if (!e) {
            fi_prof_entry n;
            memset(&n, 0, sizeof(n));
            strncpy(n.name, r.name, sizeof(n.name) - 1);
            n.unit = r.unit;
            agg.push_back(n);
            e = &agg.back();
        }
        e->launches += (uint64_t)r.launches;
        e->total_ms += ms;
        e->work += r.work;
    }
    cudaGetLastError();
    {
        std::lock_guard<std::mutex> g(p.mu);
        if (p.recs.empty()) p.used = 0;  // the event pool is reused by the next window
    }
    int n = 0;
    for (const fi_prof_entry& a : agg)
        if (out && n < max_entries) out[n++] = a;
    return (int)agg.size();
}

// ---- pinned host memory for callers that stage their own batches ------------------------------
void* fi_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) {
        set_error(FI_ERR_CUDA, "fi_host_alloc(%zu) failed: %s", bytes, cudaGetErrorString(cudaGetLastError()));
        return nullptr;
    }
    return p;
}
void fi_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

}  // extern "C"
