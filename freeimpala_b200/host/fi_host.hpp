// C++ host side above the C ABI (include/fi_learner.h): the reference's own interfaces for this path --
// SharedBuffer (include/freeimpala/data_structures.h:191-307), Model / ModelManager (:43-157, :310-481) and
// Learner (include/freeimpala/learner.h:100-207) -- with the same method names, argument meaning, return
// values and blocking behaviour, so that agent.h and the cmd/* mains compile against it unchanged
// (INTEGRATION.md shows the two-line switch). Header-only, like the reference; no CUDA or torch types.
#pragma once
#include <atomic>
#include <chrono>
#include <cstdint>
#include <cstdio>
#include <memory>
#include <mutex>
#include <optional>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "../../include/fi_learner.h"

namespace fi_host {

constexpr size_t ELEMENT_SIZE = FI_ELEMENT_SIZE;  // data_structures.h:35

// A gathered batch. The reference returns vector<vector<char>> (M heap copies under the ring mutex,
// data_structures.h:286-293); here the batch stays in HBM and empty() keeps its meaning (learner.h:79).
struct DeviceBatch {
    fi_batch raw{};
    bool failed = false;   // readBatch hit a CUDA / argument error (logged by the library): not a drain, not a spurious wake-up
    bool empty() const { return raw.num_slots == 0; }
    size_t size() const { return raw.num_slots; }
    std::vector<std::vector<char>> to_host() const {  // the reference's representation, for callers that need bytes
        std::vector<char> flat(raw.num_slots * raw.slot_bytes);
        if (!flat.empty()) fi_batch_to_host(&raw, flat.data(), flat.size());
        std::vector<std::vector<char>> out(raw.num_slots);
        for (size_t i = 0; i < raw.num_slots; i++)
            out[i].assign(flat.begin() + i * raw.slot_bytes, flat.begin() + (i + 1) * raw.slot_bytes);
        return out;
    }
};

class SharedBuffer {
public:
    explicit SharedBuffer(fi_ring* ring) : ring_(ring) {}                       // owned by the Learner
    bool write(const std::vector<char>& data) { return fi_ring_write(ring_, data.data(), data.size()) == 1; }       // :219-241
    bool write(const void* data, size_t n) { return fi_ring_write(ring_, data, n) == 1; }
    bool try_write(const std::vector<char>& data) { return fi_ring_try_write(ring_, data.data(), data.size()) == 1; } // :244-264
    DeviceBatch readBatch(size_t batch_size, void* stream = nullptr) {                                               // :267-300
        DeviceBatch b;
        if (fi_ring_read_batch(ring_, batch_size, stream, &b.raw) < 0) {   // logged by the library
            b.raw.num_slots = 0;
            b.failed = true;
        }
        return b;
    }
    void setDraining() { fi_ring_set_draining(ring_); }                                                              // :212-216
    size_t getFilledCount() { return fi_ring_filled_count(ring_); }                                                  // :303-306
    fi_ring* handle() const { return ring_; }

private:
    fi_ring* ring_;
};

// A (version, bytes) snapshot of one player's published weights (Model, :43-157).
class Model {
public:
    Model(std::vector<char> data, uint64_t version) : data_(std::move(data)), version_(version) {}
    uint64_t getVersion() const { return version_; }                         // :130-132
    std::vector<char> getData() const { return data_; }                      // :135-138
    std::shared_ptr<Model> createCopy() const { return std::make_shared<Model>(data_, version_); }  // :149-156
    // :140-147: replace the blob and the version (the MPI actor's TAG_WEIGHTS_RES handler, agent.h:139-142); like the
    // reference, a blob of another size is ignored
    void update(const std::vector<char>& new_data, uint64_t new_version) {
        if (new_data.size() != data_.size()) return;
        data_ = new_data;
        version_ = new_version;
    }
    const float* params() const { return reinterpret_cast<const float*>(data_.data()); }

private:
    std::vector<char> data_;
    uint64_t version_;
};

class ModelManager {
public:
    ModelManager(fi_learner* l, size_t players) : l_(l), players_(players) {}
    std::shared_ptr<Model> getModel(size_t p) {                               // :433-438
        if (p >= players_) return nullptr;
        std::vector<char> blob(fi_model_bytes(l_));
        uint64_t v = 0;
        if (fi_model_get(l_, (int)p, blob.data(), blob.size(), &v) != FI_OK) return nullptr;
        return std::make_shared<Model>(std::move(blob), v);
    }
    uint64_t getLatestVersion(size_t p) { return p < players_ ? fi_model_version(l_, (int)p) : 0; }                  // :475-480
    bool waitForModelUpdate(size_t p, uint64_t current_version, int timeout_ms) {                                    // :454-472
        return p < players_ && fi_model_wait_update(l_, (int)p, current_version, timeout_ms) == 1;
    }
    // File = u64 version + raw parameter bytes, exactly the reference's size and layout (:105-110). setSaveOptimizerState(true)
    // appends the Adam moments + step in a trailing section old readers ignore (exact resume; 3x the file size): opt-in.
    // Returns false (and the library has logged why) when the file could not be written; the reference's saveModel is
    // void and logs, so existing callers keep compiling.
    bool saveModel(size_t p, uint64_t current_iteration = 0) {                                                       // :388-423
        if (p >= players_) return false;
        const bool ok = fi_model_save(l_, (int)p, current_iteration, save_optimizer_state_ ? 1 : 0) == FI_OK;
        if (!ok) std::fprintf(stderr, "[fi_host][error] saveModel(player %zu, iteration %llu) failed: %s\n", p,
                              (unsigned long long)current_iteration, fi_last_error());
        return ok;
    }
    bool saveAllModels(uint64_t current_iteration = 0) {
        bool ok = true;
        for (size_t p = 0; p < players_; p++) ok = saveModel(p, current_iteration) && ok;
        return ok;
    }
    void setSaveOptimizerState(bool on) { save_optimizer_state_ = on; }
    void loadModels(const std::string& path) { if (!path.empty()) fi_model_load(l_, path.c_str()); }                 // :337-385

private:
    fi_learner* l_;
    size_t players_;
    bool save_optimizer_state_ = false;
};

// The two MetricsTracker calls the reference's trainModel makes (learner.h:34 createTrainingTimer, :48
// recordLearnerModelUpdate) are kept at the same two points of the step. In the integrated build FI_HOST_METRICS_TRACKER is
// defined before this header is included (INTEGRATION.md) and they go to the reference's own singleton
// (include/freeimpala/metrics_tracker.h:147-177, 213-217); stand-alone (tests, the harness) they feed the counters below.
struct StepMetrics {
    std::atomic<uint64_t> model_updates{0}, training_ns{0};
};
#ifdef FI_HOST_METRICS_TRACKER
#define FI_HOST_TRAINING_TIMER() auto fi_host_training_timer = MetricsTracker::getInstance()->createTrainingTimer()
#define FI_HOST_RECORD_MODEL_UPDATE() MetricsTracker::getInstance()->recordLearnerModelUpdate()
#else
#define FI_HOST_TRAINING_TIMER() (void)0
#define FI_HOST_RECORD_MODEL_UPDATE() (void)0
#endif

class Learner {
public:
    // Same order as learner.h:100-110. `r` (simulated training time) is ignored: the step is real work.
    // legal_action_mask: fi_learner_config.legal_action_mask (actor-critic only; records carry the legal word, fi_learner.h).
    Learner(size_t p, size_t B, size_t S, size_t M, size_t /*r*/, size_t c, const std::string& l, const std::string& m,
            size_t T, int device = 0, int model = FI_MODEL_MLP_ACTOR_CRITIC, bool legal_action_mask = false)
        : num_players_(p), batch_size_(M), checkpoint_frequency_(c), checkpoint_location_(l), total_iterations_(T) {
        fi_learner_config cfg;
        fi_learner_config_default(&cfg);
        cfg.device = device;
        cfg.num_players = (int)p;
        cfg.buffer_capacity = B;
        cfg.entry_size = S;
        cfg.batch_size = M;
        cfg.model = model;
        cfg.loss = model == FI_MODEL_FARMER_LSTM ? FI_LOSS_MSE : FI_LOSS_VTRACE;
        cfg.checkpoint_location = l.empty() ? nullptr : l.c_str();
        cfg.legal_action_mask = legal_action_mask ? 1 : 0;
        h_ = fi_learner_create(&cfg);
        if (!h_) throw std::runtime_error(std::string("fi_learner_create: ") + fi_last_error());
        model_manager_ = std::make_shared<ModelManager>(h_, p);
        if (!m.empty()) model_manager_->loadModels(m);                         // learner.h:129-132
        for (size_t i = 0; i < p; i++) shared_buffers_.push_back(std::make_shared<SharedBuffer>(fi_learner_ring(h_, (int)i)));
        iterations_ = std::make_unique<std::atomic<size_t>[]>(p);
        for (size_t i = 0; i < p; i++) iterations_[i].store(0);
    }
    ~Learner() {
        stop();
        if (h_) fi_learner_destroy(h_);
    }
    void start() {                                                            // learner.h:158-163
        for (size_t p = 0; p < num_players_; p++) worker_threads_.emplace_back([this, p] { workerThread(p); });
    }
    void stop() {                                                             // learner.h:166-197
        if (stopped_.exchange(true)) return;
        should_stop_.store(true);
        for (auto& b : shared_buffers_) b->setDraining();
        for (auto& t : worker_threads_) if (t.joinable()) t.join();
        worker_threads_.clear();
        for (size_t p = 0; p < num_players_; p++) fi_learner_sync(h_, (int)p);
        {
            // in-progress checkpoint threads finish BEFORE the final save (the reference saves first and joins after,
            // learner.h:184-196; with real files two writers of model_p_latest.bin must not overlap -- the library also
            // serialises saves per player and renames complete files into place)
            std::lock_guard<std::mutex> lock(checkpoint_mutex_);
            for (auto& t : checkpoint_threads_) if (t.joinable()) t.join();
            checkpoint_threads_.clear();
        }
        if (!checkpoint_location_.empty()) model_manager_->saveAllModels(total_iterations_);
    }
    std::vector<std::shared_ptr<SharedBuffer>> getSharedBuffers() { return shared_buffers_; }   // learner.h:200-202
    std::shared_ptr<ModelManager> getModelManager() { return model_manager_; }                   // learner.h:205-207
    fi_learner* handle() const { return h_; }
    size_t iterationsDone(size_t p) const { return p < num_players_ ? iterations_[p].load(std::memory_order_acquire) : 0; }
    bool failed() const { return failed_.load(); }   // a worker stopped on a failed readBatch / step (fi_last_error was logged)
    const StepMetrics& stepMetrics() const { return metrics_; }   // model updates / host time inside trainModel (stand-alone counters)
    // Losses of player p's optimiser step `step` (1-based, one of the last 8): {total, pg, baseline, entropy} for V-trace,
    // {loss,0,0,0} for the regression step. Waits only for that step's read-back (no counterpart in the reference, whose
    // trainModel computes nothing to log).
    bool lossesAt(size_t p, uint64_t step, float out[4]) const { return fi_learner_losses_at(h_, (int)p, step, out) == FI_OK; }

private:
    bool trainModel(size_t p, const DeviceBatch& batch) {                      // learner.h:32-49 (void there: no error path)
        FI_HOST_TRAINING_TIMER();                                              // learner.h:33-34
        const auto t0 = std::chrono::steady_clock::now();
        // forward, loss, backward, (all-reduce), Adam and the publication of version + 1, all enqueued on the player's stream
        if (fi_learner_step(h_, (int)p, &batch.raw) != FI_OK) {                // logged by the library; reference style: no throw
            failed_.store(true);
            should_stop_.store(true);
            return false;
        }
        metrics_.training_ns.fetch_add((uint64_t)std::chrono::duration_cast<std::chrono::nanoseconds>(
                                           std::chrono::steady_clock::now() - t0).count());
        metrics_.model_updates.fetch_add(1);
        FI_HOST_RECORD_MODEL_UPDATE();                                         // learner.h:47-48
        return true;
    }
    void checkpointModel(size_t p, uint64_t it) {                              // learner.h:52-69
        std::lock_guard<std::mutex> lock(checkpoint_mutex_);
        for (auto& t : checkpoint_threads_) if (t.joinable()) t.join();       // reap finished checkpoint threads (:56-63)
        checkpoint_threads_.clear();
        checkpoint_threads_.emplace_back([this, p, it] { model_manager_->saveModel(p, it); });
    }
    void workerThread(size_t p) {                                              // learner.h:72-97
        size_t it = 0;
        void* stream = fi_learner_stream(h_, (int)p);
        while (!should_stop_.load() && it < total_iterations_) {
            DeviceBatch batch = shared_buffers_[p]->readBatch(batch_size_, stream);
            if (batch.empty()) {
                // a failed read (sticky H2D failure, bad batch size) would fail again at once: stop instead of spinning;
                // a drained or spurious empty batch loops as in the reference (learner.h:79-84)
                if (batch.failed) { failed_.store(true); should_stop_.store(true); }
                if (should_stop_.load()) break;
                continue;
            }
            if (!trainModel(p, batch)) break;   // a failed step is not counted as an iteration
            iterations_[p].store(++it, std::memory_order_release);
            if (checkpoint_frequency_ > 0 && it % checkpoint_frequency_ == 0 && !checkpoint_location_.empty()) checkpointModel(p, it);
        }
    }

    size_t num_players_, batch_size_, checkpoint_frequency_;
    std::string checkpoint_location_;
    size_t total_iterations_;
    fi_learner* h_ = nullptr;
    std::shared_ptr<ModelManager> model_manager_;
    std::vector<std::shared_ptr<SharedBuffer>> shared_buffers_;
    std::vector<std::thread> worker_threads_, checkpoint_threads_;
    std::unique_ptr<std::atomic<size_t>[]> iterations_;   // per player; read by other threads (iterationsDone)
    std::atomic<bool> should_stop_{false}, stopped_{false}, failed_{false};
    std::mutex checkpoint_mutex_;
    StepMetrics metrics_;
};

}  // namespace fi_host
