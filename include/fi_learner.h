/* freeimpala-b200: C ABI of the B200-native learner hot path.
 *
 * This header is the drop-in boundary (SURVEY.md section 8b). The reference has no plugin /
 * FFI interface for this path: the boundary is the set of C++ call sites on
 * SharedBuffer, ModelManager and Learner::trainModel. Each export below names the
 * reference interface it replaces (file:line under the reference tree). Signatures use
 * plain pointers and sizes only: no C++ types, no torch types, no libtorch in the step.
 *
 * Conventions (the reference's: bool returns + log, no exceptions on the hot path):
 *   - functions that mirror a `bool` in the reference return 1 (true) / 0 (false);
 *   - every other function returns FI_OK (0) or a negative fi_status; fi_last_error() gives
 *     the message of the calling thread's last failure;
 *   - there is NO CPU fallback: without a CUDA device every create call fails with
 *     FI_ERR_CUDA (loudly), it never computes on the host.
 *
 * Threading (matches the reference): fi_ring_write/try_write may be called concurrently by
 * any number of actor / MPI receiver threads (agent.h:96; freeimpala_mpi_async_pool
 * main.cpp:288); fi_ring_read_batch and fi_learner_step are called by exactly one learner
 * worker thread per player (learner.h:72-97), p of them concurrently on distinct players.
 */
#ifndef FI_LEARNER_H
#define FI_LEARNER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FI_API __attribute__((visibility("default")))

typedef enum {
    FI_OK = 0,
    FI_ERR_CUDA = -1,     /* CUDA runtime / driver error, or no device */
    FI_ERR_ARG = -2,      /* invalid argument */
    FI_ERR_STATE = -3,    /* call not valid in this state */
    FI_ERR_IO = -4,       /* checkpoint file error */
    FI_ERR_NCCL = -5      /* NCCL unavailable or failed */
} fi_status;

FI_API const char* fi_last_error(void);
FI_API const char* fi_version(void);
/* Number of CUDA kernels this library has launched in this process (all streams). */
FI_API uint64_t fi_kernel_launch_count(void);

/* Per-kernel device timing. While enabled, every kernel launch of the library is bracketed by
 * CUDA events on its launching stream and tagged with its algorithmic work. fi_prof_collect
 * waits for the recorded launches, aggregates them by kernel name into out[0..max) and returns
 * the number of distinct kernels; the window is then reset. */
typedef struct fi_prof_entry {
    char name[48];
    uint64_t launches;
    double total_ms;   /* sum of device durations */
    double work;       /* sum of algorithmic bytes (unit 0) or flops (unit 1) */
    int unit;
} fi_prof_entry;
FI_API void fi_prof_enable(int on);
FI_API int fi_prof_collect(fi_prof_entry* out, int max_entries);
/* Diagnostics (tools/gemm_trace.py): with FI_TC_TRACE="<trans>,<min n>,<min k>" in the environment, matching tcgen05 GEMM
 * launches log the pipeline events of their first 4 CTAs; this copies the last log out. Layout [cta 0..3][role 0..2][4096]
 * of (clock64 << 8 | tag), 0 = unused. Returns the number of 8-byte entries or a negative fi_status. No reference counterpart. */
FI_API int fi_debug_tc_trace(void* host, size_t bytes);
/* Diagnostics / tests: selects the implementation of the FarmerLstm recurrence (reference cmd/libtorch_bench/main.cpp:25-27):
 * 1 = tcgen05 kernels over clusters of 8 CTAs (csrc/lstm_tc.cu; needs the 3xFP16 path), 0 = fp32 FFMA kernels
 * (csrc/model_farmer.cu), -1 = as FI_LSTM_TC in the environment says (default 0). No reference counterpart. */
FI_API void fi_debug_set_lstm_tc(int on);

/* ============================ trajectory ring ============================================
 * Replaces SharedBuffer (include/freeimpala/data_structures.h:191-307). One ring per
 * player. Host side: a bounded MPMC FIFO of `capacity` pinned-host slots of slot_bytes =
 * entry_size * FI_ELEMENT_SIZE bytes, mirrored by `capacity` slots in HBM. A write copies
 * the caller's bytes into the pinned slot and enqueues cudaMemcpyAsync(pinned -> HBM slot)
 * on the ring's side stream; read_batch gathers M consecutive HBM slots (FIFO, wraparound)
 * into a contiguous [M, slot_bytes] device batch with one sm_100a kernel. */
#define FI_ELEMENT_SIZE 1024 /* data_structures.h:35 */

typedef struct fi_ring fi_ring;

typedef struct fi_batch {
    void* dev_ptr;      /* device pointer, [num_slots, slot_bytes] contiguous; valid until the
                           next fi_ring_read_batch on the same ring */
    size_t num_slots;   /* M, or 0 for the "empty batch" (data_structures.h:278-280) */
    size_t slot_bytes;
    void* stream;       /* cudaStream_t on which the gather was enqueued (the learner stream) */
    uint64_t seq;       /* index of the first consumed slot since ring creation */
} fi_batch;

/* SharedBuffer ctor (data_structures.h:205-210; created per player at learner.h:135-139).
 * Slots are zero-initialised (BufferEntry ctor, :164). Returns NULL on failure. */
FI_API fi_ring* fi_ring_create(int device, size_t entry_size, size_t capacity);
FI_API void fi_ring_destroy(fi_ring* ring);

/* SharedBuffer::write (data_structures.h:219-241). Blocks while the ring is full (no
 * draining check, as in the reference). Returns 1 after the bytes are copied (the caller may
 * reuse src immediately); returns 0 if n > slot_bytes (nothing is written). Bytes
 * [n, slot_bytes) of the slot keep their previous content (:226-227). */
FI_API int fi_ring_write(fi_ring* ring, const void* src, size_t n);
/* SharedBuffer::try_write (data_structures.h:244-264): 0 if the lock is contended, the ring
 * is full, or n > slot_bytes; never blocks on ring state. */
FI_API int fi_ring_try_write(fi_ring* ring, const void* src, size_t n);

/* `count` consecutive fi_ring_write calls in one crossing of the boundary (an MPI receiver or a foreign-
 * language actor handing over a burst of trajectories): entry i is the n bytes at src + i * stride. Returns
 * the number of entries written (stops at the first one that fi_ring_write would reject). */
FI_API size_t fi_ring_write_many(fi_ring* ring, const void* src, size_t count, size_t stride, size_t n);

/* Zero-copy producer (SURVEY.md section 8f rank 1): reserve the next pinned slot (blocks
 * while full), let the caller fill it in place (e.g. MPI_Irecv straight into it), then
 * commit n bytes. Slots commit in reservation order. */
FI_API void* fi_ring_reserve(fi_ring* ring, uint64_t* ticket);
FI_API int fi_ring_commit(fi_ring* ring, uint64_t ticket, size_t n);

/* Burst form of the zero-copy producer: reserve `count` consecutive slots at once (blocks until that many are
 * free; count <= capacity), e.g. to post `count` MPI_Irecv's straight into pinned memory (slots[i] receives the
 * address of the i-th slot; may be NULL when the caller tracks addresses itself), then commit them together.
 * Returns count / 1 on success, 0 on a bad argument. */
FI_API size_t fi_ring_reserve_many(fi_ring* ring, size_t count, void** slots, uint64_t* first_ticket);
FI_API int fi_ring_commit_many(fi_ring* ring, uint64_t first_ticket, size_t count, size_t n);

/* SharedBuffer::readBatch (data_structures.h:267-300). Blocks until count >= M or draining.
 * Draining with count < M: out->num_slots = 0 and returns 0 (the caller breaks/continues,
 * learner.h:79-84). Otherwise consumes exactly M slots FIFO with wraparound, wakes all
 * writers, fills *out and returns 1. The gather runs on `stream` (cudaStream_t; NULL = the
 * ring's own learner stream). Returns a negative fi_status on CUDA errors / M > capacity. */
FI_API int fi_ring_read_batch(fi_ring* ring, size_t batch_size, void* stream, fi_batch* out);

FI_API void fi_ring_set_draining(fi_ring* ring);      /* data_structures.h:212-216 */
FI_API size_t fi_ring_filled_count(fi_ring* ring);    /* data_structures.h:303-306 */
FI_API size_t fi_ring_slot_bytes(const fi_ring* ring);
FI_API size_t fi_ring_capacity(const fi_ring* ring);
/* Test/inspection helper: synchronise the batch's stream and copy it to host memory. */
FI_API int fi_batch_to_host(const fi_batch* batch, void* dst, size_t n);

/* ============================ learner ====================================================
 * Replaces the body of Learner::trainModel (include/freeimpala/learner.h:32-49), whose
 * reference implementation is a stub (sleep + rand()), with the step whose numerics the
 * reference defines in cmd/libtorch_bench/main.cpp:117-135 (train_step), plus the V-trace
 * actor-critic step BASELINE.json's north_star adds. */
typedef enum {
    FI_MODEL_FARMER_LSTM = 0, /* FarmerLstmModel, libtorch_bench main.cpp:14-42 */
    FI_MODEL_MLP_ACTOR_CRITIC = 1 /* trunk shapes of main.cpp:17-21 per transition + policy/value head */
} fi_model_kind;
typedef enum {
    FI_LOSS_MSE = 0, FI_LOSS_MAE = 1, FI_LOSS_HUBER = 2, /* criterion, main.cpp:105-114 */
    FI_LOSS_VTRACE = 3
} fi_loss_kind;
typedef enum {
    FI_OPT_ADAM = 0, FI_OPT_SGD = 1, FI_OPT_ADAMW = 2, /* main.cpp:94-103 */
    FI_OPT_RMSPROP = 3  /* torch.optim.RMSprop, centered=False, weight_decay=0 (the IMPALA paper's optimiser) */
} fi_opt_kind;
typedef enum {
    FI_GEMM_AUTO = 0,   /* the fastest fp32-accurate tcgen05 path the shape allows, else SIMT fp32 */
    FI_GEMM_SIMT = 1,   /* fp32 FFMA kernels only */
    FI_GEMM_TCGEN05 = 2, /* require the tcgen05 3xTF32 path (error if a shape cannot use it) */
    FI_GEMM_TCGEN05_F16 = 3 /* require the tcgen05 3xFP16 path: fp16 hi/lo pairs with per-tensor power-of-two scales */
} fi_gemm_mode;

typedef struct fi_learner_config {
    int device;               /* CUDA ordinal */
    int num_players;          /* p  (learner.h ctor) */
    size_t buffer_capacity;   /* B */
    size_t entry_size;        /* S: records (FI_ELEMENT_SIZE bytes each) per trajectory = T; FarmerLstm needs S >= 8
                                 (x[484] spans records 0..7) */
    size_t batch_size;        /* M: trajectories per step on THIS rank */
    int model;                /* fi_model_kind */
    int loss;                 /* fi_loss_kind */
    int optimizer;            /* fi_opt_kind */
    double lr;                /* --learning-rate (main.cpp:157-159); README shape uses 5e-4 */
    uint64_t seed;            /* weight init seed (U(+-1/sqrt(fan_in)) like torch::nn defaults) */
    /* V-trace constants (Espeholt et al. 2018); ignored unless loss == FI_LOSS_VTRACE. Accepted ranges (checked by
       fi_learner_create for the actor-critic model): rho_bar, c_bar, pg_rho_bar > 0, +inf meaning no clipping;
       0 <= lambda_ <= 1; baseline_cost, entropy_cost finite and >= 0. */
    float rho_bar, c_bar, pg_rho_bar, lambda_, baseline_cost, entropy_cost;
    int gemm_mode;            /* fi_gemm_mode */
    int publish_every;        /* D2H the weights into the model store every k steps (>=1) */
    const char* checkpoint_location; /* -l; may be NULL */
    /* Appended after checkpoint_location; fi_learner_config_default sets 0, 0.99, 1e-8, 0 (torch's defaults). */
    double max_grad_norm;     /* clip the gradient to this global L2 norm before every update; 0 = no clipping. Applied to
                                 the all-reduced gradient, so every data-parallel rank uses the same coefficient */
    double rmsprop_alpha;     /* FI_OPT_RMSPROP: square-average decay, 0 < alpha < 1 */
    double rmsprop_eps;       /* FI_OPT_RMSPROP: added to sqrt(square average), > 0 */
    double rmsprop_momentum;  /* FI_OPT_RMSPROP: 0 <= momentum < 1 (0 = no momentum buffer) */
    /* Appended after rmsprop_momentum; fi_learner_config_default sets 0. Actor-critic model only: 1 = the V-trace loss
       head reads each record's legal-action word (FI_REC_WORD_LEGAL) and computes log pi, log mu, the entropy and the
       policy gradient over the legal set; 0 = all 16 actions, word 182 is not read. */
    int legal_action_mask;
} fi_learner_config;

/* Trajectory record (FI_ELEMENT_SIZE bytes = 256 32-bit words) of the actor-critic model, the words the loss head reads
 * (DESIGN.md section 1 has the whole layout): 0..161 observation, 162..177 behaviour logits mu (fp32), 178 action (int32,
 * clamped to [0, 15]), 179 reward, 180 discount, 181 bootstrap value (last record of a trajectory), 182 legal-action word.
 *
 * Legal-action masking (legal_action_mask = 1). Word 182 is a uint32 in which bit j set means action j was legal at this
 * step; bits 16..31 are ignored. The support is word | (1 << action): the action taken was legal by definition, so a word
 * of 0 describes a forced move (pi(a) = 1, log pi(a) = 0, no entropy and no policy gradient for that transition). Then
 *   log pi(a) = z_a - logsumexp of the learner's logits over the support
 *   log mu(a) = mu_a - logsumexp of words 162..177 over the support
 *   entropy term = sum over the support of pi log pi
 * and d(loss)/d(logit j) is exactly 0 for every j outside it. The value path, the V-trace recurrence and the clipping
 * constants are unchanged. Logits outside the support (learner or behaviour) never enter the arithmetic: -inf or NaN
 * there changes nothing.
 *
 * What the actor does: fi_learner_infer returns the raw logits of all 16 actions. The actor samples from the
 * softmax of those logits over its legal set, stores the logits it got (raw or already set to -inf outside the legal set)
 * in words 162..177, the action in 178 and the legal word in 182. */
#define FI_REC_WORD_LEGAL 182

typedef struct fi_learner fi_learner;

FI_API void fi_learner_config_default(fi_learner_config* cfg);
/* Learner ctor (learner.h:100-140): creates p rings, p models (random init), optimiser
 * state and all step workspaces in HBM. Returns NULL on failure (see fi_last_error). An unknown
 * optimiser, max_grad_norm < 0 or not finite, rmsprop_alpha outside (0, 1), rmsprop_eps <= 0 or
 * rmsprop_momentum outside [0, 1), legal_action_mask other than 0 or 1 or set to 1 for the FarmerLstm model (which has
 * no policy), and, for the actor-critic model, a V-trace constant outside the range
 * fi_learner_config states, is rejected (FI_ERR_ARG) before any device is looked for. */
FI_API fi_learner* fi_learner_create(const fi_learner_config* cfg);
FI_API void fi_learner_destroy(fi_learner* l);
/* getSharedBuffers (learner.h:200-202): ring of one player, owned by the learner. */
FI_API fi_ring* fi_learner_ring(fi_learner* l, int player);
FI_API void* fi_learner_stream(fi_learner* l, int player); /* cudaStream_t of that player */

/* The learner step: forward, loss, backward, (gradient allreduce), optimiser update, and
 * publication of the new weights as version+1 (learner.h:40-45). `batch` must come from
 * fi_ring_read_batch on that player's ring (or fi_learner_stage_batch). Asynchronous on
 * the player's stream except for the publish D2H bookkeeping. Returns FI_OK or an error. */
FI_API int fi_learner_step(fi_learner* l, int player, const fi_batch* batch);
/* Split form used by tests and by data-parallel hosts that own their own collective:
 * forward+loss+backward into the flat gradient arena, then the optimiser update. */
FI_API int fi_learner_forward_backward(fi_learner* l, int player, const fi_batch* batch);
FI_API int fi_learner_apply_update(fi_learner* l, int player);
/* Copy host bytes [num_slots, slot_bytes] into the learner's device batch buffer on the
 * player's stream (pinned staging inside) and describe it in *out. For tests/benchmarks that
 * bypass the ring. */
FI_API int fi_learner_stage_batch(fi_learner* l, int player, const void* host, size_t num_slots, fi_batch* out);

/* Results of the last step (synchronises the player's stream). losses[4]:
 * MSE-family: {loss,0,0,0}; V-trace: {total, pg, baseline, entropy}. */
FI_API int fi_learner_last_losses(fi_learner* l, int player, float losses[4]);
/* Same numbers in the double precision they are accumulated in (synchronises the stream). */
FI_API int fi_learner_last_losses_f64(fi_learner* l, int player, double losses[4]);
/* Losses of optimiser step `step` (1-based count of fi_learner_step calls on this player); valid for the last 8 steps.
 * Waits only for that step's read-back, so a host loop can log step s-1 while step s runs. */
FI_API int fi_learner_losses_at(fi_learner* l, int player, uint64_t step, float losses[4]);
/* Gradient L2 norm (before clipping, after the data-parallel all-reduce) of optimiser step `step`: same window and waiting
 * as fi_learner_losses_at. FI_ERR_STATE when the learner does not clip (max_grad_norm == 0). */
FI_API int fi_learner_grad_norm_at(fi_learner* l, int player, uint64_t step, double* norm);
/* Learning rate of this player's optimiser from its next update on (a schedule is one call per step; the step's CUDA graph
 * picks it up with the other per-step scalars). lr must be finite and >= 0; the initial value is fi_learner_config.lr. */
FI_API int fi_learner_set_lr(fi_learner* l, int player, double lr);
/* Wait until everything enqueued for this player (step and weight publication) has finished. */
FI_API int fi_learner_sync(fi_learner* l, int player);
FI_API uint64_t fi_learner_steps_done(fi_learner* l, int player);

/* Inspection for parity tests: the ReLU decisions (1 = active) of the 5 hidden layers in the last
 * forward pass of this player, [5][rows * 512] bytes (rows = M*T for the actor-critic model, M for
 * the farmer model's dense stack). */
FI_API int fi_learner_debug_relu_masks(fi_learner* l, int player, unsigned char* host, size_t n);

/* Flat fp32 parameter arena, in the reference's model.parameters() order (farmer: 16
 * tensors, 1,514,497 values = 6,057,988 bytes). */
FI_API size_t fi_learner_param_count(const fi_learner* l);
FI_API int fi_learner_num_tensors(const fi_learner* l);
FI_API int fi_learner_tensor_info(const fi_learner* l, int i, size_t* offset, size_t* numel, size_t* rows, size_t* cols);
FI_API int fi_learner_set_params(fi_learner* l, int player, const float* host, size_t n);
FI_API int fi_learner_get_params(fi_learner* l, int player, float* host, size_t n);
FI_API int fi_learner_get_grads(fi_learner* l, int player, float* host, size_t n);
FI_API int fi_learner_set_grads(fi_learner* l, int player, const float* host, size_t n);
/* Optimiser state and step count (checkpoint-with-optimiser-state tests); m / v may be NULL. Adam / AdamW: (first moment,
 * second moment, step); RMSProp: (momentum buffer, square average, step); SGD: zeros. */
FI_API int fi_learner_get_opt_state(fi_learner* l, int player, float* m, float* v, size_t n, int64_t* step);
/* Device pointers into the arenas (for hosts that run their own collective on them). */
FI_API void* fi_learner_grad_ptr(fi_learner* l, int player);
FI_API void* fi_learner_param_ptr(fi_learner* l, int player);
/* Batched actor policy inference reusing the step's forward kernels (SURVEY.md 8f rank 2):
 * host observations [rows,162] -> logits [rows,16], values [rows] (actor-critic model), or
 * z [rows,T,162], x [rows,484] -> values [rows] (farmer model; logits may be NULL). */
FI_API int fi_learner_infer(fi_learner* l, int player, const float* obs_or_z, const float* x, size_t rows, size_t t, float* logits, float* values);
/* fi_learner_infer is thread-safe and COMBINING: requests of concurrent callers (the actors of one player) are packed into one
 * host->device copy, one forward on the newest published weights and one device->host copy per batch. Counters since creation:
 * calls made, forwards run, rows served (any may be NULL). No counterpart in the reference (the hook is a comment, agent.h:52-56). */
FI_API int fi_learner_infer_stats(fi_learner* l, int player, uint64_t* calls, uint64_t* batches, uint64_t* rows);
/* FarmerLstm model only. States s = 0..states-1 with history z[s] ([t,162], row-major [states,t,162]); candidate rows
 * offsets[s] .. offsets[s+1]-1 of x ([rows,484], rows = offsets[states]) belong to state s. Runs the recurrence once per
 * state and the dense stack once per candidate, on the newest published weights, combined with concurrent callers like
 * fi_learner_infer. values[r] (may be NULL) = the value of candidate r, bit-identical to fi_learner_infer on a z repeated per
 * candidate; best[s] (may be NULL, not both) = index WITHIN state s's group of its largest value, the lowest index on ties
 * (NaN counts as largest, as in numpy's argmax).
 * FI_ERR_ARG, with the learner still usable, for an actor-critic learner, a NULL z / x / offsets, values and best both NULL,
 * states or t of 0, offsets[0] != 0, offsets not strictly increasing (every state needs a candidate), or more than 16384
 * candidate rows. fi_learner_infer_stats counts the candidate rows.
 *
 * What a DouZero-style actor does with it: for each decision it sends the state's move history once as z and one x row per
 * legal action (state and action features), and plays legal action best[s]; with many environments per actor thread it sends
 * one state per environment in one call. This replaces repeating z once per legal action for fi_learner_infer and taking the
 * argmax of the returned values on the host. Exploration (epsilon-greedy) stays with the actor: it needs no value. */
FI_API int fi_learner_infer_grouped(fi_learner* l, int player, const float* z, size_t states, size_t t, const float* x,
                                    const uint32_t* offsets /* states + 1 */, float* values, int32_t* best);

/* ---- model store: Model / ModelManager (data_structures.h:43-157, 310-481) ---- */
FI_API size_t fi_model_bytes(const fi_learner* l);                                  /* blob size, fixed */
FI_API uint64_t fi_model_version(fi_learner* l, int player);                         /* getLatestVersion :475-480 */
/* getModel()->getData() + getVersion() (:433-438,135-138): consistent (version, bytes). */
FI_API int fi_model_get(fi_learner* l, int player, void* dst, size_t n, uint64_t* version);
/* waitForModelUpdate (:454-472): 1 if latest > current_version within timeout_ms, else 0. */
FI_API int fi_model_wait_update(fi_learner* l, int player, uint64_t current_version, int timeout_ms);
/* saveModel (:388-423): writes model_{p}_{iter}.bin and model_{p}_latest.bin in
 * checkpoint_location; file = little-endian u64 version + raw bytes (:105-110). An optional
 * trailing section carries optimiser state (SURVEY.md 8f rank 4); readers of the reference
 * format load the prefix unchanged. The section is "FIOPT001" for Adam / AdamW / SGD and
 * "FIRMS001" for RMSProp (both: u64 step, u64 n, m[n], v[n] as fi_learner_get_opt_state names them).
 * A learner that finds the other family's section loads the weights only (one line on stderr). */
FI_API int fi_model_save(fi_learner* l, int player, uint64_t iteration, int with_optimizer_state);
/* loadModels (:337-385): `dir`/model_{p}_latest.bin, else the highest-numbered model_{p}_N.bin. */
FI_API int fi_model_load(fi_learner* l, const char* dir);

/* ---- data parallelism across the GPUs of one box (SURVEY.md section 8e) ---- */
#define FI_DP_ID_BYTES 128
/* Rank 0 creates one id per player (players step concurrently, so each owns a communicator);
 * the host transports them to the other ranks (MPI_Bcast in the reference's MPI mains,
 * torch.distributed in bench.py); every rank then joins. After this, fi_learner_step
 * sum-allreduces the flat gradient arena (NCCL over NVLink/NVSwitch) between backward and the
 * optimiser update, and mean losses divide by the global batch. NCCL is bound with dlopen
 * (FI_NCCL_LIB overrides the library name); FI_ERR_NCCL if it cannot be found. */
FI_API int fi_dp_create_id(void* id_out /* FI_DP_ID_BYTES */);
FI_API int fi_learner_dp_init(fi_learner* l, const void* ids /* num_players * FI_DP_ID_BYTES */, int rank, int world_size);
FI_API int fi_learner_dp_world(const fi_learner* l);

/* Pinned (page-locked, portable) host memory for callers that stage their own batches: a
 * pinned source lets fi_learner_stage_batch DMA straight from the caller's buffer. */
FI_API void* fi_host_alloc(size_t bytes);
FI_API void fi_host_free(void* p);

/* ============================ operator layer =============================================
 * Stream-ordered launches of the individual sm_100a kernels on caller-owned DEVICE
 * pointers, for kernel-level parity tests and the roofline sweeps (BASELINE.json configs[4]).
 * `stream` is a cudaStream_t (NULL = legacy default stream). */

/* dst[i, :] = ring[(first + i) % capacity, :], i < m. Bit-exact byte copy; slot_bytes % 16 == 0. */
FI_API int fi_op_gather(const void* ring_base, size_t capacity, size_t slot_bytes, size_t first, size_t m, void* dst, void* stream);

/* V-trace targets and policy-gradient advantages, trajectory-major [m,t] fp32 arrays.
 * 24 B/transition of algorithmic traffic (+4 B/trajectory). */
FI_API int fi_op_vtrace(int m, int t, const float* log_rho, const float* discount, const float* reward, const float* value, const float* bootstrap, float rho_bar, float c_bar, float pg_rho_bar, float lambda_, float* vs, float* pg_adv, void* stream);

/* Fused V-trace loss head on a gathered batch [m, t records]: reads head[m*t, ldh] (16 policy
 * logits + value per row, ldh >= 17) and the records' behaviour logits / action / reward /
 * discount / bootstrap; writes dhead (same layout), optionally vs / pg_adv [m*t], and ADDS
 * {total, pg, baseline, entropy} into losses[4] (double, zeroed by the caller). */
FI_API int fi_op_vtrace_loss_head(const void* batch, int m, int t, const float* head, int ldh, float rho_bar, float c_bar, float pg_rho_bar, float lambda_, float baseline_cost, float entropy_cost, float* dhead, float* vs, float* pg_adv, double* losses, void* stream);
/* Same, with legal-action masking: the softmaxes, entropy and d(head) run over each record's legal word | the action's bit
 * (see FI_REC_WORD_LEGAL); d(head) is 0 in every column outside that support. */
FI_API int fi_op_vtrace_loss_head_legal(const void* batch, int m, int t, const float* head, int ldh, float rho_bar, float c_bar, float pg_rho_bar, float lambda_, float baseline_cost, float entropy_cost, float* dhead, float* vs, float* pg_adv, double* losses, void* stream);

/* One fused optimiser update over n contiguous fp32 values (28 B/param for Adam).
 * step counts from 1; grad_scale multiplies g first (1/world for averaged gradients). */
FI_API int fi_op_adam(int opt_kind, double lr, int64_t step, size_t n, float* p, const float* g, float* m, float* v, float grad_scale, void* stream);

/* *norm = ||g||_2 over n fp32 values (squares and sums in double, deterministic), *coef = min(1, max_norm / (*norm + 1e-6))
 * (torch.nn.utils.clip_grad_norm_). Both outputs are device pointers; g 16-byte aligned; max_norm > 0. 4 B/param. The first
 * call on a stream allocates a small scratch that later calls on that stream reuse; that first call cannot be captured. */
FI_API int fi_op_grad_norm_clip(size_t n, const float* g, double max_norm, double* norm, float* coef, void* stream);
/* One RMSProp update (torch.optim.RMSprop, centered=False, weight_decay=0) over n fp32 values; momentum_buf is used (and may
 * be NULL otherwise) when momentum > 0. coef (device float, may be NULL) multiplies g first, e.g. fi_op_grad_norm_clip's.
 * 20 B/param (28 with momentum). */
FI_API int fi_op_rmsprop(double lr, double alpha, double eps, double momentum, size_t n, float* p, const float* g, float* square_avg,
                         float* momentum_buf, const float* coef /* may be NULL */, void* stream);

/* C[m,n] = op(A) op(B) (+bias, ReLU). trans: 0 = "NT" A[m,k] B[n,k]; 1 = "NN" A[m,k] B[k,n];
 * 2 = "TN" A[k,m] B[k,n]. mode: fi_gemm_mode. fp32 in/out, fp32-accurate accumulation. */
FI_API size_t fi_op_gemm_workspace_bytes(int trans, int m, int n, int k, int mode);
FI_API int fi_op_gemm(int trans, int m, int n, int k, const float* a, int lda, const float* b, int ldb, float* c, int ldc, const float* bias, int relu, int mode, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* FI_LEARNER_H */
