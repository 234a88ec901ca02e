// tcgen05 GEMM for sm_100a with fp32-accurate products on the 5th-generation tensor cores: every operand is carried as a
// pair of 11-bit-significand numbers and every product costs three tensor-core products. Two operand formats, one kernel
// (template parameter H):
//
//   3xTF32 (H = 0)  x = hi + lo, hi = x with the low 13 mantissa bits cleared (a TF32 number), lo = x - hi; fp32 arrays.
//   3xFP16 (H = 1)  x * s = hi + lo' / 2048 with hi, lo' fp16 arrays and s a per-tensor power of two kept on the device
//                   (HScale): kind::f16 MMAs run at twice the kind::tf32 rate on half the shared-memory bytes per
//                   reduction element. The scale of a GEMM output is derived on the device, before the GEMM runs, from the
//                   bound k * max|A| * max|B| (+ max|bias|) so nothing can overflow fp16; each epilogue measures the true
//                   max |x| of what it wrote so that bounds stay one layer loose. See DESIGN.md 3.1 for the error analysis.
//
// The learner's tolerance (parameters within 1e-5 of an fp32/float64 reference) rules out plain TF32 / bf16 operands. Each
// product needs
//     main += A_hi B_hi            corr += A_hi B_lo + A_lo B_hi      (A_lo B_lo ~ 2^-22 relative is dropped),
// issued as TWO instructions per k-slice: B_hi and B_lo tiles are adjacent in shared memory, so one N = 2*BN MMA
// computes A_hi [B_hi | B_lo] into [main | corr] (adjacent TMEM columns) and one N = BN MMA adds A_lo B_hi to corr.
// Measured on B200: the tensor core adds into its fp32 accumulator with truncation towards zero, a few ulp
// of the running sum per MMA (error grew linearly with K: 2.4e-5 at K=32, 4.6e-4 at K=512 on sums of
// magnitude ~20 when one accumulator took all of K). The products therefore accumulate in TMEM only over
// a CHUNK of K = 128 (4 k-blocks of 32 tf32 / 2 k-blocks of 64 fp16); the promotion warps then add the chunk
// (main + corr, corr scaled by 2^-11 in the fp16 format) to fp32 register accumulators with round-to-nearest (the scheme
// of Ootomo & Yokota 2022, at chunk granularity): 6.5e-5 at K=512 (1.7e-6 of the largest sum). Halving the chunk only
// gave 5.0e-5: what is left is the truncation inside each MMA's own sum, which no promotion schedule removes.
//
// Kernel anatomy (one CTA per SM, persistent over output tiles; 128 control threads + 4 or 8 promotion warps):
//   warp 0     TMA producer: cp.async.bulk.tensor 128-byte-swizzled boxes of A_hi, A_lo, B_hi, B_lo into a
//              multi-stage shared-memory ring, completion on mbarriers;
//   warp 1     MMA issuer: one elected lane issues 2 tcgen05.mma (M=128; N=2*BN and N=BN) x 4 k-slices of 32 bytes per
//              k-block; tcgen05.commit releases the smem stage / publishes a finished chunk;
//   warp 2     TMEM allocator: 2 chunk buffers of [main | corr] = 2*BN fp32 columns each, so the promotion of
//              chunk i overlaps the MMAs of chunk i+1 and the epilogue of tile j those of tile j+1;
//   warps 4..  promotion + epilogue, two warps per TMEM lane quarter (each owns half of the tile's columns):
//              tcgen05.ld (32 lanes x 32 columns) into register accumulators, then bias (through the accumulator's
//              initial value) / ReLU / ReLU-mask and either a plain fp32 store or the hi/lo split store (TMA) that feeds
//              the next GEMM.
// Operand layouts (UMMA "major"): K-major tiles are [rows][128 bytes of k] (128B swizzle, 16-byte atoms); MN-major tiles
// are boxes of [k][128 bytes of mn] (the reduction index is the slow one): tf32 only supports the 128B swizzle with
// 32-byte atoms there ([32 k][32 mn] boxes), fp16 uses the ordinary one ([64 k][64 mn] boxes). So dgrad (B = W[n,k] read
// along n) and wgrad (both operands read along the batch rows) need no transposed copies.
#include <cooperative_groups.h>
#include <cuda.h>
#include <cuda_fp16.h>

#include <cstdlib>
#include <mutex>
#include <unordered_map>

#include "fi_internal.cuh"
#include "tc_ptx.cuh"

namespace fi {

constexpr int kTcBM = 128;       // UMMA M (rows of the accumulator = TMEM lanes)
constexpr int kTcRowBytes = 128;     // one k-block of one matrix row = 128 bytes = one swizzle row:
constexpr int kTcBK = 32;            //   32 fp32 (3xTF32) or
constexpr int kTcBKh = 64;           //   64 fp16 (3xFP16) reduction elements
constexpr int kTcCtrlThreads = 128;  // warps 0..3: TMA producer, MMA issuer, TMEM allocator, (idle)
constexpr int kTcChunkK = 128;       // reduction elements accumulated in TMEM before promotion to registers (16 wide MMAs)
constexpr int kTcSmemLimit = 227 * 1024;

struct TcEpilogue {
    float* c;            // plain fp32 output (may be null)
    int ldc;
    void* c_hi;          // split output (may be null): float or __half arrays, as the operands
    void* c_lo;
    int ldc_split;
    const float* bias;   // [n] or null
    const float* mask;   // [m, ldmask]: out = mask > 0 ? out : 0 (ReLU backward), or null
    int ldmask;
    const uint32_t* mask_bits;  // bit-packed ReLU decisions [m, mask_ldw words] (bit j of word w = column 32w + j), or null
    uint32_t* mask_bits_out;    // written by a ReLU epilogue for the backward pass, or null
    int mask_ldw;
    int relu;
    int transpose_out;   // c[col * ldc + row] (plain output only)
    int tma_split;       // c_hi / c_lo are written with TMA stores (map_c_hi / map_c_lo are valid)
    float* colsum_out;   // [4 * num_m_blocks, n]: column sums of the output over each warp's 32 rows (bias gradient), or null
    size_t split_stride; // elements between split-K slabs of c
    int plain_direct;    // plain row-major fp32 output with nothing but a bias: each lane stores its row's columns as 32-byte sectors
    int step_t;          // > 0: c is the recurrent kernels' blocked gate array (lstm_tc.cu, step_block_offset): row = b * step_t + s
    int step_nblk;       //      blocks of 64 batch rows
    // 3xFP16 format only
    const HScale* a_hs;  // operand scales: the accumulator is (A * sa)(B * sb), multiplied by inv_a * inv_b on the way out
    const HScale* b_hs;
    const HScale* bias_hs;  // bounds |bias| (null without bias)
    HScale* out_hs;      // split output: scale derived from k * amax_a * amax_b (+ amax_bias); amax measured by the epilogue
};

struct TcShape {
    int m, n, k;
    int num_m_blocks, num_n_blocks, num_splits, kb_per_split, num_kb;
    int dbg;  // FI_TC_DBG knock-out bits (tools/gemm_knockout.py; results are garbage, timings say what bounds the kernel):
              // 1 no TMA loads, 2 no MMAs, 4 no promotion loads, 8 no epilogue, 16 no A_lo B_hi MMA, 32 no TMA stores
    unsigned long long* trace;  // FI_TC_TRACE: per-role event log of the first CTAs (tools/gemm_trace.py), else null
};

// ---- pipeline trace (diagnostics) ----------------------------------------------------------------------------
// CTAs 0..kTraceCtas-1 log (clock64 << 8 | tag) per role: role 0 TMA producer, 1 MMA issuer, 2 first promotion warp.
constexpr int kTraceCtas = 4, kTraceRoles = 3, kTraceCap = 4096;
struct TraceLog {
    unsigned long long* p = nullptr;
    int n = 0;
#if FI_TRACE_BUILD
    __device__ __forceinline__ void init(unsigned long long* base, int role) {
        if (base && blockIdx.x < kTraceCtas) p = base + ((size_t)blockIdx.x * kTraceRoles + role) * kTraceCap;
    }
    __device__ __forceinline__ void ev(unsigned tag) {
        if (p && n < kTraceCap) p[n++] = ((unsigned long long)clock64() << 8) | tag;
    }
#else   // product build: no hook costs an instruction (fi_internal.cuh)
    __device__ __forceinline__ void init(unsigned long long*, int) {}
    __device__ __forceinline__ void ev(unsigned) {}
#endif
};

// column sums of a 32 x 32 block held one row per lane (x[i] = column i of this lane's row) by recursive halving: after the
// step with offset o a lane keeps the half of its columns selected by its bit o, summed with its partner's; 31 shuffles, and
// lane j returns the sum of column j.
__device__ __forceinline__ float warp_colsum32(const float* x, int lane) {
    float y16[16], y8[8], y4[4], y2[2];
    const bool b16 = lane & 16, b8 = lane & 8, b4 = lane & 4, b2 = lane & 2, b1 = lane & 1;
#pragma unroll
    for (int i = 0; i < 16; i++) y16[i] = (b16 ? x[16 + i] : x[i]) + __shfl_xor_sync(0xFFFFFFFFu, b16 ? x[i] : x[16 + i], 16);
#pragma unroll
    for (int i = 0; i < 8; i++) y8[i] = (b8 ? y16[8 + i] : y16[i]) + __shfl_xor_sync(0xFFFFFFFFu, b8 ? y16[i] : y16[8 + i], 8);
#pragma unroll
    for (int i = 0; i < 4; i++) y4[i] = (b4 ? y8[4 + i] : y8[i]) + __shfl_xor_sync(0xFFFFFFFFu, b4 ? y8[i] : y8[4 + i], 4);
#pragma unroll
    for (int i = 0; i < 2; i++) y2[i] = (b2 ? y4[2 + i] : y4[i]) + __shfl_xor_sync(0xFFFFFFFFu, b2 ? y4[i] : y4[2 + i], 2);
    return (b1 ? y2[1] : y2[0]) + __shfl_xor_sync(0xFFFFFFFFu, b1 ? y2[0] : y2[1], 1);
}

// PAIR: two CTAs of a cluster (one SM pair) work on one 256 x BN tile with cta_group::2 MMAs. Each CTA holds its own
// 128 rows of A and HALF of the B tile (BN/2 rows), the tensor core reads the other half from the peer: the B operand
// traffic through each SM's shared memory halves (DESIGN.md 3.1: the 1-CTA kernel is shared-memory-bandwidth bound).
template <int BN, bool PAIR = false, bool W16 = false>
struct TcCfg {
    static constexpr int kBRows = PAIR ? BN / 2 : BN;                 // rows of the B tile held by one CTA
    static constexpr int kStageBytes = 2 * (kTcBM + kBRows) * kTcRowBytes;  // A_hi, A_lo, B_hi, B_lo
    static_assert(BN == 32 || BN == 64 || BN == 128, "BN");
    static_assert(!PAIR || BN == 128, "pair mode is built for BN = 128");
    static_assert(!W16 || BN == 128, "16 promotion warps: 128-wide tiles");
    static constexpr int kStages = PAIR ? 4 : (BN >= 128 ? 3 : 4);
    static constexpr int kTmemCols = 4 * BN;                          // 2 chunk buffers x [main | corr] (a power of two >= 32)
    // promotion + epilogue warps: two per TMEM lane quarter (each owns half of the tile's columns) once the tile is
    // wide enough, so that every SM sub-partition has two warps to interleave (one warp per scheduler issued at
    // ~0.25 instructions per clock and made the promotion side, not the MMAs, the critical path).
    // W16 (products whose every tile ends in the fp16 split epilogue: forward, dgrad): TWO GROUPS of eight such warps that
    // take the CTA's tiles alternately. A tile costs its promotion warps ~1700 clocks of promotions and ~5000 of epilogue
    // (issue-bound: ~10 instructions per output element) against ~6800 clocks of MMAs, and the two TMEM chunk buffers let
    // the issuer run only half a tile ahead: with one group the tensor pipe stood idle ~3000 clocks at every tile
    // boundary (profiles/r2_gemm_trace.md). With two groups the epilogue of tile t overlaps ALL of tile t+1's MMAs,
    // whose chunks the other group promotes. 2 control warps + 16: 576 threads, 112 registers each.
    static constexpr int kCtrlWarps = W16 ? 2 : 4;                    // TMA producer, MMA issuer (W16: also the TMEM allocator), [allocator, idle]
    static constexpr int kPromoWarps = W16 ? 16 : (BN >= 64 ? 8 : 4);
    static constexpr int kGroupWarps = W16 ? 8 : kPromoWarps;         // promotion warps working on one tile
    static constexpr int kColsPerWarp = BN / (kGroupWarps / 4);
    static constexpr int kThreads = 32 * (kCtrlWarps + kPromoWarps);
    static constexpr int kOutTileBytes = W16 ? 0 : kPromoWarps * 32 * 128;   // per promotion warp: one 32 x 128 B staging tile (W16: none)
    static constexpr int kSmemBytes = kStages * kStageBytes + kOutTileBytes + 1024 /*alignment slack*/ + 256 /*barriers*/;
    static_assert(kSmemBytes <= kTcSmemLimit, "shared memory budget");
};

// One kernel for the three operand-major combinations. A_MN / B_MN: operand is MN-major (reduction index slow).
// H: 3xFP16 operand format (fp16 hi / lo' pairs with per-tensor scales) instead of 3xTF32.
template <int BN, bool A_MN, bool B_MN, bool PAIR, bool H, bool W16 = false>
__global__ void __launch_bounds__(TcCfg<BN, PAIR, W16>::kThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
               const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo,
               const __grid_constant__ CUtensorMap map_c_hi, const __grid_constant__ CUtensorMap map_c_lo,
               const TcShape sh, const TcEpilogue ep) {
    using Cfg = TcCfg<BN, PAIR, W16>;
    static_assert(!W16 || H, "16 promotion warps exist for the fp16 format only");
    constexpr int kStages = Cfg::kStages;
    static_assert(!H || BN >= 64, "the fp16 format needs 64-wide MN blocks");
    constexpr int BK = H ? kTcBKh : kTcBK;            // reduction elements per k-block
    constexpr int kChunk = kTcChunkK / BK;            // k-blocks per TMEM chunk
    constexpr int kBoxMN = H ? 64 : 32;               // MN extent of one MN-major box (128 bytes)
    constexpr uint32_t kABytes = kTcBM * kTcRowBytes; // one of A_hi / A_lo
    constexpr uint32_t kBBytes = Cfg::kBRows * kTcRowBytes;
    const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;   // 0 = leader (issues the MMAs)
    const int unit = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;        // CTA (or CTA pair) index
    const int num_units = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    constexpr int kTileM = PAIR ? 2 * kTcBM : kTcBM;
    constexpr uint32_t kBoxBytes = BK * kTcRowBytes;  // one MN-major box: BK k-rows x 128 B
    extern __shared__ uint8_t smem_raw[];
    const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;     // swizzle atoms need 1024 B alignment
    // barriers: full[kStages], empty[kStages], main_full[2], main_empty[2]
    const uint32_t out_tiles = smem_base + kStages * Cfg::kStageBytes;    // 1024-byte aligned: TMA-store staging, 8 KB per warp
    const uint32_t bar_base = out_tiles + Cfg::kOutTileBytes;
    const uint32_t tmem_slot = bar_base + (2 * kStages + 8) * 8;
    auto full_bar = [&](int s) { return bar_base + 8u * s; };
    auto empty_bar = [&](int s) { return bar_base + 8u * (kStages + s); };
    // chunk barriers, one pair per (promotion group g, TMEM buffer b): with two tile-alternating groups (W16) each group
    // sees every phase of ITS barriers in order (a barrier shared by the groups would advance by whole tiles while one of
    // them is in its epilogue, and a parity wait cannot tell phases two apart)
    auto main_full_bar_g = [&](int g, int b) { return bar_base + 8u * (2 * kStages + 2 * g + b); };
    auto main_empty_bar_g = [&](int g, int b) { return bar_base + 8u * (2 * kStages + 4 + 2 * g + b); };
    auto main_full_bar = [&](int b) { return main_full_bar_g(0, b); };
    auto main_empty_bar = [&](int b) { return main_empty_bar_g(0, b); };

    const int warp = __shfl_sync(0xFFFFFFFFu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // warp index: provably warp-uniform
    float tmax_kernel = 0.f;  // fp16 format: running max |output| of this thread (published once at the end)
    const int tiles = sh.num_m_blocks * sh.num_n_blocks;
    const int total_work = tiles * sh.num_splits;

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kStages; s++) {
            mbar_init(full_bar(s), 1);
            mbar_init(empty_bar(s), 1);
        }
        for (int s = 0; s < (W16 ? 4 : 2); s++) {   // s = 2 * group + buffer
            mbar_init(main_full_bar_g(s >> 1, s & 1), 1);
            // one arrival per promotion warp; in pair mode the leader's barrier also collects the peer's warps
            mbar_init(main_empty_bar_g(s >> 1, s & 1), (PAIR ? 2 : 1) * Cfg::kGroupWarps);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    constexpr int kAllocWarp = W16 ? 1 : 2;
    if (warp == kAllocWarp) {
        __syncwarp();
        if constexpr (PAIR) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)Cfg::kTmemCols)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)Cfg::kTmemCols)
                         : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    tc_fence_before();
    if constexpr (PAIR) cluster_sync_all();  // both CTAs' barriers are initialised before any remote arrive / multicast commit
    else __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");
    // Programmatic dependent launch (launch_variant sets the attribute): everything above -- barrier initialisation, the TMEM
    // allocation, the cluster handshake -- touches no global memory and may run while the previous kernel of the stream is
    // still draining its last tiles; from here on this grid reads and writes what that kernel produced, so it waits for it
    // (completion and visibility of all its memory operations). Then it lets ITS successor start the same way: the
    // successor's CTAs become resident as this grid's CTAs exit and wait at this point themselves. Without the launch
    // attribute both instructions do nothing.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    // TMEM columns of chunk buffer b: main at [2b*BN, 2b*BN + BN), corr at [2b*BN + BN, 2b*BN + 2BN)

    if (warp == 0) {
        // ===================== TMA producer (warp-uniform; the loads are issued by one elected lane) =====================
        {
            int stage = 0;
            uint32_t phase = 0;
            auto load = [&](uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
                if constexpr (PAIR) tma_load_2d_pair(dst, map, bar, c0, c1);
                else tma_load_2d(dst, map, bar, c0, c1);
            };
            TraceLog tl;
            if (lane == 0) tl.init(sh.trace, 0);
            for (int w = unit; w < total_work; w += num_units) {
                const int tile = w % tiles, split = w / tiles;
                // this CTA's rows of A and rows of the B tile (pair mode: the second CTA takes the second half of each)
                const int m0 = (tile / sh.num_n_blocks) * kTileM + (int)cta_rank * kTcBM;
                const int n0 = (tile % sh.num_n_blocks) * BN + (int)cta_rank * Cfg::kBRows * (PAIR ? 1 : 0);
                const int kb0 = split * sh.kb_per_split, kb1 = min(sh.num_kb, kb0 + sh.kb_per_split);
                for (int kb = kb0; kb < kb1; kb++) {
                    mbar_wait(empty_bar(stage), phase ^ 1);
                    tl.ev(1);
                    const uint32_t bar = full_bar(stage);
                    if (!PAIR && (sh.dbg & 1)) {
                        if (elect_one()) mbar_arrive(bar);
                        __syncwarp();
                        if (++stage == kStages) { stage = 0; phase ^= 1; }
                        continue;
                    }
                    const uint32_t a_hi = smem_base + stage * Cfg::kStageBytes, a_lo = a_hi + kABytes;
                    const uint32_t b_hi = a_lo + kABytes, b_lo = b_hi + kBBytes;
                    const int k0 = kb * BK;
                    if (elect_one()) {
                    // pair mode: both CTAs' loads are credited to the leader's barrier, which expects both stages
                    if (!PAIR || cta_rank == 0) mbar_expect_tx(bar, (PAIR ? 2 : 1) * Cfg::kStageBytes);
                    if constexpr (!A_MN) {
                        load(a_hi, &map_a_hi, bar, k0, m0);
                        load(a_lo, &map_a_lo, bar, k0, m0);
                    } else {
#pragma unroll
                        for (int j = 0; j < kTcBM / kBoxMN; j++) {
                            load(a_hi + j * kBoxBytes, &map_a_hi, bar, m0 + j * kBoxMN, k0);
                            load(a_lo + j * kBoxBytes, &map_a_lo, bar, m0 + j * kBoxMN, k0);
                        }
                    }
                    if constexpr (!B_MN) {
                        load(b_hi, &map_b_hi, bar, k0, n0);
                        load(b_lo, &map_b_lo, bar, k0, n0);
                    } else {
#pragma unroll
                        for (int j = 0; j < Cfg::kBRows / kBoxMN; j++) {
                            load(b_hi + j * kBoxBytes, &map_b_hi, bar, n0 + j * kBoxMN, k0);
                            load(b_lo + j * kBoxBytes, &map_b_lo, bar, n0 + j * kBoxMN, k0);
                        }
                    }
                    }
                    __syncwarp();
                    tl.ev(2);
                    if (++stage == kStages) { stage = 0; phase ^= 1; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer (warp-uniform; MMAs and commits are issued by one elected lane) =====================
        if (cta_rank == 0) {
            const uint32_t tmem_base_u = __shfl_sync(0xFFFFFFFFu, tmem_base, 0);   // a value the compiler knows to be warp-uniform
            constexpr uint32_t idesc_wide = umma_idesc(kTcBM, 2 * BN, A_MN ? 1 : 0, B_MN ? 1 : 0, H ? 1 : 0);  // A_hi [B_hi | B_lo]
            constexpr uint32_t idesc_half = umma_idesc(kTileM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0, H ? 1 : 0);      // A_lo B_hi (pair: every product)
            // K-major (128B swizzle, 16 B atoms): a k-slice of 8 fp32 is 32 bytes inside the 128-byte row; 8-row groups
            // are 1024 B apart (SBO). MN-major (128B swizzle, 32 B atoms): a k-slice is 8 rows of 128 B = two 4-row
            // atoms 512 B apart (SBO); 32-wide MN blocks are one TMA box (4096 B) apart (LBO). The B_lo tile follows
            // the B_hi tile with the same strides, so a descriptor at B_hi with N = 2*BN covers both.
            // fp16 format: a k-slice is 16 halves = the same 32 bytes of a K-major row; MN-major tiles use the plain
            // 128B swizzle (16 B atoms) in boxes of [64 k][64 mn]: a k-slice is 16 rows = two 8-row groups 1024 B apart
            // (SBO), 64-wide MN blocks are one box (8192 B) apart (LBO).
            constexpr uint32_t kMnStep = H ? 2048u : 1024u, kMnSbo = H ? 1024u : 512u, kMnType = H ? 2u : 1u;
            constexpr uint32_t a_step = (A_MN ? kMnStep : 32u) >> 4, b_step = (B_MN ? kMnStep : 32u) >> 4;
            constexpr uint32_t a_lbo = A_MN ? kBoxBytes : 0u, b_lbo = B_MN ? kBoxBytes : 0u;
            constexpr uint32_t a_sbo = A_MN ? kMnSbo : 1024u, b_sbo = B_MN ? kMnSbo : 1024u;
            // descriptor words that never change: [32,46) SBO, [46,48) version 1, [61,64) layout type
            constexpr uint32_t a_hi_word = (a_sbo >> 4) | (1u << 14) | ((A_MN ? kMnType : 2u) << 29);
            constexpr uint32_t b_hi_word = (b_sbo >> 4) | (1u << 14) | ((B_MN ? kMnType : 2u) << 29);
            auto mma = [](uint32_t d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
                if constexpr (PAIR) {
                    if constexpr (H) tc_mma_f16_pair(d, da, db, idesc, accumulate);
                    else tc_mma_tf32_pair(d, da, db, idesc, accumulate);
                } else {
                    if constexpr (H) tc_mma_f16(d, da, db, idesc, accumulate);
                    else tc_mma_tf32(d, da, db, idesc, accumulate);
                }
            };
            auto desc = [](uint32_t hi_word, uint32_t lo_word) { return ((uint64_t)hi_word << 32) | lo_word; };
            int stage = 0, mb = 0;
            uint32_t phase = 0, mphase = 0;
            TraceLog tl;
            if (lane == 0) tl.init(sh.trace, 1);
            // W16: the group that drains this tile's chunks, the group whose chunk each TMEM buffer holds (bit b; valid from
            // the buffer's second use on) and the parity of the next drain expected from (group g, buffer b) (bit 2g + b)
            uint32_t grp = 0, owner_bits = 0, drain_parity = 0, chunk_no = 0;
            for (int w = unit; w < total_work; w += num_units) {
                const int split = w / tiles;
                const int kb0 = split * sh.kb_per_split, kb1 = min(sh.num_kb, kb0 + sh.kb_per_split);
                for (int kc = kb0; kc < kb1; kc += kChunk) {
                    if constexpr (W16) {
                        if (chunk_no >= 2) {   // the previous chunk in this TMEM buffer must have been promoted, by whichever group
                            const uint32_t pg = (owner_bits >> mb) & 1u, bit = 2u * pg + (uint32_t)mb;
                            mbar_wait(main_empty_bar_g((int)pg, mb), (drain_parity >> bit) & 1u);
                            drain_parity ^= 1u << bit;
                        }
                        owner_bits = (owner_bits & ~(1u << mb)) | (grp << mb);
                        chunk_no++;
                    } else {
                        mbar_wait(main_empty_bar(mb), mphase ^ 1);
                    }
                    tl.ev(10);
                    tc_fence_after();
                    const uint32_t tmem_main = tmem_base_u + (uint32_t)(mb * 2 * BN), tmem_corr = tmem_main + BN;
                    const int kce = min(kb1, kc + kChunk);
                    for (int kb = kc; kb < kce; kb++) {
                        mbar_wait(full_bar(stage), phase);
                        tl.ev(11);
                        tc_fence_after();
                        const uint32_t a_hi = smem_base + stage * Cfg::kStageBytes, a_lo = a_hi + kABytes, b_hi = a_lo + kABytes;
                        const uint32_t b_lo = b_hi + kBBytes;
                        // low descriptor words: [0,14) start address >> 4, [16,30) LBO >> 4
                        const uint32_t la_hi = ((a_hi >> 4) & 0x3FFFu) | ((a_lbo >> 4) << 16);
                        const uint32_t la_lo = ((a_lo >> 4) & 0x3FFFu) | ((a_lbo >> 4) << 16);
                        const uint32_t lb_hi = ((b_hi >> 4) & 0x3FFFu) | ((b_lbo >> 4) << 16);
                        const uint32_t lb_lo = ((b_lo >> 4) & 0x3FFFu) | ((b_lbo >> 4) << 16);
                        if (elect_one()) {
#pragma unroll
                        for (int ks = 0; ks < 4; ks++) {  // 4 k-slices of 32 bytes (8 tf32 / 16 fp16) per k-block
                            const uint64_t da_hi = desc(a_hi_word, la_hi + ks * a_step);
                            const uint64_t da_lo = desc(a_hi_word, la_lo + ks * a_step);
                            const uint64_t db = desc(b_hi_word, lb_hi + ks * b_step);
                            const uint32_t first = (kb > kc || ks > 0) ? 1u : 0u;
                            if constexpr (PAIR) {
                                // each CTA holds one half of B_hi and of B_lo, so the halves are not adjacent across the
                                // pair: three M=256 x N=BN products per k-slice (descriptors are CTA-local offsets, valid in both)
                                const uint64_t db_lo = desc(b_hi_word, lb_lo + ks * b_step);
                                mma(tmem_main, da_hi, db, idesc_half, first);     // main (+)= A_hi B_hi
                                mma(tmem_corr, da_hi, db_lo, idesc_half, first);  // corr (+)= A_hi B_lo
                                mma(tmem_corr, da_lo, db, idesc_half, 1u);        // corr  += A_lo B_hi
                            } else {
                                (void)lb_lo;
                                if (!(sh.dbg & 2)) mma(tmem_main, da_hi, db, idesc_wide, first);  // [main | corr] (+)= A_hi [B_hi | B_lo]
                                if (!(sh.dbg & 18)) mma(tmem_corr, da_lo, db, idesc_half, 1u);    // corr += A_lo B_hi
                            }
                        }
                        tl.ev(12);
                        // frees the smem stage (in both CTAs of a pair) once these MMAs have read it
                        if constexpr (PAIR) tc_commit_pair(empty_bar(stage));
                        else tc_commit(empty_bar(stage));
                        }
                        __syncwarp();
                        tl.ev(13);
                        if (++stage == kStages) { stage = 0; phase ^= 1; }
                    }
                    if (elect_one()) {
                        if constexpr (PAIR) tc_commit_pair(main_full_bar_g((int)grp, mb));  // chunk complete, published to both CTAs
                        else tc_commit(main_full_bar_g((int)grp, mb));
                    }
                    __syncwarp();
                    tl.ev(14);
                    if (++mb == 2) { mb = 0; mphase ^= 1; }
                }
                if constexpr (W16) grp ^= 1u;   // tiles alternate between the two promotion groups
            }
        }
    } else if (warp >= Cfg::kCtrlWarps) {
        // ===================== promotion + epilogue =====================
        constexpr int CW = Cfg::kColsPerWarp;     // columns of the tile owned by this warp
        const int pw = warp - Cfg::kCtrlWarps;
        const int q = warp & 3;                   // TMEM lane quarter this warp may access (warp id % 4)
        const int ord = pw >> 2;                  // ordinal among the promotion warps of this quarter
        const int group = W16 ? (ord >> 1) : 0;   // W16: which of the two tile-alternating groups
        constexpr int kGroups = W16 ? 2 : 1;
        const int nc0 = (W16 ? (ord & 1) : ord) * CW;   // first tile column of this warp
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        int mb = 0;
        uint32_t mphase = 0;
        // pair mode: the MMA issuer lives in CTA 0, which collects both CTAs' releases of (this group's) chunk buffers
        const uint32_t leader_main_empty0 = PAIR ? map_to_cta(main_empty_bar_g(group, 0), 0) : 0u;
        const uint32_t leader_main_empty1 = PAIR ? map_to_cta(main_empty_bar_g(group, 1), 0) : 0u;
        // fp16 format: corr carries lo' = 2048 lo; the accumulator is in units of scale_a * scale_b
        constexpr float kCorrMul = H ? (1.f / 2048.f) : 1.f;
        float out_mul = 1.f, out_scale = 1.f, acc_unit = 1.f;
        // TMA-split epilogues take the bias through the accumulator's initial value (loaded while the first chunk is
        // still being computed) instead of 64 dependent loads per thread on the epilogue's critical path
        constexpr bool kFastSplit = H && CW == 64;   // the fp16 split epilogue below
        const bool bias_prefetch = ep.bias != nullptr && (ep.tma_split || ep.plain_direct);
        const bool bias_in_acc = bias_prefetch && !(kFastSplit && ep.tma_split);   // the fp16 split epilogue adds the prefetched bias itself
        if constexpr (H) {
            out_mul = ep.a_hs->inv * ep.b_hs->inv;
            acc_unit = ep.a_hs->scale * ep.b_hs->scale;
            if (ep.out_hs) {
                const float bound = (float)sh.k * ep.a_hs->amax * ep.b_hs->amax + (ep.bias_hs ? ep.bias_hs->amax : 0.f);
                out_scale = hscale_from_bound(bound);
                if (blockIdx.x == 0 && pw == 0 && lane == 0) {
                    ep.out_hs->scale = out_scale;
                    ep.out_hs->inv = 1.f / out_scale;
                    ep.out_hs->bound = bound;
                }
            }
        }
        TraceLog tl;
        if (pw == 0 && lane == 0) tl.init(sh.trace, 2);
        float bias_next[CW / 32], bias_cur[CW / 32];
#pragma unroll
        for (int c = 0; c < CW / 32; c++) bias_next[c] = bias_cur[c] = 0.f;
        const int first_work = unit + group * num_units, work_step = kGroups * num_units;
        // W16: the issuer numbers the chunks of all the CTA's tiles consecutively (buffer = number & 1); this group's
        // tiles are every other one. No split-K on this path: every tile has the same number of chunks.
        const int chunks_per_tile = (sh.kb_per_split + kChunk - 1) / kChunk;
        int tile_seq = group;
        uint32_t full_parity = 0;   // W16: parity of the next phase of main_full(group, b) this warp waits for (bit b)
        if (bias_prefetch && first_work < total_work) {
            const int fn0 = ((first_work % tiles) % sh.num_n_blocks) * BN + nc0;
#pragma unroll
            for (int c = 0; c < CW / 32; c++) bias_next[c] = (fn0 + c * 32 + lane < sh.n) ? __ldg(ep.bias + fn0 + c * 32 + lane) : 0.f;
        }
        for (int w = first_work; w < total_work; w += work_step, tile_seq += kGroups) {
            const int tile = w % tiles, split = w / tiles;
            const int m0 = (tile / sh.num_n_blocks) * kTileM + (int)cta_rank * kTcBM, n0 = (tile % sh.num_n_blocks) * BN;
            const int kb0 = split * sh.kb_per_split, kb1 = min(sh.num_kb, kb0 + sh.kb_per_split);
            const int row = m0 + q * 32 + lane;
            const bool row_ok = row < sh.m;
            if constexpr (W16) mb = (tile_seq * chunks_per_tile) & 1;   // TMEM buffers alternate over ALL the CTA's chunks
            float acc[CW];
            if (bias_prefetch && !bias_in_acc) {
                // lane l holds the bias of column 32 c + l of this warp's range, fetched one tile ahead: the epilogue reads it
                // with shuffles (no global-load latency on the epilogue's critical path: with 227 KB of shared memory there
                // is no L1 left, every load is an L2 round trip)
#pragma unroll
                for (int c = 0; c < CW / 32; c++) bias_cur[c] = bias_next[c];
                const int wn = w + work_step;
                if (wn < total_work) {
                    const int nn0 = ((wn % tiles) % sh.num_n_blocks) * BN + nc0;
#pragma unroll
                    for (int c = 0; c < CW / 32; c++) bias_next[c] = (nn0 + c * 32 + lane < sh.n) ? __ldg(ep.bias + nn0 + c * 32 + lane) : 0.f;
                }
            }
            if (bias_in_acc) {
                // lane l holds the bias of columns l and 32 + l of this warp's range, fetched one tile ahead (below), and
                // the initial accumulators are built with shuffles: no load latency at the start of a tile, where the
                // MMAs of the next chunk are already waiting for the promotion warps
#pragma unroll
                for (int i = 0; i < CW; i++) acc[i] = __shfl_sync(0xFFFFFFFFu, i < 32 ? bias_next[0] : bias_next[CW > 32 ? 1 : 0], i & 31) * acc_unit;
                const int wn = w + work_step;
                if (wn < total_work) {
                    const int nn0 = ((wn % tiles) % sh.num_n_blocks) * BN + nc0;
#pragma unroll
                    for (int c = 0; c < CW / 32; c++) bias_next[c] = (nn0 + c * 32 + lane < sh.n) ? __ldg(ep.bias + nn0 + c * 32 + lane) : 0.f;
                }
            } else {
#pragma unroll
                for (int i = 0; i < CW; i++) acc[i] = 0.f;
            }
            // bit-packed ReLU mask of this thread's row: one 16-byte load per tile, issued before the k-loop so that
            // its latency hides behind the MMAs (a float mask read in the epilogue was latency-bound: 4 warps per SM)
            uint32_t mw[CW / 32];
#pragma unroll
            for (int c = 0; c < CW / 32; c++) mw[c] = 0xFFFFFFFFu;
            if (ep.mask_bits && row_ok) {
#pragma unroll
                for (int c = 0; c < CW / 32; c++)
                    if (n0 + nc0 + c * 32 < sh.n) mw[c] = __ldg(ep.mask_bits + (size_t)row * ep.mask_ldw + ((n0 + nc0) >> 5) + c);
            }
            for (int kc = kb0; kc < kb1; kc += kChunk) {
                if constexpr (W16) {
                    mbar_wait(main_full_bar_g(group, mb), (full_parity >> mb) & 1u);   // this group's own phase sequence per buffer
                    full_parity ^= 1u << mb;
                } else {
                    mbar_wait(main_full_bar(mb), mphase);
                }
                tl.ev(20);
                tc_fence_after();
                if (!(sh.dbg & 4)) {
                    if constexpr (W16) {   // 18 warps: 96 registers per thread, 64 of them accumulators: the chunk comes in pieces
#pragma unroll
                        for (int c = 0; c < CW / 16; c++) {
                            uint32_t v[8], u[8], v2[8], u2[8];
                            tmem_ld8(tmem_base + lane_base + (uint32_t)(mb * 2 * BN + nc0 + c * 16), v);           // main
                            tmem_ld8(tmem_base + lane_base + (uint32_t)(mb * 2 * BN + BN + nc0 + c * 16), u);      // corr
                            tmem_ld8(tmem_base + lane_base + (uint32_t)(mb * 2 * BN + nc0 + c * 16 + 8), v2);
                            tmem_ld8(tmem_base + lane_base + (uint32_t)(mb * 2 * BN + BN + nc0 + c * 16 + 8), u2);
                            tmem_ld_wait();
#pragma unroll
                            for (int i = 0; i < 8; i++) {
                                acc[c * 16 + i] += fmaf(__uint_as_float(u[i]), kCorrMul, __uint_as_float(v[i]));
                                acc[c * 16 + 8 + i] += fmaf(__uint_as_float(u2[i]), kCorrMul, __uint_as_float(v2[i]));
                            }
                        }
                    } else {
#pragma unroll
                        for (int c = 0; c < CW / 32; c++) {
                            uint32_t v[32], u[32];
                            tmem_ld32(tmem_base + lane_base + (uint32_t)(mb * 2 * BN + nc0 + c * 32), v);       // main
                            tmem_ld32(tmem_base + lane_base + (uint32_t)(mb * 2 * BN + BN + nc0 + c * 32), u);  // corr
                            tmem_ld_wait();
#pragma unroll
                            for (int i = 0; i < 32; i++)  // round-to-nearest promotion
                                acc[c * 32 + i] += H ? fmaf(__uint_as_float(u[i]), kCorrMul, __uint_as_float(v[i]))
                                                     : __uint_as_float(v[i]) + __uint_as_float(u[i]);
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) {
                    if constexpr (PAIR) mbar_arrive_cluster(mb ? leader_main_empty1 : leader_main_empty0);  // the MMA issuer lives in CTA 0
                    else mbar_arrive(main_empty_bar_g(group, mb));
                }
                tl.ev(21);
                if (++mb == 2) { mb = 0; mphase ^= 1; }
            }
            tl.ev(22);   // tile's k loop done: the epilogue runs until the next tag 20
            if (sh.dbg & 8) continue;
            if constexpr (kFastSplit) {
                if (ep.tma_split) {
                    // ---- fp16 pair output (forward: bias + ReLU + ReLU bits; dgrad: ReLU mask + column sums) ----
                    // This warp owns 32 rows x CW columns = CW * 2 bytes of halves per matrix row and output array;
                    // everything is computed in registers (lane = row).
                    const int rbase = m0 + q * 32, colw0 = n0 + nc0;
                    if (colw0 < sh.n) {  // warp-uniform
                        const float mul = out_mul * out_scale, inv_scale = 1.f / out_scale;   // powers of two: exact
#pragma unroll
                        for (int c = 0; c < CW / 32; c++) {
                            const int col0 = colw0 + c * 32;
                            float* a = acc + c * 32;
                            if (ep.bias) {
                                const float bs = bias_cur[c] * out_scale;
#pragma unroll
                                for (int i = 0; i < 32; i++) a[i] = fmaf(a[i], mul, __shfl_sync(0xFFFFFFFFu, bs, i));
                            } else {
#pragma unroll
                                for (int i = 0; i < 32; i++) a[i] *= mul;
                            }
                            if (ep.relu) {
#pragma unroll
                                for (int i = 0; i < 32; i++) a[i] = fmaxf(a[i], 0.f);
                            }
                            if (ep.mask_bits) {
#pragma unroll
                                for (int i = 0; i < 32; i++) a[i] = ((mw[c] >> i) & 1u) ? a[i] : 0.f;
                            }
                            if (col0 < sh.n) {
                                if (ep.mask_bits_out) {
                                    // bit i = (a[i] > 0): 0 - bits(a[i]) is negative exactly for positive floats (+0 -> 0, negative
                                    // floats -> positive integers), and a funnel shift moves its sign bit into the word: 2 integer
                                    // instructions per element
                                    uint32_t bits = 0;
#pragma unroll
                                    for (int i = 31; i >= 0; i--) bits = __funnelshift_l((uint32_t)(0 - __float_as_int(a[i])), bits, 1);
                                    if (row_ok) ep.mask_bits_out[(size_t)row * ep.mask_ldw + (col0 >> 5)] = bits;
                                }
                                if (ep.colsum_out && m0 < sh.m) {   // (a pair's second CTA may lie wholly beyond the matrix)
                                    const float y1 = warp_colsum32(a, lane) * inv_scale;
                                    if (col0 + lane < sh.n) ep.colsum_out[(size_t)((m0 / kTcBM) * 4 + q) * sh.n + col0 + lane] = y1;
                                }
                            }
                        }
                        tl.ev(23);
                        // hi = fp16(t), lo' = fp16((t - hi) * 2048), 16 columns at a time (two full 32-byte sectors per lane and
                        // array), written straight from the registers. No shared memory on this path: every st.shared / ld.shared
                        // of a staged epilogue (round 1: TMA store; then a coalescing transpose) queued behind the tensor core's
                        // operand reads and the TMA fills (profiles/r2_gemm_trace.md).
                        __half2 hmax = __float2half2_rn(0.f);
                        __half* hi_row = static_cast<__half*>(ep.c_hi) + (size_t)row * ep.ldc_split + colw0;
                        __half* lo_row = static_cast<__half*>(ep.c_lo) + (size_t)row * ep.ldc_split + colw0;
#pragma unroll
                        for (int j = 0; j < CW / 16; j++) {
                            uint32_t h[8], l[8];
#pragma unroll
                            for (int e = 0; e < 8; e++) {
                                const float t0 = acc[16 * j + 2 * e], t1 = acc[16 * j + 2 * e + 1];
                                const __half2 h2 = __floats2half2_rn(t0, t1);
                                hmax = __hmax2(hmax, __habs2(h2));
                                const float2 hf = __half22float2(h2);
                                // t - hf is exact in fp32; x 2048 folded into one fma
                                const __half2 l2 = __floats2half2_rn(fmaf(t0, 2048.f, -2048.f * hf.x), fmaf(t1, 2048.f, -2048.f * hf.y));
                                h[e] = *reinterpret_cast<const uint32_t*>(&h2);
                                l[e] = *reinterpret_cast<const uint32_t*>(&l2);
                            }
                            if (row_ok && colw0 + j * 16 < sh.n && !(sh.dbg & 32)) {   // n is a multiple of 16 on this path
                                st_global_v8u(hi_row + j * 16, h);
                                st_global_v8u(lo_row + j * 16, l);
                            }
                        }
                        // max |output| from the rounded hi parts (within 2^-11 of the exact value; consumers only use it in bounds)
                        tmax_kernel = fmaxf(tmax_kernel, fmaxf(__low2float(hmax), __high2float(hmax)) * (1.001f * inv_scale));
                        tl.ev(29);
                    }
                    continue;
                }
            }
            if constexpr (W16) {
                __trap();   // the 16-warp variant is only launched for products that end in the fp16 split epilogue
            } else {
            if constexpr (H) {
#pragma unroll
                for (int i = 0; i < CW; i++) acc[i] *= out_mul;   // powers of two: exact
            }
            float* cplain = ep.c ? ep.c + (size_t)split * ep.split_stride : nullptr;
            if (ep.plain_direct) {
                // Plain fp32 rows (the LSTM input projection, split-K slabs of the weight gradients): the bias came through
                // the accumulator, so the lane's 32 consecutive columns go out as four 32-byte sectors each. The transposing
                // path below costs ~3 instructions per element; the 210 MB projection output was issue-bound on it (200 us).
                if (row_ok) {
#pragma unroll
                    for (int c = 0; c < CW / 32; c++) {
                        const int col0 = n0 + nc0 + c * 32;
                        float* dst = cplain + (size_t)row * ep.ldc + col0;
#pragma unroll
                        for (int j = 0; j < 4; j++)
                            if (col0 + 8 * j < sh.n) st_global_v8u(dst + 8 * j, reinterpret_cast<const uint32_t*>(&acc[c * 32 + 8 * j]));
                    }
                }
                continue;
            }
            if (ep.transpose_out) {
                // c[col * ldc + row]: lanes hold consecutive rows, so the register layout is already coalesced
                if (row_ok && cplain) {
#pragma unroll
                    for (int c = 0; c < CW / 32; c++) {
#pragma unroll
                        for (int i = 0; i < 32; i++) {
                            const int col = n0 + nc0 + c * 32 + i;
                            if (col < sh.n) cplain[(size_t)col * ep.ldc + row] = acc[c * 32 + i];
                        }
                    }
                }
                continue;
            }
            if (ep.mask_bits) {
#pragma unroll
                for (int c = 0; c < CW / 32; c++) {
#pragma unroll
                    for (int i = 0; i < 32; i++) acc[c * 32 + i] = ((mw[c] >> i) & 1u) ? acc[c * 32 + i] : 0.f;
                }
            }
            if (!H && ep.tma_split) {
                // hi/lo pair output: bias, ReLU, the split and the ReLU bit mask are computed in registers (lane = row),
                // the 32 x 32 block goes to this warp's 128B-swizzled staging tiles with conflict-free 16-byte stores, and
                // one lane hands both tiles to the TMA (cp.async.bulk.tensor store): no per-element address arithmetic
                // and no store instructions on the critical path of the 4 promotion warps. Rows / columns beyond the
                // matrix are clipped by the TMA.
                const uint32_t stage_tile = out_tiles + (uint32_t)pw * 4096u;  // one 32 x 128 B tile, reused for hi then lo
                const int rbase = m0 + q * 32;
#pragma unroll
                for (int c = 0; c < CW / 32; c++) {
                    const int col0 = n0 + nc0 + c * 32;
                    if (col0 >= sh.n) continue;  // warp-uniform
                    float x[32];
                    uint32_t bits = 0;
#pragma unroll
                    for (int i = 0; i < 32; i++) {
                        float t = acc[c * 32 + i];   // bias arrived through the accumulator
                        if (ep.relu) t = fmaxf(t, 0.f);
                        bits |= (t > 0.f ? 1u : 0u) << i;
                        x[i] = t;
                    }
                    if (ep.mask_bits_out && row_ok) ep.mask_bits_out[(size_t)row * ep.mask_ldw + (col0 >> 5)] = bits;
                    if (ep.colsum_out) {
                        // column sums over this warp's 32 rows; rows beyond m contribute exact zeros (zero-filled A rows)
                        const float y1 = warp_colsum32(x, lane);
                        if (col0 + lane < sh.n) ep.colsum_out[(size_t)((m0 / kTcBM) * 4 + q) * sh.n + col0 + lane] = y1;
                    }
                    // hi tile, then lo tile, through the same staging buffer: the sibling warp on this scheduler runs while
                    // lane 0 waits for the previous bulk store to have read the buffer
#pragma unroll
                    for (int part = 0; part < 2; part++) {
                        if (lane == 0) tma_store_wait_read();
                        __syncwarp();
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            float4 o;
                            const float h0 = __uint_as_float(__float_as_uint(x[4 * j + 0]) & 0xFFFFE000u);
                            const float h1 = __uint_as_float(__float_as_uint(x[4 * j + 1]) & 0xFFFFE000u);
                            const float h2 = __uint_as_float(__float_as_uint(x[4 * j + 2]) & 0xFFFFE000u);
                            const float h3 = __uint_as_float(__float_as_uint(x[4 * j + 3]) & 0xFFFFE000u);
                            if (part == 0) o = make_float4(h0, h1, h2, h3);
                            else o = make_float4(x[4 * j + 0] - h0, x[4 * j + 1] - h1, x[4 * j + 2] - h2, x[4 * j + 3] - h3);
                            st_shared_v4(stage_tile + (uint32_t)lane * 128u + (uint32_t)((j ^ (lane & 7)) << 4), o);  // 128B swizzle
                        }
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> async-proxy reads
                        __syncwarp();
                        if (lane == 0) {
                            tma_store_2d(part == 0 ? &map_c_hi : &map_c_lo, stage_tile, col0, rbase);
                            tma_store_commit();
                        }
                    }
                }
                continue;
            }
            // Row-major outputs: each lane holds 32 consecutive columns of ITS row, which would make every store
            // instruction touch 32 different rows. Transpose each 32x32 block through this warp's padded shared-memory
            // tile so that a store instruction writes 128 contiguous bytes of one row; bias, ReLU and the hi/lo split are
            // applied after the transpose, where lane = column.
            float* stg = reinterpret_cast<float*>(smem_raw + (out_tiles - smem_u32(smem_raw)) + pw * 4096);  // [32][32], XOR-swizzled
            const int rbase = m0 + q * 32;
            const int rows_here = min(32, sh.m - rbase);
#pragma unroll
            for (int c = 0; c < CW / 32; c++) {
                const int col0 = n0 + nc0 + c * 32;
                if (col0 >= sh.n || rows_here <= 0) continue;  // warp-uniform
                __syncwarp();
#pragma unroll
                for (int i = 0; i < 32; i++) stg[lane * 32 + (i ^ lane)] = acc[c * 32 + i];
                __syncwarp();
                const int col = col0 + lane;
                const bool col_ok = col < sh.n;
                const float bias = (ep.bias && col_ok) ? __ldg(ep.bias + col) : 0.f;
                float* pc = cplain ? cplain + (size_t)rbase * ep.ldc + col : nullptr;
                int blk_b = 0, blk_s = 0;   // blocked gate array: batch row and step of row rbase
                if (ep.step_t > 0) { blk_b = rbase / ep.step_t; blk_s = rbase - blk_b * ep.step_t; }
                float* ph = (!H && ep.c_hi) ? static_cast<float*>(ep.c_hi) + (size_t)rbase * ep.ldc_split + col : nullptr;
                float* pl = (!H && ep.c_hi) ? static_cast<float*>(ep.c_lo) + (size_t)rbase * ep.ldc_split + col : nullptr;
                const float* pm = ep.mask ? ep.mask + (size_t)rbase * ep.ldmask + col : nullptr;
                uint32_t myword = 0;
#pragma unroll 1
                for (int rr0 = 0; rr0 < 32; rr0 += 8) {  // 8 rows per batch: 8 shared-memory reads in flight per lane
                    float tv[8], mv[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        tv[u] = stg[(rr0 + u) * 32 + (lane ^ (rr0 + u))];
                        mv[u] = 1.f;
                        if (pm && col_ok && rr0 + u < rows_here) mv[u] = __ldg(pm + (size_t)u * ep.ldmask);
                    }
#pragma unroll
                    for (int u = 0; u < 8; u++) {
                        float t = tv[u] + bias;
                        if (ep.relu) t = fmaxf(t, 0.f);
                        t = mv[u] > 0.f ? t : 0.f;
                        if (ep.mask_bits_out) {
                            const uint32_t w32 = __ballot_sync(0xFFFFFFFFu, col_ok && t > 0.f);
                            if (lane == rr0 + u) myword = w32;
                        }
                        if (ep.step_t > 0) {
                            if (col_ok && rr0 + u < rows_here) cplain[step_block_offset(blk_s, blk_b, col, ep.step_nblk)] = t;
                            if (++blk_s == ep.step_t) { blk_s = 0; blk_b++; }
                        } else if (col_ok && rr0 + u < rows_here) {
                            if (pc) pc[(size_t)u * ep.ldc] = t;
                            if (ph) {
                                const float h = __uint_as_float(__float_as_uint(t) & 0xFFFFE000u);
                                ph[(size_t)u * ep.ldc_split] = h;
                                pl[(size_t)u * ep.ldc_split] = t - h;
                            }
                        }
                    }
                    if (pc) pc += (size_t)8 * ep.ldc;
                    if (ph) { ph += (size_t)8 * ep.ldc_split; pl += (size_t)8 * ep.ldc_split; }
                    if (pm) pm += (size_t)8 * ep.ldmask;
                }
                if (ep.mask_bits_out && lane < rows_here)
                    ep.mask_bits_out[(size_t)(rbase + lane) * ep.mask_ldw + (col0 >> 5)] = myword;
            }
            }   // !W16
        }
    }

    if constexpr (H) {
        if (warp >= Cfg::kCtrlWarps && ep.out_hs) {  // max |output| over everything this warp produced: one atomic per warp
            const uint32_t wm = __reduce_max_sync(0xFFFFFFFFu, __float_as_uint(tmax_kernel));
            if (lane == 0 && wm) atomicMax(reinterpret_cast<unsigned int*>(&ep.out_hs->amax), wm);
        }
    }
    if (warp >= Cfg::kCtrlWarps && lane == 0) tma_store_wait_all();  // staged output tiles must outlive their bulk stores
    tc_fence_before();
    if constexpr (PAIR) cluster_sync_all();  // the peer may still multicast into / arrive on this CTA's barriers
    else __syncthreads();
    if (warp == kAllocWarp) {
        tc_fence_after();
        if constexpr (PAIR)
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::kTmemCols) : "memory");
        else
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::kTmemCols) : "memory");
    }
}

// Length-aware pre-passes (kLength, fi_learner_config.variable_length): x is a gathered batch of len_t-record trajectories
// and row r is record r % len_t of its trajectory; it is a valid step when that index is below the length in word 183 of the
// trajectory's record 0 (rows < 2^32, checked by the launchers). Padding rows are never read: they count as zero rows.
__device__ __forceinline__ bool row_in_length(const float* x, int ld_in, size_t r, int len_t) {
    const uint32_t rr = (uint32_t)r, s = rr % (uint32_t)len_t;
    return (int)s < traj_length(__ldg(reinterpret_cast<const uint32_t*>(x + (size_t)(rr - s) * ld_in) + kWLength), len_t);
}

// fp32 -> (hi, lo) split of a [rows, cols] matrix (row stride ld_in) into two dense [rows, ld_out] arrays;
// columns [cols, ld_out) are zero-filled. Algorithmic traffic 12 B per element.
template <bool kLength>
__global__ void split_tf32_kernel(const float* __restrict__ x, int ld_in, size_t rows, int cols, int ld_out,
                                  float* __restrict__ hi, float* __restrict__ lo, int len_t) {
    const size_t total = rows * (size_t)ld_out;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / ld_out;
        const int c = (int)(i - r * ld_out);
        float v = 0.f;
        bool in = c < cols;
        if constexpr (kLength) in = in && row_in_length(x, ld_in, r, len_t);
        if (in) v = __ldg(x + r * ld_in + c);
        const float h = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
        hi[i] = h;
        lo[i] = v - h;
    }
}

// FI_COOP=0: the fused max|x| + split pre-passes (one cooperative launch each) as separate launches (A/B measurements)
static bool coop_prepass() {
    static const bool on = [] { const char* e = getenv("FI_COOP"); return !(e && e[0] == '0'); }();
    return on;
}

static int check_len_t(int len_t, int ld_in, size_t rows, const char* what) {
    if (len_t < 0 || (len_t > 0 && (ld_in < kWLength + 1 || rows > 0xFFFFFFFFull)))
        return set_error(FI_ERR_ARG, "%s: a length-aware split needs record rows (ld_in > %d) and rows < 2^32", what, kWLength);
    return FI_OK;
}

int launch_split_tf32(const float* x, int ld_in, size_t rows, int cols, int ld_out, float* hi, float* lo, cudaStream_t st,
                      int len_t) {
    if (rows == 0 || ld_out == 0) return FI_OK;
    FI_TRY(check_len_t(len_t, ld_in, rows, "split_tf32"));
    const size_t total = rows * (size_t)ld_out;
    size_t blocks = (total + 255) / 256;
    if (blocks > (size_t)kNumSMs * 16) blocks = (size_t)kNumSMs * 16;
    // the length-aware split also reads each row's length word (4 B per row)
    LaunchScope ls(len_t ? "split_tf32_kernel_length" : "split_tf32_kernel", st,
                   4.0 * (double)rows * cols + 8.0 * (double)total + (len_t ? 4.0 * (double)rows : 0.0), kWorkBytes);
    (len_t ? split_tf32_kernel<true> : split_tf32_kernel<false>)<<<(unsigned)blocks, 256, 0, st>>>(x, ld_in, rows, cols, ld_out, hi,
                                                                                                 lo, len_t);
    return ls.done();
}

// The plain-fp32 paths' length-aware copy (the actor-critic's simt trunk, the FarmerLstm projection and W_ih gradient off the
// 3xFP16 path): out [rows, kObsLd] = the observations (words 0..161) of a gathered batch of t-record trajectories; rows past
// their trajectory's length, and columns 162..163, are zero. One warp per row: the length word is one broadcast load per row.
__global__ void obs_length_kernel(const float* __restrict__ batch, int rows, int t, float* __restrict__ out) {
    const int warp = (int)((blockIdx.x * blockDim.x + threadIdx.x) >> 5), nwarps = (int)((gridDim.x * blockDim.x) >> 5);
    const int lane = threadIdx.x & 31;
    for (int r = warp; r < rows; r += nwarps) {
        const int s = r % t;
        const float* rec = batch + (size_t)r * kRecWords;
        const bool in = s < traj_length(__ldg(reinterpret_cast<const uint32_t*>(rec - (size_t)s * kRecWords) + kWLength), t);
        for (int c = lane; c < kObsLd; c += 32) out[(size_t)r * kObsLd + c] = in && c < kZDim ? __ldg(rec + c) : 0.f;
    }
}

int launch_obs_length(const float* batch, int rows, int t, float* out, cudaStream_t st) {
    int blocks = (rows + 7) / 8;
    if (blocks > kNumSMs * 16) blocks = kNumSMs * 16;
    // algorithmic traffic per row: 162 words in, 164 out, the length word
    LaunchScope ls("obs_length_kernel", st, (4.0 * (kZDim + kObsLd) + 4.0) * rows, kWorkBytes);
    obs_length_kernel<<<blocks, 256, 0, st>>>(batch, rows, t, out);
    return ls.done();
}

// ---- 3xFP16 pre-passes ---------------------------------------------------------------------------------------
// max |x| over a [rows, cols] matrix (row stride ld_in) into hs->amax. Non-negative floats order like their bit patterns.
__global__ void amax_kernel(const float* __restrict__ x, int ld_in, size_t rows, int cols, HScale* hs) {
    float m = 0.f;
    if (rows == 1) {  // flat vector (the parameter arena)
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (size_t)cols; i += (size_t)gridDim.x * blockDim.x)
            m = fmaxf(m, fabsf(__ldg(x + i)));
    } else {          // one warp per row, lanes along the row: no per-element index arithmetic
        const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
        const int lane = threadIdx.x & 31;
        for (size_t r = warp; r < rows; r += nwarps) {
            const float* xr = x + r * ld_in;
            for (int c = lane; c < cols; c += 32) m = fmaxf(m, fabsf(__ldg(xr + c)));
        }
    }
    const uint32_t wm = __reduce_max_sync(0xFFFFFFFFu, __float_as_uint(m));
    if ((threadIdx.x & 31) == 0 && wm) atomicMax(reinterpret_cast<unsigned int*>(&hs->amax), wm);
}

int launch_amax(const float* x, int ld_in, size_t rows, int cols, HScale* hs, cudaStream_t st) {
    if (rows == 0 || cols == 0) return FI_OK;
    const size_t total = rows * (size_t)cols;
    size_t blocks = rows == 1 ? (total + 1023) / 1024 : (rows + 7) / 8;
    if (blocks > (size_t)kNumSMs * 8) blocks = (size_t)kNumSMs * 8;
    LaunchScope ls("amax_kernel", st, 4.0 * (double)total, kWorkBytes);
    amax_kernel<<<(unsigned)blocks, 256, 0, st>>>(x, ld_in, rows, cols, hs);
    return ls.done();
}

// fp32 -> fp16 (hi, lo') pair of x * scale, scale = hscale_from_bound(hs->amax): dense [rows, ld_out] arrays (ld_out even),
// columns [cols, ld_out) zero-filled. Two elements per thread (one 4-byte store per array). Traffic 4 + 4 B per element.
__global__ void split_h_kernel(const float* __restrict__ x, int ld_in, size_t rows, int cols, int ld_out, __half2* __restrict__ hi,
                               __half2* __restrict__ lo, HScale* hs, int write_scale) {
    pdl_wait();
    const float scale = hscale_from_bound(hs->amax);
    if (write_scale && blockIdx.x == 0 && threadIdx.x == 0) {
        hs->scale = scale;
        hs->inv = 1.f / scale;
        hs->bound = hs->amax;
    }
    const int ldp = ld_out >> 1;
    auto emit = [&](size_t o, float v0, float v1) {
        v0 *= scale;
        v1 *= scale;
        const __half2 h = __floats2half2_rn(v0, v1);
        const float2 hf = __half22float2(h);
        hi[o] = h;
        lo[o] = __floats2half2_rn(fmaf(v0, 2048.f, -2048.f * hf.x), fmaf(v1, 2048.f, -2048.f * hf.y));
    };
    if (rows == 1 || ldp < 32) {
        // one long row, or rows narrower than a warp (the 17-wide head gradient: a warp per row left half the lanes idle and
        // one 64-byte store per warp and trip): one thread per output pair, consecutive threads consecutive pairs
        const size_t total = rows * (size_t)ldp;
        for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
            const size_t r = i / (size_t)ldp;
            const int c = (int)(i - r * (size_t)ldp) * 2;
            const float* xr = x + r * ld_in;
            emit(i, c < cols ? __ldg(xr + c) : 0.f, c + 1 < cols ? __ldg(xr + c + 1) : 0.f);
        }
        return;
    }
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    for (size_t r = warp; r < rows; r += nwarps) {
        const float* xr = x + r * ld_in;
        for (int p = lane; p < ldp; p += 32) {
            const int c = 2 * p;
            emit(r * ldp + p, c < cols ? __ldg(xr + c) : 0.f, c + 1 < cols ? __ldg(xr + c + 1) : 0.f);
        }
    }
}

int launch_split_h(const float* x, int ld_in, size_t rows, int cols, int ld_out, void* hi, void* lo, HScale* hs, int write_scale,
                   cudaStream_t st) {
    if (rows == 0 || ld_out == 0) return FI_OK;
    if (ld_out & 1) return set_error(FI_ERR_ARG, "split_h: ld_out must be even");
    const size_t total = rows * (size_t)(ld_out / 2);
    size_t blocks = (rows == 1 || ld_out / 2 < 32) ? (total + 255) / 256 : (rows + 7) / 8;
    if (blocks > (size_t)kNumSMs * 16) blocks = (size_t)kNumSMs * 16;
    LaunchScope ls("split_h_kernel", st, 4.0 * (double)rows * cols + 4.0 * (double)rows * ld_out, kWorkBytes);
    launch_pdl(split_h_kernel, dim3((unsigned)blocks), dim3(256), 0, st, x, ld_in, rows, cols, ld_out, static_cast<__half2*>(hi),
               static_cast<__half2*>(lo), hs, write_scale);
    return ls.done();
}

// max |x| AND the fp16 (hi, lo') split of a [rows, cols] matrix in ONE cooperative launch: every warp takes the maximum over its
// rows, the grid synchronises, every warp splits the same rows again (they come out of L2 the second time). Replaces an amax
// launch + a split launch on the step's critical path (observations: 25 + 30 us as two launches that read 66 MB from HBM twice;
// the head gradient: 13 + 14 us). hs->amax must be zero on entry. kLength: padding rows (row_in_length) are zero rows.
template <bool kLength>
__global__ void __launch_bounds__(256)
amax_split_h_kernel(const float* __restrict__ x, int ld_in, size_t rows, int cols, int ld_out, __half2* __restrict__ hi,
                    __half2* __restrict__ lo, HScale* hs, int len_t) {
    const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((size_t)gridDim.x * blockDim.x) >> 5;
    const int lane = threadIdx.x & 31;
    // Four rows per warp and trip, 8-byte loads where the layout allows: one row at a time with scalar loads left the pass
    // latency-bound (2.5 TB/s on the observations: six dependent 4-byte loads per lane and row)
    const bool vec2 = (ld_in & 1) == 0 && (cols & 1) == 0 && (reinterpret_cast<uintptr_t>(x) & 7) == 0;
    constexpr int kRowsPerTrip = 4;
    float m = 0.f;
    bool ok[kRowsPerTrip];   // kLength: row r0 + j exists and is a valid step
    auto live = [&](size_t r0, int j) {
        if constexpr (kLength) return ok[j];
        else return r0 + j < rows;
    };
    auto set_live = [&](size_t r0) {
        if constexpr (kLength) {
#pragma unroll
            for (int j = 0; j < kRowsPerTrip; j++) ok[j] = r0 + j < rows && row_in_length(x, ld_in, r0 + j, len_t);
        }
    };
    for (size_t r0 = warp * kRowsPerTrip; r0 < rows; r0 += nwarps * kRowsPerTrip) {
        set_live(r0);
        if (vec2) {
            for (int c = 2 * lane; c < cols; c += 64) {
                float2 v[kRowsPerTrip];
#pragma unroll
                for (int j = 0; j < kRowsPerTrip; j++)
                    v[j] = live(r0, j) ? __ldg(reinterpret_cast<const float2*>(x + (r0 + j) * ld_in + c)) : make_float2(0.f, 0.f);
#pragma unroll
                for (int j = 0; j < kRowsPerTrip; j++) m = fmaxf(m, fmaxf(fabsf(v[j].x), fabsf(v[j].y)));
            }
        } else {
            for (int c = lane; c < cols; c += 32) {
                float v[kRowsPerTrip];
#pragma unroll
                for (int j = 0; j < kRowsPerTrip; j++) v[j] = live(r0, j) ? __ldg(x + (r0 + j) * ld_in + c) : 0.f;
#pragma unroll
                for (int j = 0; j < kRowsPerTrip; j++) m = fmaxf(m, fabsf(v[j]));
            }
        }
    }
    const uint32_t wm = __reduce_max_sync(0xFFFFFFFFu, __float_as_uint(m));
    if (lane == 0 && wm) atomicMax(reinterpret_cast<unsigned int*>(&hs->amax), wm);
    cooperative_groups::this_grid().sync();
    const float amax = *reinterpret_cast<volatile float*>(&hs->amax);
    const float scale = hscale_from_bound(amax);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        hs->scale = scale;
        hs->inv = 1.f / scale;
        hs->bound = amax;
    }
    const int ldp = ld_out >> 1;
    for (size_t r0 = warp * kRowsPerTrip; r0 < rows; r0 += nwarps * kRowsPerTrip) {
        set_live(r0);
        for (int p = lane; p < ldp; p += 32) {
            const int c = 2 * p;
            float2 v[kRowsPerTrip];
#pragma unroll
            for (int j = 0; j < kRowsPerTrip; j++) {
                v[j] = make_float2(0.f, 0.f);
                if (live(r0, j)) {
                    const float* xr = x + (r0 + j) * ld_in;
                    if (vec2) {
                        if (c < cols) v[j] = __ldg(reinterpret_cast<const float2*>(xr + c));
                    } else {
                        v[j] = make_float2(c < cols ? __ldg(xr + c) : 0.f, c + 1 < cols ? __ldg(xr + c + 1) : 0.f);
                    }
                }
            }
#pragma unroll
            for (int j = 0; j < kRowsPerTrip; j++) {
                if (r0 + j >= rows) break;
                const float v0 = v[j].x * scale, v1 = v[j].y * scale;
                const __half2 h = __floats2half2_rn(v0, v1);
                const float2 hf = __half22float2(h);
                hi[(r0 + j) * ldp + p] = h;
                lo[(r0 + j) * ldp + p] = __floats2half2_rn(fmaf(v0, 2048.f, -2048.f * hf.x), fmaf(v1, 2048.f, -2048.f * hf.y));
            }
        }
    }
}

int launch_amax_split_h(const float* x, int ld_in, size_t rows, int cols, int ld_out, void* hi, void* lo, HScale* hs, cudaStream_t st,
                        int len_t) {
    FI_TRY(check_len_t(len_t, ld_in, rows, "amax_split_h"));
    if (!coop_prepass() && !len_t) {   // FI_COOP=0: two ordinary launches
        FI_TRY(launch_amax(x, ld_in, rows, cols, hs, st));
        return launch_split_h(x, ld_in, rows, cols, ld_out, hi, lo, hs, 1, st);
    }
    if (rows == 0 || ld_out == 0) return FI_OK;
    if (ld_out & 1) return set_error(FI_ERR_ARG, "split_h: ld_out must be even");
    // every block must be resident for the grid barrier: as many blocks as fit (queried once per device), capped by the work
    static std::mutex mu;
    static int blocks_per_sm[2][64] = {};
    const void* kernel = len_t ? (const void*)amax_split_h_kernel<true> : (const void*)amax_split_h_kernel<false>;
    int dev = 0;
    cudaGetDevice(&dev);
    int bps;
    {
        std::lock_guard<std::mutex> g(mu);
        int& cached = blocks_per_sm[len_t ? 1 : 0][dev & 63];
        if (!cached) {
            int n = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, 256, 0) != cudaSuccess || n < 1) n = 1;
            cached = n > 4 ? 4 : n;
        }
        bps = cached;
    }
    size_t blocks = (rows + 31) / 32;   // 8 warps x 4 rows per trip
    if (blocks < 1) blocks = 1;
    if (blocks > (size_t)kNumSMs * bps) blocks = (size_t)kNumSMs * bps;
    __half2* hi2 = static_cast<__half2*>(hi);
    __half2* lo2 = static_cast<__half2*>(lo);
    void* args[] = {(void*)&x, (void*)&ld_in, (void*)&rows, (void*)&cols, (void*)&ld_out, (void*)&hi2, (void*)&lo2, (void*)&hs,
                    (void*)&len_t};
    // the length-aware pass also reads each row's length word, once per pass (8 B per row)
    LaunchScope ls(len_t ? "amax_split_h_kernel_length" : "amax_split_h_kernel", st,
                   8.0 * (double)rows * cols + 4.0 * (double)rows * ld_out + (len_t ? 8.0 * (double)rows : 0.0), kWorkBytes);
    const cudaError_t e = cudaLaunchCooperativeKernel(kernel, dim3((unsigned)blocks), dim3(256), args, 0, st);
    if (e != cudaSuccess) return set_error(FI_ERR_CUDA, "cooperative launch of amax_split_h_kernel failed: %s", cudaGetErrorString(e));
    return ls.done();
}

// The parameter arena's pre-pass in one cooperative launch: max |p| over the flat arena, grid barrier, then the fp16 split of
// the arena (same element offsets) AND of one weight matrix re-laid out to padded rows (dense1.w: 162 -> ld2 columns), both
// with the arena's scale. Replaces amax + two split launches. hs->amax must be zero on entry.
__global__ void __launch_bounds__(256)
amax_split_params_kernel(const float* __restrict__ p, int n, int ld_flat, __half2* __restrict__ hi, __half2* __restrict__ lo,
                         const float* __restrict__ w, int w_rows, int w_cols, int ld2, __half2* __restrict__ hi2, __half2* __restrict__ lo2,
                         HScale* hs) {
    const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x, nthreads = (size_t)gridDim.x * blockDim.x;
    float m = 0.f;
    for (size_t i = tid; i < (size_t)n; i += nthreads) m = fmaxf(m, fabsf(__ldg(p + i)));
    const uint32_t wm = __reduce_max_sync(0xFFFFFFFFu, __float_as_uint(m));
    if ((threadIdx.x & 31) == 0 && wm) atomicMax(reinterpret_cast<unsigned int*>(&hs->amax), wm);
    cooperative_groups::this_grid().sync();
    const float amax = *reinterpret_cast<volatile float*>(&hs->amax);
    const float scale = hscale_from_bound(amax);
    if (tid == 0) {
        hs->scale = scale;
        hs->inv = 1.f / scale;
        hs->bound = amax;
    }
    auto emit = [&](__half2* oh, __half2* ol, size_t o, float v0, float v1) {
        v0 *= scale;
        v1 *= scale;
        const __half2 h = __floats2half2_rn(v0, v1);
        const float2 hf = __half22float2(h);
        oh[o] = h;
        ol[o] = __floats2half2_rn(fmaf(v0, 2048.f, -2048.f * hf.x), fmaf(v1, 2048.f, -2048.f * hf.y));
    };
    const size_t flat_pairs = (size_t)(ld_flat >> 1), w_pairs = (size_t)w_rows * (ld2 >> 1);
    for (size_t i = tid; i < flat_pairs + w_pairs; i += nthreads) {
        if (i < flat_pairs) {
            const int c = (int)i * 2;
            emit(hi, lo, i, c < n ? __ldg(p + c) : 0.f, c + 1 < n ? __ldg(p + c + 1) : 0.f);
        } else {
            const size_t j = i - flat_pairs;
            const int r = (int)(j / (ld2 >> 1)), c = (int)(j % (ld2 >> 1)) * 2;
            const float* wr = w + (size_t)r * w_cols;
            emit(hi2, lo2, j, c < w_cols ? __ldg(wr + c) : 0.f, c + 1 < w_cols ? __ldg(wr + c + 1) : 0.f);
        }
    }
}

int launch_amax_split_params(const float* p, int n, int ld_flat, void* hi, void* lo, const float* w, int w_rows, int w_cols, int ld2,
                             void* hi2, void* lo2, HScale* hs, cudaStream_t st) {
    if (!coop_prepass()) {   // FI_COOP=0: three ordinary launches
        FI_TRY(launch_amax(p, n, 1, n, hs, st));
        FI_TRY(launch_split_h(p, n, 1, n, ld_flat, hi, lo, hs, 1, st));
        return launch_split_h(w, w_cols, w_rows, w_cols, ld2, hi2, lo2, hs, 0, st);
    }
    if ((ld_flat & 1) || (ld2 & 1)) return set_error(FI_ERR_ARG, "split_h: row strides must be even");
    __half2 *a = static_cast<__half2*>(hi), *b = static_cast<__half2*>(lo), *c = static_cast<__half2*>(hi2), *d = static_cast<__half2*>(lo2);
    void* args[] = {(void*)&p, (void*)&n, (void*)&ld_flat, (void*)&a, (void*)&b, (void*)&w, (void*)&w_rows, (void*)&w_cols, (void*)&ld2,
                    (void*)&c, (void*)&d, (void*)&hs};
    LaunchScope ls("amax_split_params_kernel", st, 8.0 * n + 4.0 * ld_flat + 4.0 * w_rows * (w_cols + ld2), kWorkBytes);
    const cudaError_t e = cudaLaunchCooperativeKernel((const void*)amax_split_params_kernel, dim3(kNumSMs), dim3(256), args, 0, st);
    if (e != cudaSuccess) return set_error(FI_ERR_CUDA, "cooperative launch of amax_split_params_kernel failed: %s", cudaGetErrorString(e));
    return ls.done();
}

// ---- host side ------------------------------------------------------------------------------------------------
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                   const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        cudaGetLastError();
    });
    return fn;
}

// 2-D fp32 tensor map: inner (contiguous) extent `inner`, outer extent `outer`, row stride ld elements;
// box = 32 inner elements (128 B, the swizzle span) x box_outer rows. Out-of-bounds elements read as zero.
// Encoding a tensor map is a driver call (a few microseconds); a learner step needs ~100 of them and always the same
// ones (fixed buffers, fixed shapes), so they are cached by their defining tuple. With 8 ranks sharing 16 host cores the
// step was host-enqueue bound before this cache (profiles/r1_bench_8gpu.json: 0.96 ms of gaps per 5.3 ms step).
struct MapKey {
    const void* base;
    uint64_t inner, outer, ld;
    uint32_t box_outer, mn_major;  // mn_major: bit 0 = MN-major operand, bit 1 = fp16 elements
    bool operator==(const MapKey& o) const {
        return base == o.base && inner == o.inner && outer == o.outer && ld == o.ld && box_outer == o.box_outer && mn_major == o.mn_major;
    }
};
struct MapKeyHash {
    size_t operator()(const MapKey& k) const {
        uint64_t h = reinterpret_cast<uintptr_t>(k.base) * 0x9E3779B97F4A7C15ull;
        h ^= (k.inner + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2));
        h ^= (k.outer * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2));
        h ^= (k.ld * 0x165667B19E3779F9ull) ^ ((uint64_t)k.box_outer << 33) ^ k.mn_major;
        return (size_t)h;
    }
};

static int make_map_uncached(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t ld, uint32_t box_outer,
                             bool mn_major, bool half);

static int make_map(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t ld, uint32_t box_outer,
                    bool mn_major, bool half = false) {
    static std::mutex mu;
    static std::unordered_map<MapKey, CUtensorMap, MapKeyHash> cache;
    const MapKey key{base, inner, outer, ld, box_outer, (mn_major ? 1u : 0u) | (half ? 2u : 0u)};
    {
        std::lock_guard<std::mutex> g(mu);
        auto it = cache.find(key);
        if (it != cache.end()) {
            *map = it->second;
            return FI_OK;
        }
    }
    FI_TRY(make_map_uncached(map, base, inner, outer, ld, box_outer, mn_major, half));
    std::lock_guard<std::mutex> g(mu);
    if (cache.size() > 4096) cache.clear();  // operator-level callers with ever-changing buffers: bound the table
    cache.emplace(key, *map);
    return FI_OK;
}

static int make_map_uncached(CUtensorMap* map, const void* base, uint64_t inner, uint64_t outer, uint64_t ld, uint32_t box_outer,
                             bool mn_major, bool half) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return set_error(FI_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    const uint64_t esz = half ? 2 : 4;
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (ld * esz) % 16)
        return set_error(FI_ERR_ARG, "tcgen05 GEMM: operand base / row stride must be 16-byte aligned (ld=%llu)", (unsigned long long)ld);
    cuuint64_t dims[2] = {inner, outer};
    cuuint64_t strides[1] = {ld * esz};
    cuuint32_t box[2] = {(cuuint32_t)(128 / esz), box_outer};   // 128 bytes of the contiguous dimension = the swizzle span
    cuuint32_t estr[2] = {1, 1};
    // MN-major tf32 operands only exist with 32-byte swizzle atoms; fp16 uses the plain 128B swizzle for both majors
    CUresult r = fn(map, half ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides,
                    box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    (mn_major && !half) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(FI_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return FI_OK;
}

// A [rows b][steps t][cols] array (row (b, s) at (b * t + s) * cols) as the 3-D tensor (cols, t, b) with boxes of
// (box_cols, 1, box_rows): one box = the columns [c0, c0 + box_cols) of step s for box_rows consecutive batch rows -- what one CTA
// of the recurrent kernels (lstm_tc.cu) loads or stores per step. swizzle_bytes = box_cols * elem_bytes: 32 or 64.
int make_step_tensor_map(CUtensorMap* map, const void* base, int elem_bytes, uint64_t cols, uint64_t t, uint64_t rows, uint32_t box_cols,
                         uint32_t box_rows, int swizzle_bytes) {
    EncodeTiledFn fn = encode_fn();
    if (!fn) return set_error(FI_ERR_CUDA, "cuTensorMapEncodeTiled is not available from this driver");
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (cols * elem_bytes) % 16 || (int)box_cols * elem_bytes != swizzle_bytes)
        return set_error(FI_ERR_ARG, "step tensor map: base / row stride must be 16-byte aligned and the box row must span the swizzle");
    cuuint64_t dims[3] = {cols, t, rows};
    cuuint64_t strides[2] = {cols * (uint64_t)elem_bytes, t * cols * (uint64_t)elem_bytes};
    cuuint32_t box[3] = {box_cols, 1, box_rows};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = fn(map, elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims,
                    strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    swizzle_bytes == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error(FI_ERR_CUDA, "cuTensorMapEncodeTiled (3-D) failed with CUresult %d", (int)r);
    return FI_OK;
}

// FI_TC_TRACE="<trans>,<min n>,<min k>[,<max k>]": launches of that operand-major combination with n >= min n and min k <= k <= max k log their
// pipeline events into a device buffer (each matching launch starts a fresh log); fi_debug_tc_trace copies it out.
static unsigned long long* g_tc_trace = nullptr;
static unsigned long long* tc_trace_buffer(int trans, int /*m*/, int n, int k) {
    struct Filter { int on, trans, n, k, kmax; };
    static const Filter f = [] {
        const char* e = getenv("FI_TC_TRACE");
        Filter r{0, 0, 0, 0, 1 << 30};
        if (e) r.on = sscanf(e, "%d,%d,%d,%d", &r.trans, &r.n, &r.k, &r.kmax) >= 1;
        return r;
    }();
    if (!f.on || !trace_hooks_built("FI_TC_TRACE") || trans != f.trans || n < f.n || k < f.k || k > f.kmax) return nullptr;
    const size_t bytes = (size_t)kTraceCtas * kTraceRoles * kTraceCap * sizeof(unsigned long long);
    if (!g_tc_trace && cudaMalloc((void**)&g_tc_trace, bytes) != cudaSuccess) return nullptr;
    cudaMemset(g_tc_trace, 0, bytes);   // legacy-stream memset: diagnostics only
    return g_tc_trace;
}

static int pick_bn(int n, bool half = false) { return n > 64 ? 128 : ((n > 32 || half) ? 64 : 32); }

// CTA-pair mode (cta_group::2, 256 x 128 tiles: each CTA loads its 128 rows of A and HALF of the B tile, 48 KB per
// k-block instead of 64). Every big product of the learner step is bound by the L2 -> shared-memory fill rate (the TMA
// loads of 148 CTAs draw 10-12.5 TB/s; profiles/r2_gemm_trace.md), so a quarter less operand traffic is a quarter less
// time once nothing else is in the way. Round 1 measured pairs slower and kept them off in the fp16 format: their
// promotion warps released each chunk with a cluster-scope release (a full memory barrier, 2000-3500 clocks per chunk).
// With a CTA-scope release, pairs win. FI_TC_PAIR=0 never, =1 (default) wherever the tile shape allows, =2 the same.
static int pair_policy() {
    static const int policy = [] {
        const char* e = getenv("FI_TC_PAIR");
        return e ? atoi(e) : 1;
    }();
    return policy;
}
static bool use_pair(int trans, int m, int n, bool half) {
    const int policy = pair_policy();
    if (policy == 0 || pick_bn(n, half) != 128 || m < 2 * kTcBM) return false;
    return half || trans == 2 || policy >= 2;   // 3xTF32: the split-K wgrad products only, as measured in round 1
}

static int tc_splits(int trans, int m, int n, int k, bool pair, bool half = false) {
    if (trans != 2) return 1;
    const int bn = pick_bn(n, half);
    const int tile_m = pair ? 2 * kTcBM : kTcBM, units = pair ? kNumSMs / 2 : kNumSMs;
    const int tiles = ((m + tile_m - 1) / tile_m) * ((n + bn - 1) / bn);
    const int bk = half ? kTcBKh : kTcBK;
    const int num_kb = (k + bk - 1) / bk;
    int s = units / tiles;               // all CTAs of one wave; CTAs of the same split share operand rows in L2
    if (s > num_kb / 4) s = num_kb / 4;  // at least 4 k-blocks per split
    return s < 1 ? 1 : s;
}

size_t gemm_tc_split_workspace_bytes(int trans, int m, int n, int k) {
    int s = 1;                           // either CTA mode and either operand format may be chosen at launch time
    for (int pair = 0; pair < 2; pair++)
        for (int half = 0; half < 2; half++) {
            const int v = tc_splits(trans, m, n, k, pair != 0, half != 0);
            if (v > s) s = v;
        }
    return s > 1 ? (size_t)s * m * n * sizeof(float) : 0;
}

template <int BN, bool A_MN, bool B_MN, bool PAIR, bool H, bool W16 = false>
static int launch_variant(const CUtensorMap* maps, const TcShape& sh, const TcEpilogue& ep, int grid, cudaStream_t st) {
    using Cfg = TcCfg<BN, PAIR, W16>;
    static std::atomic<uint64_t> attr_devices{0};
    FI_TRY(ensure_dynamic_smem(attr_devices, (const void*)gemm_tc_kernel<BN, A_MN, B_MN, PAIR, H, W16>, Cfg::kSmemBytes));
    // profiling label: forward-like (NT), dgrad-like (NN), wgrad-like (TN, split-K)
    // (the odd-shaped products of a learner step -- layer 1's short K, the 17-wide head -- are timed under their own names)
    const bool narrow = sh.n < 64, short_k = !A_MN && sh.k < 256;
    const char* label = H ? (!B_MN ? (narrow ? "gemm_tc_kernel<f16x3,NT,head>" : short_k ? "gemm_tc_kernel<f16x3,NT,k162>" : "gemm_tc_kernel<f16x3,NT>")
                                   : (!A_MN ? (short_k ? "gemm_tc_kernel<f16x3,NN,head>" : "gemm_tc_kernel<f16x3,NN>")
                                            : (narrow ? "gemm_tc_kernel<f16x3,TN,head>" : sh.n < 256 ? "gemm_tc_kernel<f16x3,TN,n162>" : "gemm_tc_kernel<f16x3,TN>")))
                          : (!B_MN ? "gemm_tc_kernel<NT>" : (!A_MN ? "gemm_tc_kernel<NN>" : "gemm_tc_kernel<TN>"));
    LaunchScope ls(label, st, 2.0 * (double)sh.m * sh.n * sh.k, kWorkFlops);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(Cfg::kThreads);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    int na = 0;
    if constexpr (PAIR) {
        attr[na].id = cudaLaunchAttributeClusterDimension;  // the two CTAs of a cluster land on one SM pair
        attr[na].val.clusterDim.x = 2;
        attr[na].val.clusterDim.y = 1;
        attr[na].val.clusterDim.z = 1;
        na++;
    }
    // FI_PDL=0: plain stream serialisation (the kernel's griddepcontrol instructions are then no-ops)
    static const bool pdl = [] { const char* e = getenv("FI_PDL"); return !(e && e[0] == '0'); }();
    if (pdl) {
        attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[na].val.programmaticStreamSerializationAllowed = 1;
        na++;
    }
    cfg.attrs = attr;
    cfg.numAttrs = (unsigned)na;
    const cudaError_t le =
        cudaLaunchKernelEx(&cfg, gemm_tc_kernel<BN, A_MN, B_MN, PAIR, H, W16>, maps[0], maps[1], maps[2], maps[3], maps[4], maps[5], sh, ep);
    if (le != cudaSuccess) return set_error(FI_ERR_CUDA, "launch of %s failed: %s", label, cudaGetErrorString(le));
    return ls.done();
}

// C = op(A) op(B) with pre-split operands. trans as in launch_gemm: 0 "NT" A[m,k] B[n,k]; 1 "NN" A[m,k] B[k,n];
// 2 "TN" A[k,m] B[k,n] (split-K through `workspace`, reduced into out.c; no epilogue ops).
int launch_gemm_tc_split(int trans, int m, int n, int k, SplitMat a, SplitMat b, TcOut out, const float* bias, int relu,
                         const float* mask, int ldmask, void* workspace, size_t workspace_bytes, cudaStream_t st) {
    if (m <= 0 || n <= 0 || k <= 0) return FI_OK;
    if (trans < 0 || trans > 2) return set_error(FI_ERR_ARG, "gemm: trans must be 0, 1 or 2");
    if (!a.hi || !a.lo || !b.hi || !b.lo || (!out.c && !out.c_hi)) return set_error(FI_ERR_ARG, "tcgen05 GEMM: null operand");
    const bool a_mn = trans == 2, b_mn = trans != 0;
    const bool half = a.hs != nullptr;
    if (half != (b.hs != nullptr)) return set_error(FI_ERR_ARG, "tcgen05 GEMM: operands are in different split formats");
    const int bn = pick_bn(n, half), bk = half ? kTcBKh : kTcBK;
    const bool pair = use_pair(trans, m, n, half);
    TcShape sh;
    sh.m = m; sh.n = n; sh.k = k;
    sh.num_m_blocks = pair ? (m + 2 * kTcBM - 1) / (2 * kTcBM) : (m + kTcBM - 1) / kTcBM;
    sh.num_n_blocks = (n + bn - 1) / bn;
    sh.num_kb = (k + bk - 1) / bk;
    sh.num_splits = tc_splits(trans, m, n, k, pair, half);
    static const int dbg_flags = [] { const char* e = getenv("FI_TC_DBG"); return e ? atoi(e) : 0; }();
    sh.dbg = dbg_flags;
    sh.trace = tc_trace_buffer(trans, m, n, k);
    TcEpilogue ep;
    ep.c = out.c; ep.ldc = out.ldc; ep.c_hi = out.c_hi; ep.c_lo = out.c_lo; ep.ldc_split = out.ld_split;
    ep.bias = bias; ep.relu = relu; ep.mask = mask; ep.ldmask = ldmask; ep.transpose_out = out.transpose; ep.split_stride = 0;
    ep.mask_bits = out.mask_bits_in; ep.mask_bits_out = out.mask_bits_out; ep.mask_ldw = out.mask_ldw;
    ep.colsum_out = out.colsum_out;
    ep.step_t = out.step_t; ep.step_nblk = out.step_nblk;
    static const bool direct_on = [] { const char* e = getenv("FI_TC_DIRECT"); return !(e && e[0] == '0'); }();
    ep.plain_direct = direct_on && out.c && !out.c_hi && !out.transpose && !relu && !mask && !out.mask_bits_in && !out.mask_bits_out &&
                      !out.colsum_out && out.step_t == 0 && n % 8 == 0 && out.ldc % 8 == 0 && (reinterpret_cast<uintptr_t>(out.c) & 31) == 0;
    if (out.step_t > 0 && (out.c_hi || out.transpose || !out.c || relu || mask || out.mask_bits_in || out.mask_bits_out || n != 512 || m % out.step_t))
        return set_error(FI_ERR_ARG, "tcgen05 GEMM: the blocked gate-array output is a plain fp32 [b * t + s, 512] product");
    ep.a_hs = a.hs; ep.b_hs = b.hs; ep.bias_hs = bias ? out.bias_hs : nullptr; ep.out_hs = out.c_hi ? out.out_hs : nullptr;
    if (half && out.c_hi && (!out.out_hs || (bias && !out.bias_hs) || bn != 128))
        return set_error(FI_ERR_ARG, "tcgen05 GEMM (fp16 format): a split output needs n > 64, its HScale and a bound for the bias");
    if (ep.colsum_out && (bias || relu)) return set_error(FI_ERR_ARG, "tcgen05 GEMM: fused column sums exclude bias/ReLU");
    if (ep.mask_bits && (bias || relu || (n > 32 && (ep.mask_ldw % 4 || (reinterpret_cast<uintptr_t>(ep.mask_bits) & 15)))))
        return set_error(FI_ERR_ARG, "tcgen05 GEMM: a bit mask excludes bias/ReLU and needs 16-byte aligned rows");
    if (sh.num_splits > 1) {
        const size_t need = (size_t)sh.num_splits * m * n * sizeof(float);
        if (!workspace || workspace_bytes < need || bias || relu || mask || out.c_hi || !out.c || out.mask_bits_in || out.mask_bits_out ||
            out.step_t > 0) {
            sh.num_splits = 1;  // no room for partials (or an epilogue is requested): one split per tile
        } else {
            ep.c = static_cast<float*>(workspace);
            ep.split_stride = (size_t)m * n;
            if (out.transpose ? out.ldc != m : out.ldc != n)
                return set_error(FI_ERR_ARG, "tcgen05 GEMM: split-K needs a dense output (ldc=%d)", out.ldc);
        }
    }
    sh.kb_per_split = (sh.num_kb + sh.num_splits - 1) / sh.num_splits;
    sh.num_splits = (sh.num_kb + sh.kb_per_split - 1) / sh.kb_per_split;
    CUtensorMap maps[6];
    if (!a_mn) {
        FI_TRY(make_map(&maps[0], a.hi, (uint64_t)k, (uint64_t)m, (uint64_t)a.ld, kTcBM, false, half));
        FI_TRY(make_map(&maps[1], a.lo, (uint64_t)k, (uint64_t)m, (uint64_t)a.ld, kTcBM, false, half));
    } else {
        FI_TRY(make_map(&maps[0], a.hi, (uint64_t)m, (uint64_t)k, (uint64_t)a.ld, (uint32_t)bk, true, half));
        FI_TRY(make_map(&maps[1], a.lo, (uint64_t)m, (uint64_t)k, (uint64_t)a.ld, (uint32_t)bk, true, half));
    }
    if (!b_mn) {
        // K-major B: one box per CTA = its rows of the tile (pair mode: half of them)
        FI_TRY(make_map(&maps[2], b.hi, (uint64_t)k, (uint64_t)n, (uint64_t)b.ld, (uint32_t)(pair ? bn / 2 : bn), false, half));
        FI_TRY(make_map(&maps[3], b.lo, (uint64_t)k, (uint64_t)n, (uint64_t)b.ld, (uint32_t)(pair ? bn / 2 : bn), false, half));
    } else {
        FI_TRY(make_map(&maps[2], b.hi, (uint64_t)n, (uint64_t)k, (uint64_t)b.ld, (uint32_t)bk, true, half));
        FI_TRY(make_map(&maps[3], b.lo, (uint64_t)n, (uint64_t)k, (uint64_t)b.ld, (uint32_t)bk, true, half));
    }
    ep.tma_split = 0;
    if (ep.c_hi && !ep.transpose_out && out.ld_split % (half ? 8 : 4) == 0 &&
        ((reinterpret_cast<uintptr_t>(ep.c_hi) | reinterpret_cast<uintptr_t>(ep.c_lo)) & 15) == 0 && !ep.c && !ep.mask) {
        // one store box per promotion warp: 32 rows x 128 bytes (32 fp32 or 64 fp16 columns)
        FI_TRY(make_map(&maps[4], ep.c_hi, (uint64_t)n, (uint64_t)m, (uint64_t)out.ld_split, 32, false, half));
        FI_TRY(make_map(&maps[5], ep.c_lo, (uint64_t)n, (uint64_t)m, (uint64_t)out.ld_split, 32, false, half));
        ep.tma_split = 1;
        if (half && (n % 16 || out.ld_split % 16 || ((reinterpret_cast<uintptr_t>(ep.c_hi) | reinterpret_cast<uintptr_t>(ep.c_lo)) & 31)))
            return set_error(FI_ERR_ARG, "tcgen05 GEMM (fp16 format): a split output needs n and its row stride to be multiples of 16 "
                                         "and 32-byte aligned arrays (n=%d, ld=%d)", n, out.ld_split);
    } else {
        maps[4] = maps[0];
        maps[5] = maps[0];
        if (ep.colsum_out) return set_error(FI_ERR_ARG, "tcgen05 GEMM: fused column sums need the TMA split-output path");
        if (half && ep.c_hi) return set_error(FI_ERR_ARG, "tcgen05 GEMM (fp16 format): the split output must be alone, dense and 16-byte aligned");
    }
    const int total = sh.num_m_blocks * sh.num_n_blocks * sh.num_splits;
    const int units = pair ? kNumSMs / 2 : kNumSMs;
    const int grid = (total < units ? total : units) * (pair ? 2 : 1);
    int rc;
#define FI_TC(BNV, PAIRV, HV)                                                                                \
    (trans == 0 ? launch_variant<BNV, false, false, PAIRV, HV>(maps, sh, ep, grid, st)                       \
                : trans == 1 ? launch_variant<BNV, false, true, PAIRV, HV>(maps, sh, ep, grid, st)           \
                             : launch_variant<BNV, true, true, PAIRV, HV>(maps, sh, ep, grid, st))
    if (half) {
        // products whose every tile ends in the fp16 split epilogue (forward, dgrad) run with 16 promotion warps
        static const bool w16_on = [] { const char* e = getenv("FI_TC_W16"); return !e || atoi(e) != 0; }();
        const bool w16 = bn == 128 && w16_on && ep.tma_split && trans != 2;
        if (w16 && pair)
            rc = trans == 0 ? launch_variant<128, false, false, true, true, true>(maps, sh, ep, grid, st)
                            : launch_variant<128, false, true, true, true, true>(maps, sh, ep, grid, st);
        else if (bn == 128 && pair) rc = FI_TC(128, true, true);
        else if (w16)
            rc = trans == 0 ? launch_variant<128, false, false, false, true, true>(maps, sh, ep, grid, st)
                            : launch_variant<128, false, true, false, true, true>(maps, sh, ep, grid, st);
        else if (bn == 128) rc = FI_TC(128, false, true);
        else rc = FI_TC(64, false, true);
    } else if (bn == 128 && pair) rc = FI_TC(128, true, false);
    else if (bn == 128) rc = FI_TC(128, false, false);
    else if (bn == 64) rc = FI_TC(64, false, false);
    else rc = FI_TC(32, false, false);
#undef FI_TC
    FI_TRY(rc);
    if (out.deferred_splits) *out.deferred_splits = sh.num_splits;
    if (sh.num_splits > 1 && !out.deferred_splits) {
        const size_t total_out = (size_t)m * n;
        FI_TRY(launch_reduce_splits(static_cast<const float*>(workspace), sh.num_splits, total_out, total_out, out.c, st));
    }
    return FI_OK;
}

bool gemm_tc_available() { return encode_fn() != nullptr; }

int tc_trace_copy(void* host, size_t bytes) {
    const size_t have = (size_t)kTraceCtas * kTraceRoles * kTraceCap * sizeof(unsigned long long);
    if (!g_tc_trace) return set_error(FI_ERR_STATE, "no tcgen05 trace was recorded (set FI_TC_TRACE)");
    if (bytes < have) return set_error(FI_ERR_ARG, "trace buffer needs %zu bytes", have);
    FI_CUDA_OK(cudaDeviceSynchronize());
    FI_CUDA_OK(cudaMemcpy(host, g_tc_trace, have, cudaMemcpyDeviceToHost));
    return (int)(have / sizeof(unsigned long long));
}

// ---- plain fp32 entry (fi_op_gemm, FarmerLstm dense stack): split the operands into the workspace first --------
static size_t pad4(size_t x) { return (x + 3) & ~(size_t)3; }
static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

bool gemm_tc_supported(int trans, int m, int n, int k, const float*, int, const float*, int, const float*, int) {
    // tiny problems are launch-latency bound either way; the tensor-core path needs one full k-block
    return trans >= 0 && trans <= 2 && m >= 1 && n >= 1 && k >= 1 && encode_fn() != nullptr;
}

size_t gemm_tc_workspace_bytes(int trans, int m, int n, int k) {
    const size_t a_rows = trans == 2 ? k : m, a_cols = trans == 2 ? m : k;
    const size_t b_rows = trans == 0 ? n : k, b_cols = trans == 0 ? k : n;
    return 2 * align256(a_rows * pad4(a_cols) * 4) + 2 * align256(b_rows * pad4(b_cols) * 4) +
           align256(gemm_tc_split_workspace_bytes(trans, m, n, k));
}

int launch_gemm_tc(int trans, int m, int n, int k, const float* a, int lda, const float* b, int ldb, float* c, int ldc,
                   const float* bias, int relu, const float* mask, int ldmask, void* workspace, size_t workspace_bytes,
                   cudaStream_t st) {
    if (m <= 0 || n <= 0) return FI_OK;
    if (workspace_bytes < gemm_tc_workspace_bytes(trans, m, n, k) || !workspace)
        return set_error(FI_ERR_ARG, "tcgen05 GEMM: workspace too small (need %zu bytes)", gemm_tc_workspace_bytes(trans, m, n, k));
    const size_t a_rows = trans == 2 ? k : m, a_cols = trans == 2 ? m : k;
    const size_t b_rows = trans == 0 ? n : k, b_cols = trans == 0 ? k : n;
    const size_t a_ld = pad4(a_cols), b_ld = pad4(b_cols);
    char* ws = static_cast<char*>(workspace);
    float* a_hi = reinterpret_cast<float*>(ws); ws += align256(a_rows * a_ld * 4);
    float* a_lo = reinterpret_cast<float*>(ws); ws += align256(a_rows * a_ld * 4);
    float* b_hi = reinterpret_cast<float*>(ws); ws += align256(b_rows * b_ld * 4);
    float* b_lo = reinterpret_cast<float*>(ws); ws += align256(b_rows * b_ld * 4);
    FI_TRY(launch_split_tf32(a, lda, a_rows, (int)a_cols, (int)a_ld, a_hi, a_lo, st));
    FI_TRY(launch_split_tf32(b, ldb, b_rows, (int)b_cols, (int)b_ld, b_hi, b_lo, st));
    SplitMat sa{a_hi, a_lo, (int)a_ld}, sb{b_hi, b_lo, (int)b_ld};
    TcOut out{c, ldc, nullptr, nullptr, 0, 0, nullptr, nullptr, 0, nullptr};
    const size_t split_ws = gemm_tc_split_workspace_bytes(trans, m, n, k);
    if (trans == 2 && ldc != n) {  // split-K partials need a dense output
        return launch_gemm_tc_split(trans, m, n, k, sa, sb, out, bias, relu, mask, ldmask, nullptr, 0, st);
    }
    return launch_gemm_tc_split(trans, m, n, k, sa, sb, out, bias, relu, mask, ldmask, split_ws ? ws : nullptr, split_ws, st);
}

// ---- plain fp32 entry, 3xFP16 format: max |x| and split pre-passes for both operands, then the fp16 kernel --------
static size_t pad8(size_t x) { return (x + 7) & ~(size_t)7; }

size_t gemm_h_workspace_bytes(int trans, int m, int n, int k) {
    const size_t a_rows = trans == 2 ? k : m, a_cols = trans == 2 ? m : k;
    const size_t b_rows = trans == 0 ? n : k, b_cols = trans == 0 ? k : n;
    return 256 + 2 * align256(a_rows * pad8(a_cols) * 2) + 2 * align256(b_rows * pad8(b_cols) * 2) +
           align256(gemm_tc_split_workspace_bytes(trans, m, n, k));
}

int launch_gemm_h(int trans, int m, int n, int k, const float* a, int lda, const float* b, int ldb, float* c, int ldc,
                  const float* bias, int relu, const float* mask, int ldmask, void* workspace, size_t workspace_bytes,
                  cudaStream_t st) {
    if (m <= 0 || n <= 0) return FI_OK;
    if (workspace_bytes < gemm_h_workspace_bytes(trans, m, n, k) || !workspace)
        return set_error(FI_ERR_ARG, "tcgen05 GEMM (fp16 format): workspace too small (need %zu bytes)", gemm_h_workspace_bytes(trans, m, n, k));
    const size_t a_rows = trans == 2 ? k : m, a_cols = trans == 2 ? m : k;
    const size_t b_rows = trans == 0 ? n : k, b_cols = trans == 0 ? k : n;
    const size_t a_ld = pad8(a_cols), b_ld = pad8(b_cols);
    char* ws = static_cast<char*>(workspace);
    HScale* hs = reinterpret_cast<HScale*>(ws); ws += 256;
    void* a_hi = ws; ws += align256(a_rows * a_ld * 2);
    void* a_lo = ws; ws += align256(a_rows * a_ld * 2);
    void* b_hi = ws; ws += align256(b_rows * b_ld * 2);
    void* b_lo = ws; ws += align256(b_rows * b_ld * 2);
    FI_CUDA_OK(cudaMemsetAsync(hs, 0, 2 * sizeof(HScale), st));
    FI_TRY(launch_amax(a, lda, a_rows, (int)a_cols, hs + 0, st));
    FI_TRY(launch_amax(b, ldb, b_rows, (int)b_cols, hs + 1, st));
    FI_TRY(launch_split_h(a, lda, a_rows, (int)a_cols, (int)a_ld, a_hi, a_lo, hs + 0, 1, st));
    FI_TRY(launch_split_h(b, ldb, b_rows, (int)b_cols, (int)b_ld, b_hi, b_lo, hs + 1, 1, st));
    SplitMat sa{a_hi, a_lo, (int)a_ld, hs + 0}, sb{b_hi, b_lo, (int)b_ld, hs + 1};
    TcOut out{c, ldc, nullptr, nullptr, 0, 0, nullptr, nullptr, 0, nullptr};
    const size_t split_ws = gemm_tc_split_workspace_bytes(trans, m, n, k);
    if (trans == 2 && ldc != n) return launch_gemm_tc_split(trans, m, n, k, sa, sb, out, bias, relu, mask, ldmask, nullptr, 0, st);
    return launch_gemm_tc_split(trans, m, n, k, sa, sb, out, bias, relu, mask, ldmask, split_ws ? ws : nullptr, split_ws, st);
}

}  // namespace fi

// Diagnostics: the pipeline event log of the last traced tcgen05 GEMM launch (see FI_TC_TRACE above).
extern "C" int fi_debug_tc_trace(void* host, size_t bytes) { return fi::tc_trace_copy(host, bytes); }
