// V-trace targets, policy-gradient advantages and the fused policy/value/entropy loss head.
//
// NOT in the reference (SURVEY.md section 0): BASELINE.json's north_star adds it. Restates
// Espeholt et al. 2018 (arXiv:1802.01561) eq. (1) + Remark 2 (lambda) and section 4.2:
//   rho_s = min(rho_bar, e^{log_rho_s})      c_s = lambda * min(c_bar, e^{log_rho_s})
//   delta_s = rho_s (r_s + g_s V_{s+1} - V_s),            V_T = bootstrap
//   acc_s = delta_s + g_s c_s acc_{s+1}, acc_T = 0;       vs_s = V_s + acc_s
//   pg_adv_s = min(pg_rho_bar, e^{log_rho_s}) (r_s + g_s vs_{s+1} - V_s),  vs_T = bootstrap
// The reverse-time first-order recurrence is associative under (a1,b1)o(a2,b2) =
// (a1 a2, b1 + a1 b2), so each warp scans 32 time steps at once with shuffles and carries one
// scalar across 32-step chunks (last chunk first).
#include "fi_internal.cuh"

namespace fi {

// Reverse inclusive scan of acc_l = b_l + a_l * acc_{l+1} over the 32 lanes of a warp.
// On return (a,b) is the composition of lanes l..31, i.e. acc_l = b + a * carry_in.
__device__ __forceinline__ void warp_reverse_linear_scan(float& a, float& b, int lane) {
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const float a2 = __shfl_down_sync(0xffffffffu, a, off);
        const float b2 = __shfl_down_sync(0xffffffffu, b, off);
        if (lane + off < 32) {
            b = fmaf(a, b2, b);
            a *= a2;
        }
    }
}

// ---------------------------------------------------------------- standalone scan -------
// Arrays are trajectory-major [m, t] fp32, so 32 lanes x V consecutive time steps are one coalesced
// request per array. One warp owns one trajectory and walks it from the end in chunks of 32*V steps:
// each lane folds its V steps into one (a, b) pair, the warp combines the 32 pairs with shuffles, and
// the lane unfolds its V results; the next chunk's four loads are issued before the current chunk is
// computed (register double-buffering). Algorithmic traffic: 16 B in + 8 B out per transition
// (+4 B per trajectory for the bootstrap); HBM-bound.
// (Round-1 measurement: the first version staged whole trajectories through shared memory per CTA,
// load -> __syncthreads -> scan -> __syncthreads -> store, and was latency-bound at 29 % of the HBM
// roofline on 39 MB; see profiles/.)
template <int V>
struct ScanChunk {
    float lr[V], g[V], r[V], v[V];
};

template <int V>
__device__ __forceinline__ void scan_load(ScanChunk<V>& d, const float* __restrict__ log_rho,
                                          const float* __restrict__ discount, const float* __restrict__ reward,
                                          const float* __restrict__ value, size_t base, int s0, int t) {
    if constexpr (V == 4) {
        if (s0 + 3 < t) {
            const float4 a = __ldg(reinterpret_cast<const float4*>(log_rho + base + s0));
            const float4 b = __ldg(reinterpret_cast<const float4*>(discount + base + s0));
            const float4 c = __ldg(reinterpret_cast<const float4*>(reward + base + s0));
            const float4 e = __ldg(reinterpret_cast<const float4*>(value + base + s0));
            d.lr[0] = a.x; d.lr[1] = a.y; d.lr[2] = a.z; d.lr[3] = a.w;
            d.g[0] = b.x; d.g[1] = b.y; d.g[2] = b.z; d.g[3] = b.w;
            d.r[0] = c.x; d.r[1] = c.y; d.r[2] = c.z; d.r[3] = c.w;
            d.v[0] = e.x; d.v[1] = e.y; d.v[2] = e.z; d.v[3] = e.w;
            return;
        }
    }
#pragma unroll
    for (int e = 0; e < V; e++) {
        const bool ok = s0 + e < t;
        d.lr[e] = ok ? __ldg(log_rho + base + s0 + e) : 0.f;
        d.g[e] = ok ? __ldg(discount + base + s0 + e) : 0.f;
        d.r[e] = ok ? __ldg(reward + base + s0 + e) : 0.f;
        d.v[e] = ok ? __ldg(value + base + s0 + e) : 0.f;
    }
}

template <int V>
__global__ void __launch_bounds__(256)
vtrace_scan_kernel(int m, int t, const float* __restrict__ log_rho, const float* __restrict__ discount,
                   const float* __restrict__ reward, const float* __restrict__ value,
                   const float* __restrict__ bootstrap, float rho_bar, float c_bar, float pg_rho_bar, float lambda_,
                   float* __restrict__ vs_out, float* __restrict__ adv_out) {
    const int lane = threadIdx.x & 31;
    const int traj = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (traj >= m) return;
    constexpr int CH = 32 * V;
    const size_t base = (size_t)traj * t;
    const float boot = __ldg(bootstrap + traj);
    float carry = 0.f;            // acc at the first step of the chunk after this one
    float vs_next_chunk = boot;   // vs at that step
    float v_next_chunk = boot;    // V at that step
    ScanChunk<V> cur, nxt;
    int c0 = ((t - 1) / CH) * CH;
    scan_load<V>(cur, log_rho, discount, reward, value, base, c0 + lane * V, t);
    for (; c0 >= 0; c0 -= CH) {
        if (c0 >= CH) scan_load<V>(nxt, log_rho, discount, reward, value, base, c0 - CH + lane * V, t);
        const int s0 = c0 + lane * V;
        // V of the step after this lane's last one
        float v_after = __shfl_down_sync(0xffffffffu, cur.v[0], 1);
        if (lane == 31) v_after = v_next_chunk;
        float is[V], a[V], b[V];
#pragma unroll
        for (int e = 0; e < V; e++) {
            const int s = s0 + e;
            is[e] = expf(cur.lr[e]);
            float v_next = e + 1 < V ? cur.v[e + 1] : v_after;
            if (s >= t - 1) v_next = boot;
            const bool valid = s < t;
            a[e] = valid ? cur.g[e] * lambda_ * fminf(c_bar, is[e]) : 0.f;
            b[e] = valid ? fminf(rho_bar, is[e]) * (cur.r[e] + cur.g[e] * v_next - cur.v[e]) : 0.f;  // delta_s
        }
        // fold the lane's V steps: acc_first = B + A * (carry into the lane)
        float A = a[V - 1], B = b[V - 1];
#pragma unroll
        for (int e = V - 2; e >= 0; e--) {
            B = fmaf(a[e], B, b[e]);
            A *= a[e];
        }
        warp_reverse_linear_scan(A, B, lane);
        const float acc_first = fmaf(A, carry, B);
        float lane_carry = __shfl_down_sync(0xffffffffu, acc_first, 1);
        if (lane == 31) lane_carry = carry;
        float acc[V], vs[V];
        float run = lane_carry;
#pragma unroll
        for (int e = V - 1; e >= 0; e--) {
            run = fmaf(a[e], run, b[e]);
            acc[e] = run;
            vs[e] = cur.v[e] + run;
        }
        float vs_after = __shfl_down_sync(0xffffffffu, vs[0], 1);
        if (lane == 31) vs_after = vs_next_chunk;
        float adv[V];
#pragma unroll
        for (int e = 0; e < V; e++) {
            const int s = s0 + e;
            float vs_next = e + 1 < V ? vs[e + 1] : vs_after;
            if (s >= t - 1) vs_next = boot;
            adv[e] = fminf(pg_rho_bar, is[e]) * (cur.r[e] + cur.g[e] * vs_next - cur.v[e]);
        }
        bool stored = false;
        if constexpr (V == 4) {
            if (s0 + 3 < t) {
                *reinterpret_cast<float4*>(vs_out + base + s0) = make_float4(vs[0], vs[1], vs[2], vs[3]);
                if (adv_out) *reinterpret_cast<float4*>(adv_out + base + s0) = make_float4(adv[0], adv[1], adv[2], adv[3]);
                stored = true;
            }
        }
        if (!stored) {
#pragma unroll
            for (int e = 0; e < V; e++)
                if (s0 + e < t) {
                    vs_out[base + s0 + e] = vs[e];
                    if (adv_out) adv_out[base + s0 + e] = adv[e];
                }
        }
        carry = __shfl_sync(0xffffffffu, acc[0], 0);
        vs_next_chunk = __shfl_sync(0xffffffffu, vs[0], 0);
        v_next_chunk = __shfl_sync(0xffffffffu, cur.v[0], 0);
        cur = nxt;
    }
}

int launch_vtrace_scan(int m, int t, const float* log_rho, const float* discount, const float* reward,
                       const float* value, const float* bootstrap, float rho_bar, float c_bar,
                       float pg_rho_bar, float lambda_, float* vs, float* pg_adv, cudaStream_t stream) {
    if (m <= 0 || t <= 0) return FI_OK;
    if (!log_rho || !discount || !reward || !value || !bootstrap || !vs)
        return set_error(FI_ERR_ARG, "vtrace: null argument");
    const uintptr_t al = (uintptr_t)log_rho | (uintptr_t)discount | (uintptr_t)reward | (uintptr_t)value | (uintptr_t)vs |
                         (uintptr_t)pg_adv;
    // 16-byte accesses need every trajectory to start on a 16-byte boundary
    const bool vec = (al & 15) == 0 && (t % 4) == 0 && t >= 64;
    const int warps = 8;
    const int grid = (m + warps - 1) / warps;
    // algorithmic traffic: 16 B in + 8 B out per transition, + 4 B per trajectory (bootstrap)
    LaunchScope ls("vtrace_scan_kernel", stream, (pg_adv ? 24.0 : 20.0) * (double)m * t + 4.0 * m, kWorkBytes);
    if (vec)
        vtrace_scan_kernel<4><<<grid, 32 * warps, 0, stream>>>(m, t, log_rho, discount, reward, value, bootstrap, rho_bar, c_bar,
                                                             pg_rho_bar, lambda_, vs, pg_adv);
    else
        vtrace_scan_kernel<1><<<grid, 32 * warps, 0, stream>>>(m, t, log_rho, discount, reward, value, bootstrap, rho_bar, c_bar,
                                                             pg_rho_bar, lambda_, vs, pg_adv);
    return ls.done();
}

// ---------------------------------------------------------------- fused loss head -------
// One warp per trajectory of a gathered batch [m, t, 256 words]. For every transition the
// lane reads the learner head row (16 logits + value), the record's behaviour logits, action,
// reward and discount, and in ONE reverse pass produces: log-softmax, log_rho, the V-trace
// scan, pg advantages, the three losses and d(total)/d(head) -- no [m,t] intermediates go
// through HBM between "scan" and "loss". Losses are accumulated in double (4 atomics/warp).
// Memory staging (per warp, shared memory): the 32 head rows of a chunk are one contiguous span of 32*ldh
// floats, loaded with coalesced accesses and read back one row per lane (row stride 17: conflict-free); the
// record fields are six 16-byte loads per lane (words 160..183 of the 1024-byte record); the gradient rows
// go through padded tiles and leave as 128-byte coalesced stores. (The first version read and wrote every
// row element by element from its own lane: 36 us for 22 MB, 0.09 of the HBM roofline.)
// kLegal (fi_learner_config.legal_action_mask): both softmaxes, the entropy and d(head) run over the support
// legal word (record word 182) | bit of the taken action. Outside the support every per-action operand is replaced before
// use (-inf into fmaxf and expf, 0 as log pi), so logits there (-inf or NaN included) never reach the arithmetic, p = 0
// and d(head) is exactly 0; the replacements are selects, not branches. The word sits in the record fields already
// loaded, so the masked head reads no extra bytes.
constexpr int kLossWarps = 4;
template <bool kLegal>
__global__ void __launch_bounds__(32 * kLossWarps)
vtrace_loss_head_kernel(const float* __restrict__ batch, int m, int t, const float* __restrict__ head, int ldh,
                        float rho_bar, float c_bar, float pg_rho_bar, float lambda_, float baseline_cost,
                        float entropy_cost, float* __restrict__ dhead, float* __restrict__ vs_out,
                        float* __restrict__ adv_out, double* __restrict__ losses, float* __restrict__ dhead_hi,
                        float* __restrict__ dhead_lo, int ld_split, HScale* __restrict__ dhead_hs) {
    __shared__ float s_head[kLossWarps][32 * kHead];
    __shared__ float s_out[kLossWarps][2][32 * 33];
    pdl_wait();
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int traj = blockIdx.x * kLossWarps + wib;
    if (traj >= m) return;
    float* hs = s_head[wib];
    float* o_a = s_out[wib][0];   // plain / hi tile, [32][33]
    float* o_b = s_out[wib][1];   // lo tile
    const float* slot = batch + (size_t)traj * t * kRecWords;
    const float boot = __ldg(slot + (size_t)(t - 1) * kRecWords + kWAux);
    float carry = 0.f, vs_next_chunk = boot, v_next_chunk = boot;
    double l_pg = 0.0, l_bl = 0.0, l_ent = 0.0;
    float dmax = 0.f;
    for (int c0 = ((t - 1) >> 5) << 5; c0 >= 0; c0 -= 32) {
        const int s = c0 + lane;
        const bool valid = s < t;
        const size_t row = (size_t)traj * t + (valid ? s : t - 1);
        const float* rec = slot + (size_t)(valid ? s : t - 1) * kRecWords;
        // stage the chunk's head rows: rows base_row .. base_row + nvalid - 1
        const int nvalid = min(32, t - c0);
        const size_t base_row = (size_t)traj * t + c0;
        __syncwarp();
        if (ldh == kHead) {
            for (int i = lane; i < nvalid * kHead; i += 32) hs[i] = __ldg(head + base_row * kHead + i);
        } else {
            for (int i = lane; i < nvalid * kHead; i += 32) hs[i] = __ldg(head + (base_row + i / kHead) * ldh + i % kHead);
        }
        // record fields: words 160..183 (obs tail, mu[16], action, reward, discount, aux, 2 unused)
        float rf[24];
        {
            const float4* r4 = reinterpret_cast<const float4*>(rec + 160);
#pragma unroll
            for (int k = 0; k < 6; k++) {
                const float4 q4 = __ldg(r4 + k);
                rf[4 * k] = q4.x; rf[4 * k + 1] = q4.y; rf[4 * k + 2] = q4.z; rf[4 * k + 3] = q4.w;
            }
        }
        __syncwarp();
        const float* h = hs + (valid ? lane : nvalid - 1) * kHead;
        float z[kNumActions], p[kNumActions];
        float mx = -INFINITY, mmx = -INFINITY;
        uint32_t sup = ~0u;   // support: bit j set = action j enters the softmaxes
        if constexpr (kLegal) {
            int a = __float_as_int(rf[kWAction - 160]);
            a = a < 0 ? 0 : (a >= kNumActions ? kNumActions - 1 : a);
            sup = __float_as_uint(rf[kWLegal - 160]) | (1u << a);
        }
        auto on = [&](int j) { return !kLegal || ((sup >> j) & 1u); };
#pragma unroll
        for (int j = 0; j < kNumActions; j++) {
            z[j] = h[j];
            mx = fmaxf(mx, on(j) ? z[j] : -INFINITY);
        }
        const float v = h[kNumActions];
        int act = __float_as_int(rf[kWAction - 160]);
        act = act < 0 ? 0 : (act >= kNumActions ? kNumActions - 1 : act);
        float se = 0.f, mu_se = 0.f, mu_a = 0.f, z_a = 0.f;
#pragma unroll
        for (int j = 0; j < kNumActions; j++) {
            const float mu = rf[kWMu - 160 + j];
            p[j] = mu;  // parked until the behaviour max is known
            mmx = fmaxf(mmx, on(j) ? mu : -INFINITY);
            se += expf(on(j) ? z[j] - mx : -INFINITY);
            if (j == act) { mu_a = mu; z_a = z[j]; }
        }
#pragma unroll
        for (int j = 0; j < kNumActions; j++) mu_se += expf(on(j) ? p[j] - mmx : -INFINITY);
        const float lse = mx + logf(se);
        const float logp_a = z_a - lse;
        const float log_mu_a = mu_a - (mmx + logf(mu_se));
        float plogp = 0.f;
#pragma unroll
        for (int j = 0; j < kNumActions; j++) {
            const float lp = on(j) ? z[j] - lse : 0.f;   // outside the support: p = 0 and a finite log pi
            p[j] = expf(on(j) ? lp : -INFINITY);
            z[j] = lp;  // z now holds log pi
            plogp = fmaf(p[j], lp, plogp);
        }
        const float r = rf[kWReward - 160], g = rf[kWDiscount - 160];
        const float is = expf(logp_a - log_mu_a);
        float v_next = __shfl_down_sync(0xffffffffu, v, 1);
        if (lane == 31 || s >= t - 1) v_next = v_next_chunk;
        float a = 0.f, b = 0.f;
        if (valid) {
            b = fminf(rho_bar, is) * (r + g * v_next - v);
            a = g * lambda_ * fminf(c_bar, is);
        }
        warp_reverse_linear_scan(a, b, lane);
        const float acc = fmaf(a, carry, b);
        const float vs = v + acc;
        float vs_next = __shfl_down_sync(0xffffffffu, vs, 1);
        if (lane == 31 || s >= t - 1) vs_next = vs_next_chunk;
        const float adv = fminf(pg_rho_bar, is) * (r + g * vs_next - v);
        float dv[kHead];
#pragma unroll
        for (int j = 0; j < kNumActions; j++) {
            const float d_pg = adv * (p[j] - (j == act ? 1.f : 0.f));
            const float d_ent = p[j] * (z[j] - plogp);
            dv[j] = fmaf(entropy_cost, d_ent, d_pg);   // 0 outside the support: p = 0 and j != act
        }
        dv[kNumActions] = -baseline_cost * (vs - v);
        if (valid) {
#pragma unroll
            for (int j = 0; j < kHead; j++) dmax = fmaxf(dmax, fabsf(dv[j]));
            if (vs_out) vs_out[row] = vs;
            if (adv_out) adv_out[row] = adv;
            l_pg += (double)(-logp_a * adv);
            l_bl += 0.5 * (double)(vs - v) * (double)(vs - v);
            l_ent += (double)plogp;
        }
        if (dhead) {  // plain rows: the chunk is one contiguous span of nvalid * ldh floats when ldh == 17
            __syncwarp();
#pragma unroll
            for (int j = 0; j < kHead; j++) o_a[lane * 33 + j] = dv[j];
            __syncwarp();
            for (int i = lane; i < nvalid * kHead; i += 32) {
                const int rr = i / kHead, j = i % kHead;
                dhead[(base_row + rr) * ldh + j] = o_a[rr * 33 + j];
            }
        }
        if (dhead_hi) {  // hi/lo pair for the tcgen05 3xTF32 GEMMs of the backward pass, padded rows of ld_split floats
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 32; j++) {
                float hv = 0.f, lv = 0.f;
                if (j < kHead) {
                    hv = __uint_as_float(__float_as_uint(dv[j]) & 0xFFFFE000u);
                    lv = dv[j] - hv;
                }
                o_a[lane * 33 + j] = hv;
                o_b[lane * 33 + j] = lv;
            }
            __syncwarp();
            if (ld_split == 32) {  // 128 contiguous bytes per row: one coalesced store per row and array
                for (int rr = 0; rr < nvalid; rr++) {
                    dhead_hi[(base_row + rr) * 32 + lane] = o_a[rr * 33 + lane];
                    dhead_lo[(base_row + rr) * 32 + lane] = o_b[rr * 33 + lane];
                }
            } else {
                for (int i = lane; i < nvalid * kHead; i += 32) {
                    const int rr = i / kHead, j = i % kHead;
                    dhead_hi[(base_row + rr) * ld_split + j] = o_a[rr * 33 + j];
                    dhead_lo[(base_row + rr) * ld_split + j] = o_b[rr * 33 + j];
                }
            }
        }
        carry = __shfl_sync(0xffffffffu, acc, 0);
        vs_next_chunk = __shfl_sync(0xffffffffu, vs, 0);
        v_next_chunk = __shfl_sync(0xffffffffu, v, 0);
    }
    if (dhead_hs) {   // max |dhead| for the fp16 split that follows: no separate pass over the array
        const uint32_t wm = __reduce_max_sync(0xffffffffu, __float_as_uint(dmax));
        if (lane == 0 && wm) atomicMax(reinterpret_cast<unsigned int*>(&dhead_hs->amax), wm);
    }
    l_pg = warp_sum(l_pg);
    l_bl = warp_sum(l_bl);
    l_ent = warp_sum(l_ent);
    if (lane == 0) {
        atomicAdd(losses + 1, l_pg);
        atomicAdd(losses + 2, l_bl);
        atomicAdd(losses + 3, l_ent);
        atomicAdd(losses + 0, l_pg + (double)baseline_cost * l_bl + (double)entropy_cost * l_ent);
    }
}

int launch_vtrace_loss_head(const void* batch, int m, int t, const float* head, int ldh, float rho_bar,
                            float c_bar, float pg_rho_bar, float lambda_, float baseline_cost,
                            float entropy_cost, bool legal, float* dhead, float* vs, float* pg_adv, double* losses,
                            cudaStream_t stream, float* dhead_hi, float* dhead_lo, int ld_split, HScale* dhead_hs) {
    if (m <= 0 || t <= 0) return FI_OK;
    if (!batch || !head || (!dhead && !dhead_hi) || !losses || ldh < kHead || (dhead_hi && (!dhead_lo || ld_split < kHead)))
        return set_error(FI_ERR_ARG, "vtrace loss head: bad argument");
    const int warps = kLossWarps;
    if ((reinterpret_cast<uintptr_t>(batch) & 15) != 0) return set_error(FI_ERR_ARG, "vtrace loss head: batch must be 16-byte aligned");
    // algorithmic traffic per transition: head row in (17 x 4 B) + dhead row out (17 x 4 B) + the record's
    // behaviour logits, action, reward, discount (19 x 4 B) = 212 B (+ 8 B when vs / pg_adv are written)
    // (the masked head's legal word lies in the same 16-byte load as the discount and aux words: no extra traffic)
    LaunchScope ls(legal ? "vtrace_loss_head_kernel_legal" : "vtrace_loss_head_kernel", stream,
                   (212.0 + (vs ? 4.0 : 0.0) + (pg_adv ? 4.0 : 0.0)) * (double)m * t, kWorkBytes);
    launch_pdl(legal ? vtrace_loss_head_kernel<true> : vtrace_loss_head_kernel<false>, dim3((m + warps - 1) / warps),
               dim3(32 * warps), 0, stream, (const float*)batch, m, t, head, ldh, rho_bar, c_bar, pg_rho_bar, lambda_,
               baseline_cost, entropy_cost, dhead, vs, pg_adv, losses, dhead_hi, dhead_lo, ld_split, dhead_hs);
    return ls.done();
}

}  // namespace fi

extern "C" {

int fi_op_vtrace(int m, int t, const float* log_rho, const float* discount, const float* reward, const float* value,
                 const float* bootstrap, float rho_bar, float c_bar, float pg_rho_bar, float lambda_, float* vs,
                 float* pg_adv, void* stream) {
    return fi::launch_vtrace_scan(m, t, log_rho, discount, reward, value, bootstrap, rho_bar, c_bar, pg_rho_bar,
                                  lambda_, vs, pg_adv, (cudaStream_t)stream);
}

int fi_op_vtrace_loss_head(const void* batch, int m, int t, const float* head, int ldh, float rho_bar, float c_bar,
                           float pg_rho_bar, float lambda_, float baseline_cost, float entropy_cost, float* dhead,
                           float* vs, float* pg_adv, double* losses, void* stream) {
    return fi::launch_vtrace_loss_head(batch, m, t, head, ldh, rho_bar, c_bar, pg_rho_bar, lambda_, baseline_cost,
                                       entropy_cost, false, dhead, vs, pg_adv, losses, (cudaStream_t)stream);
}

int fi_op_vtrace_loss_head_legal(const void* batch, int m, int t, const float* head, int ldh, float rho_bar, float c_bar,
                                 float pg_rho_bar, float lambda_, float baseline_cost, float entropy_cost, float* dhead,
                                 float* vs, float* pg_adv, double* losses, void* stream) {
    return fi::launch_vtrace_loss_head(batch, m, t, head, ldh, rho_bar, c_bar, pg_rho_bar, lambda_, baseline_cost,
                                       entropy_cost, true, dhead, vs, pg_adv, losses, (cudaStream_t)stream);
}
}
