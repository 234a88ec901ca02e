// PopArt value normalisation (van Hasselt et al. 2016, "Learning values across many orders of magnitude"; Hessel et al. 2019,
// "Multi-task deep RL with PopArt"): the two small kernels around the loss head's kPopArt instantiation (vtrace.cu).
//
//  * popart_sums_kernel reduces the loss head's per-trajectory partials {sum vs, sum vs^2, valid steps} to S1, S2, N in a fixed
//    order, before the data-parallel all-reduce carries them with the loss sums: the statistics feed the parameters, so two
//    identical runs must give the same bits (double atomics would not).
//  * popart_update_kernel runs after the optimiser: mu, nu <- (1 - beta) (mu, nu) + beta (S1 / N, S2 / N), then the value row of
//    the head (head.w row 16, head.b[16]) is rescaled so that sigma n + mu is unchanged, and, when the step publishes, the
//    snapshot's value row is written in reward units (w_pub = sigma w, b_pub = sigma b + mu). Every quantity is computed in double
//    and rounded to fp32 once. With update = 0 it only publishes (after the device-to-device snapshot copy of publish_async).
// The rules are stated in include/fi_learner.h (popart_beta) and restated in float64 by tests/popart_reference.py.
#include "fi_internal.cuh"

namespace fi {

constexpr int kSumsThreads = 256;
__global__ void __launch_bounds__(kSumsThreads) popart_sums_kernel(const double* __restrict__ part, int m, double* __restrict__ sums) {
    __shared__ double sh[3][kSumsThreads];
    pdl_wait();
    double a[3] = {0.0, 0.0, 0.0};
    for (int b = threadIdx.x; b < m; b += kSumsThreads)
        for (int k = 0; k < 3; k++) a[k] += part[3 * (size_t)b + k];
    for (int k = 0; k < 3; k++) sh[k][threadIdx.x] = a[k];
    __syncthreads();
    for (int w = kSumsThreads / 2; w > 0; w >>= 1) {   // a fixed tree: the same order on every launch
        if ((int)threadIdx.x < w)
            for (int k = 0; k < 3; k++) sh[k][threadIdx.x] += sh[k][threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x < 3) sums[threadIdx.x] = sh[threadIdx.x][0];
}

int launch_popart_sums(const double* part, int m, double* sums, cudaStream_t st) {
    if (m <= 0) return FI_OK;
    if (!part || !sums) return set_error(FI_ERR_ARG, "popart sums: null argument");
    LaunchScope ls("popart_sums_kernel", st, 24.0 * m + 24.0, kWorkBytes);
    launch_pdl(popart_sums_kernel, dim3(1), dim3(kSumsThreads), 0, st, part, m, sums);
    return ls.done();
}

__global__ void __launch_bounds__(kHid)
popart_update_kernel(PopArtState* __restrict__ st, const double* __restrict__ sums, double beta, float* __restrict__ params,
                     float* __restrict__ snap, int w_off, int b_off, int update) {
    const double mu0 = st->mu, nu0 = st->nu;
    double mu = mu0, nu = nu0;
    const bool upd = update && sums[2] > 0.0;
    if (upd) {
        const double n = sums[2], keep = __dsub_rn(1.0, beta);
        mu = __dadd_rn(__dmul_rn(keep, mu0), __dmul_rn(beta, __ddiv_rn(sums[0], n)));
        nu = __dadd_rn(__dmul_rn(keep, nu0), __dmul_rn(beta, __ddiv_rn(sums[1], n)));
    }
    const double sig0 = popart_sigma(mu0, nu0), sig = popart_sigma(mu, nu);
    const int i = threadIdx.x;
    float w = params[w_off + i];
    if (upd) {
        w = (float)__ddiv_rn(__dmul_rn((double)w, sig0), sig);
        params[w_off + i] = w;
    }
    if (snap) snap[w_off + i] = popart_publish_w(sig, w);
    if (i == 0) {
        float b = params[b_off];
        if (upd) {
            b = (float)__ddiv_rn(__dsub_rn(__dadd_rn(__dmul_rn(sig0, (double)b), mu0), mu), sig);
            params[b_off] = b;
        }
        if (snap) snap[b_off] = popart_publish_b(sig, mu, b);
    }
    __syncthreads();   // every thread has read the old statistics
    if (i == 0 && upd) {
        st->mu = mu;
        st->nu = nu;
        st->mu_f = (float)mu;
        st->sigma_f = (float)sig;
    }
}

void popart_launch_desc(PopArtState* st, const double* sums, double beta, float* params, float* snap, int w_off, int b_off, int update,
                        PopArtLaunchDesc* d) {
    d->func = (const void*)popart_update_kernel;
    d->st = st; d->sums = sums; d->beta = beta; d->params = params; d->snap = snap;
    d->w_off = w_off; d->b_off = b_off; d->update = update;
    d->args[0] = &d->st; d->args[1] = &d->sums; d->args[2] = &d->beta; d->args[3] = &d->params; d->args[4] = &d->snap;
    d->args[5] = &d->w_off; d->args[6] = &d->b_off; d->args[7] = &d->update;
}

int launch_popart_update(PopArtLaunchDesc* d, cudaStream_t stream) {
    // algorithmic traffic: the 513-value row in and out (+ out to the snapshot), the statistics and sums
    LaunchScope ls("popart_update_kernel", stream, 513.0 * 4.0 * (d->update ? 2.0 : 1.0) + (d->snap ? 513.0 * 4.0 : 0.0) + 72.0,
                   kWorkBytes);
    const cudaError_t e = cudaLaunchKernel(d->func, dim3(1), dim3(kHid), d->args, 0, stream);
    if (e != cudaSuccess) return set_error(FI_ERR_CUDA, "launch of popart_update_kernel failed: %s", cudaGetErrorString(e));
    return ls.done();
}

}  // namespace fi
