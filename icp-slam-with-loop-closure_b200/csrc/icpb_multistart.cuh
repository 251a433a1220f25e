// Multi-start alignment (icpb_run_multistart_host): every scan pair is aligned from K shared start
// transforms and the start with the smallest error wins.  Two small kernels around the unchanged
// alignment kernel:
//   - the expansion writes the problems of one slice of pairs -- pair (p, start k) is problem
//     p_local * K + k, so a pair's K starts sit next to each other in the queue and run at the same
//     time on different CTAs -- with the composed guess G = init[p] . S[k] of include/icpb.h;
//   - the selection reads each pair's K errors and keeps the first smallest one (np.argmin's rule).
// The problems themselves go through the ordinary launch, so each one gives the bits of icpb_run_host
// on the expanded pair list.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace icpb {

constexpr int kMultistartThreads = 256;

// One composed guess, 2x3 rows: G = I . S with every product and sum rounded to nearest on its own
// (no FMA contraction), left to right -- the formula of include/icpb.h, which numpy's element-wise
// `*` and `+` evaluate to the same bits.
__device__ __forceinline__ void compose_start(const double *I, const double *S, double *G)
{
    for (int r = 0; r < 2; ++r) {
        const double a = I[3 * r], b = I[3 * r + 1], t = I[3 * r + 2];
        G[3 * r]     = __dadd_rn(__dmul_rn(a, S[0]), __dmul_rn(b, S[3]));
        G[3 * r + 1] = __dadd_rn(__dmul_rn(a, S[1]), __dmul_rn(b, S[4]));
        G[3 * r + 2] = __dadd_rn(__dadd_rn(__dmul_rn(a, S[2]), __dmul_rn(b, S[5])), t);
    }
}

// The n * K problems of a slice of n pairs: epairs[q] = pairs[q / K], eG[q] = init[q / K] . S[q % K]
// (init == nullptr: the identity).  A slice split by scan length also gets its queue order:
// pair_order (n entries) lists the slice's pairs in queue order, and every one of them stands for its
// K problems, order[q] = pair_order[q / K] * K + q % K.
__global__ void __launch_bounds__(kMultistartThreads)
multistart_expand_kernel(const int32_t *pairs, const double *init, const double *starts, int32_t K, int64_t n,
                         const int32_t *pair_order, int32_t *epairs, double *eG, int32_t *order)
{
    const int64_t nq = n * K;
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t pl = q / K;
        const int32_t k = (int32_t)(q - pl * K);
        epairs[2 * q] = pairs[2 * pl];
        epairs[2 * q + 1] = pairs[2 * pl + 1];
        double I[6] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0};
        if (init)
            for (int j = 0; j < 6; ++j) I[j] = init[6 * pl + j];
        double G[6];
        compose_start(I, starts + 6 * k, G);
        for (int j = 0; j < 6; ++j) eG[6 * q + j] = G[j];
        if (order) order[q] = pair_order[pl] * K + k;
    }
}

// One thread per pair: the smallest of its K errors, the first one on ties (strict < over ascending k),
// and that problem's transform, error and pass count.
__global__ void __launch_bounds__(kMultistartThreads)
multistart_select_kernel(const double *eT, const double *eerr, const int32_t *epasses, int32_t K, int64_t n,
                         double *T, double *err, int32_t *passes, int32_t *start)
{
    for (int64_t p = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; p < n; p += (int64_t)gridDim.x * blockDim.x) {
        const double *e = eerr + p * K;
        double best = e[0];
        int32_t kb = 0;
        for (int32_t k = 1; k < K; ++k) {
            const double v = e[k];
            if (v < best) { best = v; kb = k; }
        }
        const int64_t w = p * K + kb;
        for (int j = 0; j < 6; ++j) T[6 * p + j] = eT[6 * w + j];
        err[p] = best;
        passes[p] = epasses[w];
        start[p] = kb;
    }
}

}  // namespace icpb
