// Submaps (icpb_set_submaps): scans of the resident table merged into new scans appended to it.  One
// kernel, one thread per output point (grid-stride): the point's member is found by a binary search in
// the per-member output offsets, its base point is read, mapped by the member's 2x3 transform with the
// fixed formula of include/icpb.h, and either stored (write mode) or only tested against ICPB_MAX_COORD
// (check mode, out == nullptr).  The host runs the check first and writes only a table it has accepted,
// so a rejected call never touches the resident table.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace icpb {

constexpr int kSubmapThreads = 256;

// One merged point: every product and sum rounded to nearest on its own (no FMA contraction), the sum of
// the two products first -- numpy's element-wise (T00 * x + T01 * y) + T02 gives the same bits.
__device__ __forceinline__ double2 submap_point(const double *T, double2 p)
{
    return make_double2(__dadd_rn(__dadd_rn(__dmul_rn(T[0], p.x), __dmul_rn(T[1], p.y)), T[2]),
                        __dadd_rn(__dadd_rn(__dmul_rn(T[3], p.x), __dmul_rn(T[4], p.y)), T[5]));
}

// n_members members, in submap order; member k is base points [src[k], src[k] + mout[k+1] - mout[k]) of
// xy and becomes output points [mout[k], mout[k+1]) (mout[0] = 0).  Write mode stores them at out;
// check mode (out == nullptr) sets *bad when a merged coordinate is not within ICPB_MAX_COORD.
__global__ void __launch_bounds__(kSubmapThreads)
submap_merge_kernel(const double2 *xy, const int64_t *src, const int64_t *mout, const double *T, int64_t n_members,
                    double2 *out, int32_t *bad)
{
    const int64_t total = mout[n_members];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t lo = 0, hi = n_members - 1;                     // the last member with mout[k] <= i
        while (lo < hi) {
            const int64_t mid = (lo + hi + 1) >> 1;
            if (mout[mid] <= i) lo = mid; else hi = mid - 1;
        }
        const double2 q = submap_point(T + 6 * lo, xy[src[lo] + (i - mout[lo])]);
        if (out)
            out[i] = q;
        else if (!(fabs(q.x) <= ICPB_MAX_COORD) || !(fabs(q.y) <= ICPB_MAX_COORD))
            *bad = 1;
    }
}

}  // namespace icpb
