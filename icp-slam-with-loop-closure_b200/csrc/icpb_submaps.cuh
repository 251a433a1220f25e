// Submaps (icpb_set_submaps): scans of the resident table merged into new scans appended to it.  One
// kernel, one thread per output point (grid-stride): the point's member is found by a binary search in
// the per-member output offsets, its base point is read, mapped by the member's 2x3 transform with the
// fixed formula of include/icpb.h, and either stored (write mode) or only tested against ICPB_MAX_COORD
// (check mode, out == nullptr).  The host runs the check first and writes only a table it has accepted,
// so a rejected call never touches the resident table.  With a voxel filter (icpb_set_submaps_voxel) the write
// mode merges into scratch instead, and the kernels below keep the first point of every grid cell.
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

// ---- Voxel filter (icpb_set_submaps_voxel): of every submap, the first merged point of every grid cell.
// The merged points sit in scratch, submap m at [soff[m], soff[m+1]).  Each submap has its own open-addressing
// hash of cells, slots [hoff[m], hoff[m+1]) of `hash` (a power-of-two capacity of at least twice the submap's
// length, so a probe always ends; empty = -1), holding int32 indices local to the submap.
//
// Determinism.  A slot is claimed once, by a CAS from empty, and from then on only atomicMin stores into it,
// and only an index of the point whose cell the claiming point had.  So every index a slot ever holds belongs
// to one cell, and the value only decreases.  Linear probing without deletion puts a cell in at most one slot:
// a point walks past a slot only when it holds another cell, and a slot never changes cell or becomes empty.
// Every point of a cell ends at that slot and stores its index there with a CAS or an atomicMin, so the final
// value is the smallest index of the cell -- its first point in merged order -- whatever the thread order.

// The cell of a point: floor(x / voxel) with the division correctly rounded; numpy's
// np.floor(x / v).astype(np.int64) gives the same bits.  Exact in int64 for |x| <= ICPB_MAX_COORD and
// voxel >= ICPB_MIN_VOXEL (|x / voxel| <= 1e16).
__device__ __forceinline__ longlong2 voxel_cell(double2 p, double voxel)
{
    return make_longlong2(__double2ll_rz(floor(__ddiv_rn(p.x, voxel))), __double2ll_rz(floor(__ddiv_rn(p.y, voxel))));
}

__device__ __forceinline__ uint64_t voxel_hash(longlong2 c)
{
    uint64_t h = (uint64_t)c.x * 0x9E3779B97F4A7C15ull ^ (uint64_t)c.y * 0xC2B2AE3D27D4EB4Full;
    h ^= h >> 31; h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 29;
    return h;
}

// The last k in [0, n) with off[k] <= i (off[0] = 0 <= i).
__device__ __forceinline__ int64_t voxel_owner(const int64_t *off, int64_t n, int64_t i)
{
    int64_t lo = 0, hi = n - 1;
    while (lo < hi) {
        const int64_t mid = (lo + hi + 1) >> 1;
        if (off[mid] <= i) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// One thread per merged point: its cell into its submap's hash (the rule above).
__global__ void __launch_bounds__(kSubmapThreads)
submap_voxel_insert_kernel(const double2 *pts, const int64_t *soff, const int64_t *hoff, int64_t n_submaps,
                           double voxel, int32_t *hash)
{
    const int64_t total = soff[n_submaps];
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t m = voxel_owner(soff, n_submaps, i);
        const double2 *P = pts + soff[m];
        int32_t *H = hash + hoff[m];
        const uint64_t mask = (uint64_t)(hoff[m + 1] - hoff[m]) - 1;
        const int32_t l = (int32_t)(i - soff[m]);
        const longlong2 c = voxel_cell(P[l], voxel);
        for (uint64_t s = voxel_hash(c) & mask;; s = (s + 1) & mask) {
            const int32_t o = atomicCAS(&H[s], -1, l);
            if (o < 0) break;
            const longlong2 oc = voxel_cell(P[o], voxel);
            if (oc.x == c.x && oc.y == c.y) {
                if (l < o) atomicMin(&H[s], l);
                break;
            }
        }
    }
}

// One thread per hash slot: the first point of the slot's cell gets keep flag 1 (flag is zeroed before).
__global__ void __launch_bounds__(kSubmapThreads)
submap_voxel_keep_kernel(const int32_t *hash, const int64_t *soff, const int64_t *hoff, int64_t n_submaps,
                         int64_t *flag)
{
    const int64_t total = hoff[n_submaps];
    for (int64_t s = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; s < total; s += (int64_t)gridDim.x * blockDim.x) {
        const int32_t v = hash[s];
        if (v >= 0) flag[soff[voxel_owner(hoff, n_submaps, s)] + v] = 1;
    }
}

// After the exclusive scan of the flags (pos, n_submaps + 1 boundaries): the kept points before each submap.
__global__ void submap_voxel_bounds_kernel(const int64_t *pos, const int64_t *soff, int64_t n_submaps, int64_t *kept_off)
{
    for (int64_t m = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; m <= n_submaps; m += (int64_t)gridDim.x * blockDim.x)
        kept_off[m] = pos[soff[m]];
}

// One thread per merged point: a kept point (its scan value steps) to its place in the compacted submaps.
__global__ void __launch_bounds__(kSubmapThreads)
submap_voxel_scatter_kernel(const double2 *pts, const int64_t *pos, int64_t n_pts, double2 *out)
{
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n_pts; i += (int64_t)gridDim.x * blockDim.x)
        if (pos[i + 1] != pos[i]) out[pos[i]] = pts[i];
}

}  // namespace icpb
