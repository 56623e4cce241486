// rdf_cells.cuh -- the exclusive scan of the counting sort, shared by the cell lists of
// orthorhombic (rdf_cells.cu) and triclinic (rdf_tri.cu) cells.  Grid: any per-frame
// struct with the frame's cell count in `ncell`.
#pragma once

#include "rdf_device.cuh"

namespace {

using namespace rdfdev;

struct ScanFilter {            // optional: build the frames' FrameFilter in the scan kernel
    const FrameBox *boxes;     // [F] (already offset to the group of frames)
    const unsigned *ext1, *ext2;
    FrameFilter *out;
    FilterPrep prep;
};

// pass 2: exclusive scan of the per-cell counts; grid = (frames, groups), one block each.
// Tiles of kScanTile counters go through shared memory: coalesced load, every thread scans
// its own 32 consecutive counters (rows padded by one word per 32: conflict-free), block
// scan of the row sums by warp shuffles, coalesced store.
constexpr int kScanTile = 32768;
constexpr int kScanPer = kScanTile / 1024;

template <class Grid>
__global__ void __launch_bounds__(1024)
    cells_scan_kernel(const int *__restrict__ cnt, int *__restrict__ start, int cstride,
                      int n_frames, const Grid *__restrict__ grids, const ScanFilter F)
{
    extern __shared__ int tile[];                      // kScanTile + kScanTile / 32 words
    __shared__ int warp_sums[32];
    const int frame = blockIdx.x, group = blockIdx.y;
    const int ncell = grids[frame].ncell;
    const int64_t base = ((int64_t)group * n_frames + frame) * cstride;
    const int *c = cnt + base;
    int *s = start + base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int carry = 0;
    for (int t0 = 0; t0 < ncell; t0 += kScanTile) {
        const int n = min(kScanTile, ncell - t0);
        for (int k = tid; k < kScanTile; k += 1024) tile[k + (k >> 5)] = k < n ? c[t0 + k] : 0;
        __syncthreads();
        const int k0 = tid * kScanPer;
        int v[kScanPer], local = 0;
#pragma unroll
        for (int j = 0; j < kScanPer; ++j) {
            v[j] = tile[k0 + j + ((k0 + j) >> 5)];
            local += v[j];
        }
        int incl = local;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) warp_sums[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            int w = warp_sums[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t = __shfl_up_sync(0xffffffffu, w, o);
                if (lane >= o) w += t;
            }
            warp_sums[lane] = w;
        }
        __syncthreads();
        int run = carry + incl - local + (warp ? warp_sums[warp - 1] : 0);
#pragma unroll
        for (int j = 0; j < kScanPer; ++j) {
            tile[k0 + j + ((k0 + j) >> 5)] = run;
            run += v[j];
        }
        carry += warp_sums[31];
        __syncthreads();
        for (int k = tid; k < n; k += 1024) s[t0 + k] = tile[k + (k >> 5)];
        __syncthreads();
    }
    if (tid == 0) s[ncell] = carry;
    if (F.out != nullptr && group == 0 && tid == 0) {
        unsigned e1[6], e2[6];
        for (int k = 0; k < 6; ++k) {
            const unsigned a = F.ext1[frame * 6 + k], b = F.ext2[frame * 6 + k];
            e1[k] = k < 3 ? ~a : a;
            e2[k] = k < 3 ? ~b : b;
        }
        F.out[frame] = filter_prepare_frame(F.boxes[frame], e1, e2, F.prep);
    }
}

}  // namespace
