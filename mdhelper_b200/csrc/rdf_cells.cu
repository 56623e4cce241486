// rdf_cells.cu -- cell-list variant of the pair histogram (cut-off runs).
//
// Same per-pair arithmetic and binning as rdf.cu / rdf_filter.cu (rdf_device.cuh); only
// the set of candidate pairs shrinks: each frame's particles are counting-sorted into
// cells of edge >= r_cut*(1+1e-5) and every cell meets the 27 surrounding cells of the j
// group (with drop_axis: one cell along the dropped axis, and the 9 cells of the plane).
// This is the role MDAnalysis' grid search ("nsgrid") plays behind
// capped_distance for the reference (call site
// /root/reference/src/mdhelper/analysis/structure.py:93-96; SURVEY.md Appendix A items 2
// and 4).  Counts are identical to the all-pairs kernels by construction: a pair closer
// than r_cut always lies in adjacent cells, and every other candidate falls above the
// last threshold and is not counted.
//
// Pipeline per group of frames (sized so that its working set stays in L2):
//   cells_bin_kernel      raw float[n][3] -> (cell, rank-in-cell) + per-cell counts +
//                         coordinate extents (for the fp32 filter's error bound)
//   cells_scan_kernel     exclusive scan of the counts, one block per (frame, group);
//                         also builds the frame's FrameFilter (no extra launch)
//   cells_scatter_kernel  raw -> cell-sorted float4 (x, y, z, exclusion block id)
//   rdf_cellpair_kernel   the pair kernel (below); frames it declines go to
//   rdf_cells_kernel      the fp64 kernel (every pair through the reference arithmetic)
// No packed or pair-interleaved copy of the coordinates is made any more: the raw
// floats are read twice (second time from L2) and the sorted float4 array is the only
// intermediate.
//
// rdf_cellpair_kernel.  One WARP per cell, persistent warps fetching chunks of cells
// from a global counter.  The cell's particles and the particles of its stencil cells
// (half stencil of 13 cells + itself when the two groups coincide, 27 cells otherwise) are
// contiguous runs of the sorted array -- three x-adjacent cells are one run -- and are
// copied into a per-warp shared-memory buffer with one bulk copy (cp.async.bulk, the TMA
// unit's 1-D mode) per run, completion on a per-warp mbarrier; the copy of the next cell
// is in flight while the current one is computed.  The cell's n_i particles are then
// dealt to the lanes IPT at a time (ni = ceil(n_i / IPT) lanes hold them all) and the 32
// lanes split into ways = 32 / ni groups that walk the candidate list with stride `ways`:
// every lane-step evaluates IPT pairs (two per packed f32x2 instruction) against ONE
// candidate read as a 16-byte shared-memory load (lanes of a way read the same address:
// broadcast; the ways read consecutive 16-byte words: one wavefront).  The arithmetic,
// the fixed-point bin coordinate, the uncertainty window and the histogram update are
// those of rdf_filter.cu (same device functions -> same bits); uncertain pairs go to a
// per-warp list that is re-evaluated with the fp64 arithmetic as soon as the cell is done,
// from the same shared-memory buffer.  A candidate list that does not fit the buffer (a
// dense cluster) is copied and computed in segments; a cell with more particles than that
// is handed to the fp64 kernel, whose thread-per-particle layout spreads it over the device.

#include <stdio.h>

#include <algorithm>
#include <type_traits>

#include "rdf_cells.cuh"
#include "rdf_device.cuh"

using namespace rdfdev;

namespace {

// Grid axis k runs along physical axis axis[k]; box, inv_w and nc are per GRID axis.  The
// axes are the physical ones in order, except with a dropped axis (two-dimensional runs):
// that one becomes grid axis 2 with a single cell, so that the stencils keep their runs of
// three x-adjacent cells along a kept axis and only have to leave out the rows at dz != 0.
struct CellGrid {          // per frame
    double box[3];
    double inv_w[3];       // nc / box
    int nc[3];
    int axis[3];
    int ncell;
};

__device__ __forceinline__ int cell_coord(float x, double box, double inv_w, int nc)
{
    double w = (double)x;
    if (!(w >= 0.0 && w < box))              // into [0, box) for cell assignment only
        w -= floor(w / box) * box;
    int c = (int)(w * inv_w);
    return min(max(c, 0), nc - 1);
}

__device__ __forceinline__ int cell_id(float x, float y, float z, const CellGrid &g, int &cx,
                                       int &cy, int &cz)
{
    auto pick = [&](int a) { return a == 0 ? x : (a == 1 ? y : z); };
    cx = cell_coord(pick(g.axis[0]), g.box[0], g.inv_w[0], g.nc[0]);
    cy = cell_coord(pick(g.axis[1]), g.box[1], g.inv_w[1], g.nc[1]);
    cz = cell_coord(pick(g.axis[2]), g.box[2], g.inv_w[2], g.nc[2]);
    return (cz * g.nc[1] + cy) * g.nc[0] + cx;
}

// the coordinate the pair arithmetic sees: a dropped axis is zeroed first, as
// rdf_pack_kernel does for the all-pairs kernels, then the grid-search wrap if the frame
// takes it (ortho_pbc_f32 keeps +0 at +0)
__device__ __forceinline__ float4 cells_coords(float x, float y, float z, int drop_axis,
                                               const FrameBox &fb)
{
    if (drop_axis == 0) x = 0.f;
    if (drop_axis == 1) y = 0.f;
    if (drop_axis == 2) z = 0.f;
    if (fb.prewrap) {
        x = ortho_pbc_f32(x, fb.box[0]);
        y = ortho_pbc_f32(y, fb.box[1]);
        z = ortho_pbc_f32(z, fb.box[2]);
    }
    return make_float4(x, y, z, 0.f);
}

// ---- counting sort, straight from the raw coordinates ------------------------------

// 256 particles per step: their 768 floats are read as one contiguous run (coalesced,
// unlike three stride-3 loads per thread) and regrouped through shared memory.
__device__ __forceinline__ void load_xyz_256(const float *__restrict__ src, int64_t i0, int64_t n,
                                             float *stage, int tid)
{
    const int64_t f0 = 3 * i0, fend = 3 * n;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int64_t f = f0 + k * 256 + tid;
        stage[k * 256 + tid] = f < fend ? src[f] : 0.f;
    }
}

// pass 1: cell of every particle, rank inside its cell (old value of the cell counter),
// coordinate extents of the frame (ext == nullptr: not wanted) as order-preserving keys:
// ext[frame][0..2] = ~(smallest key) per axis, ext[frame][3..5] = largest key, both kept
// with atomicMax so that one zero fill initialises them
__global__ void __launch_bounds__(256)
    cells_bin_kernel(const float *__restrict__ raw, int64_t frame_stride, int n,
                     const CellGrid *__restrict__ grids, int *__restrict__ cnt, int cstride,
                     int2 *__restrict__ keyrank, unsigned *__restrict__ ext,
                     const FrameBox *__restrict__ boxes, int drop_axis)
{
    __shared__ float stage[3 * 256];
    __shared__ unsigned red[8][6];
    const int frame = blockIdx.y, tid = threadIdx.x;
    const CellGrid g = grids[frame];
    const FrameBox fb = boxes[frame];
    const float *src = raw + (int64_t)frame * frame_stride;
    unsigned lo[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, hi[3] = {0u, 0u, 0u};
    for (int64_t i0 = (int64_t)blockIdx.x * 256; i0 < n; i0 += (int64_t)gridDim.x * 256) {
        load_xyz_256(src, i0, n, stage, tid);
        __syncthreads();
        const int64_t i = i0 + tid;
        // warp-aggregated counter update: neighbours in the input often share a cell (atoms
        // of a molecule, lattice-ordered fluids), and 32 atomics on a few addresses serialise
        const unsigned active = __ballot_sync(0xffffffffu, i < n);
        if (i < n) {
            const float4 v = cells_coords(stage[3 * tid], stage[3 * tid + 1], stage[3 * tid + 2],
                                          drop_axis, fb);
            const float x = v.x, y = v.y, z = v.z;
            int cx, cy, cz;
            const int cell = cell_id(x, y, z, g, cx, cy, cz);
            const unsigned peers = __match_any_sync(active, cell);
            const int leader = __ffs(peers) - 1, lane = tid & 31;
            int base = 0;
            if (lane == leader)
                base = atomicAdd(&cnt[(int64_t)frame * cstride + cell], __popc(peers));
            base = __shfl_sync(peers, base, leader);
            const int r = base + __popc(peers & ((1u << lane) - 1u));
            keyrank[(int64_t)frame * n + i] = make_int2(cell, r);
            const unsigned kx = ext_key(x), ky = ext_key(y), kz = ext_key(z);
            lo[0] = min(lo[0], kx); hi[0] = max(hi[0], kx);
            lo[1] = min(lo[1], ky); hi[1] = max(hi[1], ky);
            lo[2] = min(lo[2], kz); hi[2] = max(hi[2], kz);
        }
        __syncthreads();
    }
    if (ext) {
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const unsigned l = __reduce_min_sync(0xffffffffu, lo[k]);
            const unsigned h = __reduce_max_sync(0xffffffffu, hi[k]);
            if ((tid & 31) == 0) { red[tid >> 5][k] = l; red[tid >> 5][3 + k] = h; }
        }
        __syncthreads();
        if (tid < 6) {
            unsigned v = red[0][tid];
            for (int w = 1; w < 8; ++w) v = tid < 3 ? min(v, red[w][tid]) : max(v, red[w][tid]);
            if (tid < 3) { if (v != 0xffffffffu) atomicMax(&ext[frame * 6 + tid], ~v); }
            else if (v != 0u) atomicMax(&ext[frame * 6 + tid], v);
        }
    }
}

// pass 3: raw -> cell-sorted float4 (x, y, z, exclusion block id)
__global__ void __launch_bounds__(256)
    cells_scatter_kernel(const float *__restrict__ raw, int64_t frame_stride, int n, int64_t excl,
                         const int *__restrict__ start, int cstride,
                         const int2 *__restrict__ keyrank, float4 *__restrict__ sorted,
                         const FrameBox *__restrict__ boxes, int drop_axis)
{
    __shared__ float stage[3 * 256];
    const int frame = blockIdx.y, tid = threadIdx.x;
    const float *src = raw + (int64_t)frame * frame_stride;
    const int *st = start + (int64_t)frame * cstride;
    for (int64_t i0 = (int64_t)blockIdx.x * 256; i0 < n; i0 += (int64_t)gridDim.x * 256) {
        load_xyz_256(src, i0, n, stage, tid);
        __syncthreads();
        const int64_t i = i0 + tid;
        if (i < n) {
            const int2 kr = keyrank[(int64_t)frame * n + i];
            // the same values the binning pass saw
            float4 v = cells_coords(stage[3 * tid], stage[3 * tid + 1], stage[3 * tid + 2],
                                    drop_axis, boxes[frame]);
            v.w = __int_as_float((int)(excl > 0 ? i / excl : i));
            sorted[(int64_t)frame * n + st[kr.x] + kr.y] = v;
        }
        __syncthreads();
    }
}

// ---- fp64 kernel: every candidate pair through the reference arithmetic ----------------

struct CellParams {
    const float4 *s1, *s2;        // cell-sorted particles, [F][n]
    int n1, n2;
    const int *start2;            // [F][cstride]
    int cstride;
    const CellGrid *grids;
    const FrameBox *boxes;
    const double *thr;
    int n_bins;
    BinGuess guess;
    unsigned long long *counts;
    unsigned long long *evals;
    int half;                     // same group: half stencil, weight 2
    const FrameFilter *filt;      // != nullptr: frames with wlim != 0 were done by the
                                  // fp32-filter kernel and are skipped here -- except the
    const int *cellflag;          // cells it flagged ([F][cstride], != 0: too crowded for
    const int *nflag;             // one warp) -- nflag[F]: how many per frame
};

template <int HIST>
__host__ __device__ inline size_t cells_smem_bytes(int n_bins)
{
    return align16(sizeof(double) * (n_bins + 1)) + hist_smem_bytes<HIST>(n_bins);
}

template <int HIST, bool EXCL, bool FAST>
__global__ void __launch_bounds__(kThreads, 2) rdf_cells_kernel(const CellParams P)
{
    extern __shared__ __align__(16) unsigned char smem[];
    double *sT = reinterpret_cast<double *>(smem);
    unsigned *sH =
        reinterpret_cast<unsigned *>(smem + align16(sizeof(double) * (P.n_bins + 1)));

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int frame = blockIdx.y;
    // frames the fp32-filter kernel has taken are not done again, apart from the cells it
    // handed over (a cluster far denser than the rest: one thread per particle spreads
    // that work over the device, one warp per cell would not)
    bool flagged_only = false;
    if (P.filt != nullptr && P.filt[frame].wlim != 0u) {
        if (P.nflag == nullptr || P.nflag[frame] == 0) return;
        flagged_only = true;
    }
    const int n_bins = P.n_bins;
    const int n_words = priv_words(n_bins);
    for (int k = tid; k <= n_bins; k += kThreads) sT[k] = P.thr[k];
    const int n_hist_words = (int)(hist_smem_bytes<HIST>(n_bins) / sizeof(unsigned));
    for (int k = tid; k < n_hist_words; k += kThreads) sH[k] = 0;
    __syncthreads();

    unsigned *myhist = (HIST == MDH_HIST_WARP_ATOMIC)
                           ? sH + warp * warp_hist_words(n_bins) + 1
                           : sH + (size_t)warp * n_words * 32;
    unsigned *bhist = sH + (size_t)kWarps * n_words * 32;
    unsigned char *lane_base = reinterpret_cast<unsigned char *>(myhist) + 4 * lane;
    const unsigned hist32 = (unsigned)__cvta_generic_to_shared(myhist);
    const unsigned trash32 = hist32 + 4u * (unsigned)(n_bins + lane);
    const BinGuess guess = P.guess;

    const CellGrid g = P.grids[frame];
    const FrameBox fb = P.boxes[frame];
    const float4 *s1 = P.s1 + (int64_t)frame * P.n1;
    const float4 *s2 = P.s2 + (int64_t)frame * P.n2;
    const int *start = P.start2 + (int64_t)frame * P.cstride;

    const int i = blockIdx.x * kThreads + tid;
    bool valid = i < P.n1;
    const float4 pi = s1[min(i, P.n1 - 1)];
    const int gi = __float_as_int(pi.w);
    int cx, cy, cz;
    const int my_cell = cell_id(pi.x, pi.y, pi.z, g, cx, cy, cz);
    if (flagged_only) valid = valid && P.cellflag[(int64_t)frame * P.cstride + my_cell] != 0;

    int steps = 0;                       // warp-uniform: increments since the last flush
    unsigned long long my_evals = 0;

    // One range of candidate partners [b, b + len) per lane; the loop bound is the
    // warp maximum so that flushes stay warp-uniform.  The first partner carries
    // weight w_first, the others w_rest (half-stencil runs: 1 for the self pair, 2
    // for every unordered pair).  The next partner is fetched one iteration ahead.
    auto sweep = [&](int b, int len, unsigned w_first, unsigned w_rest) {
        const int maxlen = __reduce_max_sync(0xffffffffu, len);
        my_evals += len;
        float4 nxt = __ldg(s2 + (len > 0 ? b : 0));
        for (int t = 0; t < maxlen; ++t) {
            const bool act = t < len;
            const float4 pj = nxt;
            nxt = __ldg(s2 + (t + 1 < len ? b + t + 1 : 0));
            const unsigned w = t == 0 ? w_first : w_rest;
            const double d2 = pair_d2(pi.x, pi.y, pi.z, pj, fb);
            const bool keep = act && !(EXCL && gi == __float_as_int(pj.w));
            if (HIST == MDH_HIST_WARP_ATOMIC && FAST) {
                bool below;
                const int j = slot_fast_parts(d2, sT, n_bins, guess, below);
                unsigned a = (below ? hist32 - 4u : hist32) + 4u * (unsigned)j;
                if ((!below && j == n_bins) || !keep) a = trash32;
                red_shared(a, w);
            } else {
                int slot = slot_of<FAST>(d2, sT, n_bins, guess);
                if (!keep) slot = 0;
                if (HIST == MDH_HIST_WARP_ATOMIC) {
                    if ((unsigned)(slot - 1) < (unsigned)n_bins)
                        atomicAdd(&myhist[slot - 1], w);
                } else {
                    priv_add(lane_base, slot, w);
                    steps += 2;
                    if (steps >= 253) {
                        priv_flush(myhist, bhist, n_words, n_bins, lane, 1u);
                        steps = 0;
                    }
                }
            }
        }
    };
    auto wrap = [](int v, int n) { return v < 0 ? v + n : (v >= n ? v - n : v); };
    // the three x-adjacent cells of row (y, z) are one contiguous range of the sorted
    // array, plus one more cell when the x stencil wraps around the box
    auto sweep_row = [&](int y, int z, unsigned w) {
        const int row = (z * g.nc[1] + y) * g.nc[0];
        const int xa = max(cx - 1, 0), xb = min(cx + 1, g.nc[0] - 1);
        const int b0 = start[row + xa];
        sweep(b0, valid ? start[row + xb + 1] - b0 : 0, w, w);
        const int xw = (cx == 0) ? g.nc[0] - 1 : (cx == g.nc[0] - 1 ? 0 : -1);
        const int bw = xw >= 0 ? start[row + xw] : 0;
        sweep(bw, (valid && xw >= 0) ? start[row + xw + 1] - bw : 0, w, w);
    };

    // a single cell along grid z (a dropped axis): the rows at dz = -1 and +1 would be the
    // own row again -- the stencil is the 9 cells (half: 4 + own) of the plane
    const int dz_max = g.nc[2] > 1 ? 1 : 0;
    if (!P.half) {
        // full stencil: every ordered (i, j) pair once
        for (int dz = -dz_max; dz <= dz_max; ++dz)
            for (int dy = -1; dy <= 1; ++dy)
                sweep_row(wrap(cy + dy, g.nc[1]), wrap(cz + dz, g.nc[2]), 1u);
    } else {
        // same group: half stencil.  Forward offsets (dz, dy, dx) > (0, 0, 0) in
        // lexicographic order visit every unordered pair of distinct cells exactly
        // once (the reverse offset belongs to the partner cell); weight 2 stands for
        // both orders.  The own cell contributes j >= i: the self pair once.
        if (dz_max)
            for (int dy = -1; dy <= 1; ++dy)
                sweep_row(wrap(cy + dy, g.nc[1]), wrap(cz + 1, g.nc[2]), 2u);
        sweep_row(wrap(cy + 1, g.nc[1]), cz, 2u);
        const int row = (cz * g.nc[1] + cy) * g.nc[0];
        const int xr = wrap(cx + 1, g.nc[0]);
        const int br = start[row + xr];
        sweep(br, valid ? start[row + xr + 1] - br : 0, 2u, 2u);
        sweep(i, valid ? start[row + cx + 1] - i : 0, 1u, 2u);
    }
    if (HIST == MDH_HIST_LANE_PRIVATE)
        priv_flush(myhist, bhist, n_words, n_bins, lane, 1u);
    __syncthreads();

    for (int k = tid; k < n_bins; k += kThreads) {
        unsigned long long s = 0;
        if (HIST == MDH_HIST_WARP_ATOMIC) {
#pragma unroll
            for (int w = 0; w < kWarps; ++w) s += sH[w * warp_hist_words(n_bins) + 1 + k];
        } else {
            s = bhist[k];
        }
        if (s) atomicAdd(&P.counts[k], s);
    }
    // evaluations actually performed (for the roofline bookkeeping)
    for (int o = 16; o; o >>= 1) my_evals += __shfl_xor_sync(0xffffffffu, my_evals, o);
    if (lane == 0 && my_evals) atomicAdd(P.evals, my_evals);
}

template <int HIST, bool EXCL, bool FAST>
int launch_cells(mdh_ctx *c, const CellParams &P, dim3 grid)
{
    const size_t smem = cells_smem_bytes<HIST>(P.n_bins);
    auto kern = rdf_cells_kernel<HIST, EXCL, FAST>;
    static thread_local size_t cached_smem = 0;
    static thread_local int cached_dev = -1;
    if (cached_smem < smem || cached_dev != c->device) {
        MDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)smem));
        cached_smem = smem;
        cached_dev = c->device;
    }
    kern<<<grid, kThreads, smem, c->stream>>>(P);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    return MDH_OK;
}

// ---- fp32-filter pair kernel: one warp per cell ------------------------------------------

#ifndef MDH_CP_THREADS
#define MDH_CP_THREADS 192
#endif
#ifndef MDH_CP_BLOCKS
#define MDH_CP_BLOCKS 2
#endif
constexpr int kCpThreads = MDH_CP_THREADS;     // 6 warps x 2 blocks per SM at 168 registers: measured
                                               // 22 % faster than 8 warps x 2 at 128 (profiles/README.md)
constexpr int kCpWarps = kCpThreads / 32;
constexpr int kCpRanges = 19;            // own cell + 9 rows x (main run, wrapped cell)
constexpr int kCpListCap = 64;           // deferred entries per warp and cell pass
constexpr int kCpSlack = 32;             // buffer words a strided walk may read past the list

struct CellPairParams {
    const float4 *s1, *s2;        // cell-sorted particles, [F][n1], [F][n2]
    int n1, n2;
    const int *start1, *start2;   // [F][cstride]
    int cstride;
    const CellGrid *grids;
    const FrameBox *boxes;
    const FrameFilter *filt;
    const double *thr;
    int n_bins;
    BinGuess guess;
    FilterConst fc;               // fc.sb: sub-bins of THIS kernel's histograms
    int fast_bins;
    unsigned long long *counts, *evals, *fstats;
    unsigned *work;               // work-item counter (zero at launch)
    int *cellflag, *nflag;        // cells handed over to the fp64 kernel ([F][cstride], [F])
    int n_frames;
    int max_ncell;                // largest cell count of the frames of this launch
    int chunk_cells;              // cells per work item
    int cap;                      // buffer capacity in particles (multiple of 32)
    unsigned long long sign2;     // 0x8000000080000000: the sign bits of a packed f32x2
};

__host__ __device__ inline size_t cp_smem_bytes(int n_bins, int sb, int cap)
{
    return 256 + align16(sizeof(double) * (n_bins + 1)) +
           (size_t)kCpWarps * 2 * (cap + kCpSlack) * sizeof(float4) +
           sizeof(unsigned) * (size_t)kCpWarps * ((((size_t)n_bins + 2) << sb) + 32) +
           sizeof(unsigned) * kCpWarps * kCpListCap + sizeof(int2) * kCpWarps * 2 * 32;
}

__device__ __forceinline__ void cp_mbar_init(unsigned bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void cp_mbar_expect(unsigned bar, unsigned bytes)
{
    asm volatile("{\n\t.reg .b64 st;\n\t"
                 "mbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}"
                 :: "r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_mbar_wait(unsigned bar, unsigned parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra W_%=;\n\t}"
        :: "r"(bar), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared (TMA unit), completion counted in bytes on `bar`
__device__ __forceinline__ void cp_bulk_g2s(unsigned dst, const void *src, unsigned bytes,
                                            unsigned bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
        :: "r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// ---- cold paths, kept out of line so that the hot loops stay small in the instruction
// cache (the first version inlined them and spent most of its stall cycles waiting for
// instructions) ---------------------------------------------------------------------------

// fp64 re-evaluation of the uncertain pairs between the lane particles ip[0 .. nv) and the
// candidate *jp: the main loop has added every one of them to the slot the fp32 arithmetic
// suggested; move the count if the reference arithmetic disagrees.  A pair with
// ip + k == jp is a self pair (own-cell pass) and was never counted.
template <bool EXCL, bool LOWER, int IPT>
__device__ __noinline__ void cp_fix(const CellPairParams &P, int frame, const float4 *ip, int nv,
                                    const float4 *jp, unsigned weight, const double *sT,
                                    unsigned hist32)
{
    const FrameFilter ff = P.filt[frame];
    const FrameBox fb = P.boxes[frame];
    const FilterConst fc = P.fc;
    const float4 pj = *jp;
    const unsigned span_l = LOWER ? fc.span : fc.cbits + fc.span;
    const int shift = fc.k - fc.sb;
    for (int k0 = 0; k0 < IPT; k0 += 2) {
        // the same fp32 function as the main loop (identical bits); which two particles
        // share a packed instruction does not matter, the halves are independent
        const float4 a0 = ip[min(k0, nv - 1)], a1 = ip[min(k0 + 1, nv - 1)];
        unsigned uu[2];
        filter_eval2<LOWER>(pk2(-a0.x, -a1.x), pk2(-a0.y, -a1.y), pk2(-a0.z, -a1.z),
                            pk2(pj.x, pj.x), pk2(pj.y, pj.y), pk2(pj.z, pj.z), ff, fc.scale,
                            ff.offm, fc.cbits, uu[0], uu[1]);
        for (int h = 0; h < 2; ++h) {
            const int k = k0 + h;
            const float4 a = h ? a1 : a0;
            const unsigned u = uu[h];
            if (k >= nv || ip + k == jp) continue;
            if (!(u < span_l) || !((u & ((1u << fc.k) - 1u)) < ff.wlim)) continue;
            if (EXCL && __float_as_int(a.w) == __float_as_int(pj.w)) continue;
            const unsigned word = (LOWER ? u : u - fc.cbits) >> shift;
            const double d2 = pair_d2(a.x, a.y, a.z, pj, fb);
            const int slot = P.fast_bins ? slot_fast(d2, sT, P.n_bins, P.guess)
                                         : slot_search(d2, sT, P.n_bins);
            if ((word >> fc.sb) == (unsigned)slot) continue;
            red_shared(hist32 + 4u * word, 0u - weight);
            red_shared(hist32 + 4u * ((unsigned)slot << fc.sb), weight);
        }
    }
}

template <bool HALF, bool EXCL, bool LOWER, bool AUDIT, int IPT>
__global__ void __launch_bounds__(kCpThreads, MDH_CP_BLOCKS)
    rdf_cellpair_kernel(const __grid_constant__ CellPairParams P)
{
    static_assert(IPT == 2 || IPT == 4, "particles are processed in packed pairs");
    extern __shared__ __align__(16) unsigned char smem[];
    const int n_bins = P.n_bins;
    const FilterConst fc = P.fc;
    const int cap = P.cap, bufw = cap + kCpSlack;
    const int hwords = ((n_bins + 2) << fc.sb) + 32;
    // layout: mbarriers | thresholds | candidate buffers | histograms | lists | ranges
    unsigned long long *sBar = reinterpret_cast<unsigned long long *>(smem);
    double *sT = reinterpret_cast<double *>(smem + 256);
    float4 *sBuf =
        reinterpret_cast<float4 *>(smem + 256 + align16(sizeof(double) * (n_bins + 1)));
    unsigned *sH = reinterpret_cast<unsigned *>(sBuf + (size_t)kCpWarps * 2 * bufw);
    unsigned *sList = sH + kCpWarps * hwords;
    int2 *sRng = reinterpret_cast<int2 *>(sList + kCpWarps * kCpListCap);
    unsigned *sCount = reinterpret_cast<unsigned *>(smem + 128);      // [kCpWarps]

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int k = tid; k <= n_bins; k += kCpThreads) sT[k] = P.thr[k];
    for (int k = tid; k < kCpWarps * hwords; k += kCpThreads) sH[k] = 0;
    if (tid < kCpWarps) sCount[tid] = 0;
    const unsigned bar32 = (unsigned)__cvta_generic_to_shared(sBar + 2 * warp);
    if (lane == 0) {
        cp_mbar_init(bar32, 1);
        cp_mbar_init(bar32 + 8, 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    float4 *wbuf = sBuf + (size_t)warp * 2 * bufw;            // two buffers of this warp
    const unsigned wbuf32 = (unsigned)__cvta_generic_to_shared(wbuf);
    int2 *wrng = sRng + warp * 2 * 32;
    unsigned *wlist = sList + warp * kCpListCap;
    unsigned *wcount = sCount + warp;
    const unsigned hist32 = (unsigned)__cvta_generic_to_shared(sH + warp * hwords);
    const int shift = fc.k - fc.sb;
    const unsigned hbase = hist32 - (LOWER ? 0u : ((fc.cbits >> shift) << 2));
    const unsigned span_l = LOWER ? fc.span : fc.cbits + fc.span;
    const unsigned trash_w = (span_l >> shift) + (unsigned)lane;
    const unsigned fmask = (1u << fc.k) - 1u;
    const float scale = fc.scale;
    // self pairs of a same-group run (distance 0) are not evaluated: their bin is known
    const int slot_zero = slot_search(0.0, sT, n_bins);
    const bool count_self = HALF && !EXCL && slot_zero >= 1 && slot_zero <= n_bins;

    unsigned phase = 0;                       // bit s: parity the next wait on buffer s uses
    unsigned long long my_evals = 0;          // lane 0 only
    unsigned acc_w = 0, n_deferred = 0, n_inline = 0;
    unsigned long long audit_bad = 0, audit_unc = 0;

    const int items_per_frame = (P.max_ncell + P.chunk_cells - 1) / P.chunk_cells;
    const int n_items = items_per_frame * P.n_frames;

    for (;;) {
        int item = 0;
        if (lane == 0) item = (int)atomicAdd(P.work, 1u);
        item = __shfl_sync(0xffffffffu, item, 0);
        if (item >= n_items) break;
        const int frame = item / items_per_frame;
        const int c0 = (item - frame * items_per_frame) * P.chunk_cells;
        const FrameFilter ff = P.filt[frame];
        if (ff.wlim == 0u) {                  // left to the fp64 kernel
            if (c0 == 0 && lane == 0) atomicAdd(&P.fstats[4], 1ull);
            continue;
        }
        const float offm = ff.offm;
        const int ncx = P.grids[frame].nc[0], ncy = P.grids[frame].nc[1],
                  ncz = P.grids[frame].nc[2];
        const int c1 = min(c0 + P.chunk_cells, ncx * ncy * ncz);

        // Stage 1 of the per-cell pipeline: the runs of the sorted arrays that make up the
        // candidate list of cell (cx, cy, cz).  Lane r describes run r: r = 0 the cell's own
        // particles (group 1), r >= 1 the stencil runs of group 2.  Only LOADS the run
        // bounds; they are consumed one cell later, so their latency is hidden.
        auto plan = [&](int cell, int cx, int cy, int cz, int &b, int &e) {
            const int *st1 = P.start1 + (int64_t)frame * P.cstride;
            const int *st2 = P.start2 + (int64_t)frame * P.cstride;
            auto wrap = [](int v, int n) { return v < 0 ? v + n : (v >= n ? v - n : v); };
            const int *pb = st1, *pe = st1;          // empty run: b == e
            if (lane == 0) {
                pb = st1 + cell;
                pe = pb + 1;
            } else if (lane < kCpRanges) {
                const int r = lane - 1;              // 0..17: row r / 2, run r & 1
                const int row_i = r >> 1;            // 0..8 = (dz + 1) * 3 + (dy + 1)
                const int dz = row_i / 3 - 1, dy = row_i % 3 - 1;
                // same group: forward half only -- the rows at z + 1 (all dy), the row
                // (y + 1, z) and the cell (x + 1, y, z) of the own row.  One cell along z
                // (a dropped axis): the rows of the own plane only
                bool use = (!HALF || dz == 1 || (dz == 0 && dy >= 0)) && (ncz > 1 || dz == 0);
                int xa, xb;                          // cells [xa, xb] of the row
                const int row = (wrap(cz + dz, ncz) * ncy + wrap(cy + dy, ncy)) * ncx;
                if (HALF && dz == 0 && dy == 0) {
                    xa = xb = wrap(cx + 1, ncx);
                    use = (r & 1) == 0;
                } else if ((r & 1) == 0) {
                    xa = max(cx - 1, 0); xb = min(cx + 1, ncx - 1);
                } else {
                    const int xw = (cx == 0) ? ncx - 1 : (cx == ncx - 1 ? 0 : -1);
                    use = use && xw >= 0;
                    xa = xb = max(xw, 0);
                }
                if (use) {
                    pb = st2 + row + xa;
                    pe = st2 + row + xb + 1;
                }
            }
            b = __ldg(pb);
            e = __ldg(pe);
        };
        // Stage 2: lays the runs out in buffer `slot` and starts their copy.  Returns
        // (warp-uniform) n_i, total and the mode: 0 nothing to do, 1 buffered (copy in
        // flight), 2 list longer than the buffer (copied and computed in segments), 3 cell
        // too crowded for that as well (handed to the fp64 kernel).
        auto launch = [&](int slot, int b, int e, int &n_i, int &total) -> int {
            const int len = e - b;
            int pre = len;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int v = __shfl_up_sync(0xffffffffu, pre, o);
                if (lane >= o) pre += v;
            }
            total = __shfl_sync(0xffffffffu, pre, 31);
            pre -= len;
            n_i = __shfl_sync(0xffffffffu, len, 0);
            if (n_i == 0 || (!HALF && total == n_i)) return 0;
            if (total > cap) {
                if (n_i > cap - 64) return 3;
                wrng[slot * 32 + lane] = make_int2(b, len);   // the segments walk the runs
                __syncwarp();
                return 2;
            }
            const unsigned bar = bar32 + 8u * slot;
            if (lane == 0) cp_mbar_expect(bar, (unsigned)total * 16u);
            __syncwarp();
            if (len > 0)
                cp_bulk_g2s(wbuf32 + 16u * (unsigned)(slot * bufw + pre),
                            (lane == 0 ? P.s1 + (int64_t)frame * P.n1
                                       : P.s2 + (int64_t)frame * P.n2) + b,
                            (unsigned)len * 16u, bar);
            return 1;
        };
        // Mode 2: the next segment of an over-long candidate list into buffer `slot`
        // (the cell's own particles first), synchronously.  (r, o): run and offset to
        // continue from.  Returns the number of candidates copied to buf[n_i ..).
        auto fill_segment = [&](int slot, int n_i, int &r, int &o, bool first) -> int {
            const unsigned bar = bar32 + 8u * slot;
            const int room = cap - n_i;
            int filled = 0, rr = r, oo = o;
            while (rr < kCpRanges && filled < room) {      // what fits (warp-uniform)
                const int take = min(wrng[slot * 32 + rr].y - oo, room - filled);
                filled += take;
                oo += take;
                if (oo == wrng[slot * 32 + rr].y) { ++rr; oo = 0; }
            }
            if (lane == 0) {
                cp_mbar_expect(bar, (unsigned)(filled + (first ? n_i : 0)) * 16u);
                if (first)
                    cp_bulk_g2s(wbuf32 + 16u * (unsigned)(slot * bufw),
                                P.s1 + (int64_t)frame * P.n1 + wrng[slot * 32].x,
                                (unsigned)n_i * 16u, bar);
                int at = n_i, q = r, qo = o, left = filled;
                while (left > 0) {
                    const int2 rg = wrng[slot * 32 + q];
                    const int take = min(rg.y - qo, left);
                    if (take > 0)
                        cp_bulk_g2s(wbuf32 + 16u * (unsigned)(slot * bufw + at),
                                    P.s2 + (int64_t)frame * P.n2 + rg.x + qo,
                                    (unsigned)take * 16u, bar);
                    at += take; left -= take; qo += take;
                    if (qo == rg.y) { ++q; qo = 0; }
                }
            }
            r = rr; o = oo;
            __syncwarp();
            return filled;
        };

        // All pairs of the cell's particles buf[0 .. n_i) with the candidates buf[n_i .. je)
        // (weight 2 when the groups coincide: the half stencil stands for both orders) and,
        // if do_self, with each other (ordered pairs, weight 1, a particle never with itself).
        auto compute = [&](int slot, int n_i, int je, bool do_self) {
            const float4 *buf = wbuf + slot * bufw;
            const int total = je;
            // chunks of at most 8 * IPT particles (nearly always one)
            int cs = n_i;
            if (n_i > 8 * IPT) {
                const int n_chunks = (n_i + 8 * IPT - 1) / (8 * IPT);
                cs = (n_i + n_chunks - 1) / n_chunks;
            }
            for (int off = 0; off < n_i; off += cs) {
                const int cn = min(cs, n_i - off);
                // ni <= 8 lanes hold the chunk; lane / ni without an integer division
                // ((lane + 1/2) / ni is at least 1/16 away from every integer)
                const int ni = (cn + IPT - 1) / IPT;
                const float rni = __frcp_rn((float)ni);
                const int ways = (int)(32.5f * rni);
                const float rways = __frcp_rn((float)ways);
                const int way = (int)(((float)lane + 0.5f) * rni), il = lane - way * ni;
                const bool lane_ok = way < ways;
                const int ipos0 = off + il * IPT;
                // the lane's particles: negated coordinates packed in pairs (the operands of
                // the f32x2 arithmetic), exclusion ids, validity
                f32x2 nx[IPT / 2], ny[IPT / 2], nz[IPT / 2];
                int gi[IPT];
                unsigned vmask = 0;                   // bit k: particle k exists
                {
                    float4 a[IPT];
#pragma unroll
                    for (int k = 0; k < IPT; ++k) {
                        if (lane_ok && ipos0 + k < off + cn) vmask |= 1u << k;
                        a[k] = buf[min(ipos0 + k, n_i - 1)];
                        gi[k] = __float_as_int(a[k].w);
                    }
#pragma unroll
                    for (int ip = 0; ip < IPT / 2; ++ip) {
                        // negated by flipping the sign bits with a mask the compiler cannot
                        // see through (a kernel parameter): the result is a fresh aligned
                        // register pair.  Packed from the halves of two LDS.128 quads,
                        // ptxas would re-assemble the pair with two moves at every use.
                        nx[ip] = pk2(a[2 * ip].x, a[2 * ip + 1].x) ^ P.sign2;
                        ny[ip] = pk2(a[2 * ip].y, a[2 * ip + 1].y) ^ P.sign2;
                        nz[ip] = pk2(a[2 * ip].z, a[2 * ip + 1].z) ^ P.sign2;
                    }
                }

                // the packed fp32 arithmetic of one candidate against the lane's particles
                auto eval_row = [&](const float4 &pj, unsigned *uu) {
#pragma unroll
                    for (int ip = 0; ip < IPT / 2; ++ip)
                        filter_eval2<LOWER>(nx[ip], ny[ip], nz[ip], pk2(pj.x, pj.x),
                                            pk2(pj.y, pj.y), pk2(pj.z, pj.z), ff, scale, offm,
                                            fc.cbits, uu[2 * ip], uu[2 * ip + 1]);
                };
                // histogram updates of one row (wk: weight per particle, 0 = absent);
                // returns the smallest fraction of the row's bin coordinates
                auto hist_row = [&](const float4 &pj, const unsigned *uu, int jpos,
                                    const unsigned *wk, auto self_tag) -> unsigned {
                    constexpr bool SELF = decltype(self_tag)::value;
                    unsigned vmin = 0xffffffffu;
#pragma unroll
                    for (int k = 0; k < IPT; ++k) {
                        const unsigned u = uu[k];
                        unsigned w = min(u >> shift, trash_w);
                        if (EXCL && gi[k] == __float_as_int(pj.w)) w = trash_w;
                        if (SELF && jpos == ipos0 + k) {
                            // a particle with itself: never counted here, never uncertain
                            w = trash_w;
                        } else {
                            vmin = min(vmin, u & fmask);
                        }
                        red_shared_hot(hbase + (w << 2), wk[k]);
                        if (AUDIT && wk[k] != 0u && !(SELF && jpos == ipos0 + k)) {
                            const bool unc = (u & fmask) < ff.wlim, in = u < span_l;
                            const float4 a = buf[ipos0 + k];
                            const double d2 = pair_d2(a.x, a.y, a.z, pj, P.boxes[frame]);
                            const int slot_e = slot_search(d2, sT, n_bins);
                            const unsigned fs = in ? ((LOWER ? u : u - fc.cbits) >> fc.k)
                                                   : (unsigned)(n_bins + 1);
                            const bool counted = slot_e >= 1 && slot_e <= n_bins;
                            if (in && unc) ++audit_unc;
                            if (!(in && unc) && (unsigned)slot_e != fs &&
                                (counted || (fs >= 1u && fs <= (unsigned)n_bins)))
                                ++audit_bad;
                        }
                    }
                    return vmin;
                };
                // a row with an uncertain pair: remember it (re-evaluated after the pass), or
                // re-evaluate on the spot when the list is full
                auto push_row = [&](const unsigned *uu, int jpos, unsigned weight) {
                    // only pairs inside the histogram range can change a count (5 of 6
                    // candidates of a cut-off run lie beyond it)
                    bool any = false;
#pragma unroll
                    for (int k = 0; k < IPT; ++k)
                        any = any || ((uu[k] & fmask) < ff.wlim && uu[k] < span_l);
                    if (!any) return;
                    const unsigned idx = atomicAdd(wcount, 1u);
                    if (idx < (unsigned)kCpListCap) {
                        wlist[idx] = ((unsigned)lane << 16) | (unsigned)jpos;
                    } else {
                        cp_fix<EXCL, LOWER, IPT>(P, frame, buf + ipos0,
                                                 min(IPT, off + cn - ipos0), buf + jpos, weight,
                                                 sT, hist32);
                        ++n_inline;
                    }
                };
                // candidates buf[jb .. jb + cnt): lane (way, il) takes jb + way, jb + way +
                // ways, ...; two rows per iteration, the next two fetched ahead (rows past
                // the list are clamped to its last entry and carry weight 0)
                auto run_list = [&](int jb, int cnt, unsigned weight, auto self_tag) {
                    if (cnt <= 0) return;
                    // cnt / ways without an integer division (cnt <= 1024, ways <= 32:
                    // (cnt + 1/2) / ways stays 1/64 away from every integer)
                    const int full = (int)(((float)cnt + 0.5f) * rways), rem = cnt - full * ways;
                    const int jmax = jb + cnt - 1;
                    unsigned wi[IPT];
#pragma unroll
                    for (int k = 0; k < IPT; ++k) {
                        wi[k] = ((vmask >> k) & 1u) ? weight : 0u;
                        // keep the weights in registers (as predicates they cost a SEL per pair)
                        asm volatile("" : "+r"(wi[k]));
                    }
                    int j = jb + (lane_ok ? way : 0);
                    float4 r0 = buf[min(j, jmax)], r1 = buf[min(j + ways, jmax)];
                    int t = 0;
#pragma unroll 1
                    for (; t + 2 <= full; t += 2) {
                        const float4 a0 = r0, a1 = r1;
                        r0 = buf[min(j + 2 * ways, jmax)];
                        r1 = buf[min(j + 3 * ways, jmax)];
                        unsigned u0[IPT], u1[IPT];
                        eval_row(a0, u0);
                        eval_row(a1, u1);
                        const unsigned v0 = hist_row(a0, u0, j, wi, self_tag);
                        const unsigned v1 = hist_row(a1, u1, j + ways, wi, self_tag);
                        if (min(v0, v1) < ff.wlim && lane_ok) {
                            if (v0 < ff.wlim) push_row(u0, j, weight);
                            if (v1 < ff.wlim) push_row(u1, j + ways, weight);
                        }
                        j += 2 * ways;
                    }
                    // at most one more full row and the partial row (rows that do not exist
                    // for this lane carry weight 0)
                    const int left = (full - t) + (rem ? 1 : 0);      // 0, 1 or 2 rows
                    if (left > 0) {
                        unsigned w0[IPT];
                        const bool ok0 = lane_ok && (t < full || way < rem);
#pragma unroll
                        for (int k = 0; k < IPT; ++k) w0[k] = ok0 ? wi[k] : 0u;
                        unsigned u0[IPT];
                        eval_row(r0, u0);
                        const unsigned v0 = hist_row(r0, u0, j, w0, self_tag);
                        if (v0 < ff.wlim && ok0) push_row(u0, j, weight);
                    }
                    if (left > 1) {
                        unsigned w1[IPT];
                        const bool ok1 = lane_ok && way < rem;
#pragma unroll
                        for (int k = 0; k < IPT; ++k) w1[k] = ok1 ? wi[k] : 0u;
                        unsigned u1[IPT];
                        eval_row(r1, u1);
                        const unsigned v1 = hist_row(r1, u1, j + ways, w1, self_tag);
                        if (v1 < ff.wlim && ok1) push_row(u1, j + ways, weight);
                    }
                };

                const unsigned w_fwd = HALF ? 2u : 1u;
                if (HALF && do_self) run_list(0, n_i, 1u, std::integral_constant<bool, true>());
                run_list(n_i, total - n_i, w_fwd, std::integral_constant<bool, false>());
                __syncwarp();

                // drain: the uncertain rows of this pass, re-evaluated from the buffer
                const unsigned n_push = *wcount;
                if (n_push) {
                    const unsigned n_list = min(n_push, (unsigned)kCpListCap);
                    for (unsigned e = lane; e < n_list; e += 32) {
                        const unsigned entry = wlist[e];
                        const int src = (int)(entry >> 16), jpos = (int)(entry & 0xffffu);
                        const int e_i0 =
                            off + (src - (int)(((float)src + 0.5f) * rni) * ni) * IPT;
                        cp_fix<EXCL, LOWER, IPT>(P, frame, buf + e_i0, min(IPT, off + cn - e_i0),
                                                 buf + jpos, jpos < n_i ? 1u : w_fwd, sT, hist32);
                    }
                    n_deferred += n_list;
                    __syncwarp();
                    if (lane == 0) *wcount = 0;
                    __syncwarp();
                }
                // the per-warp u32 words must not wrap: hand them over in time
                acc_w += (unsigned)cn * (unsigned)total * 2u;      // each term < 2^31
                if (acc_w >= (1u << 31)) {
                    for (int k = lane; k < n_bins; k += 32) {
                        unsigned sum = 0;
                        for (int q = 0; q < (1 << fc.sb); ++q) {
                            unsigned *w = sH + warp * hwords + ((k + 1) << fc.sb) + q;
                            sum += *w;
                            *w = 0;
                        }
                        if (sum) atomicAdd(&P.counts[k], (unsigned long long)sum);
                    }
                    acc_w = 0;
                    __syncwarp();
                }
            }
        };

        // software pipeline over the cells of the item: run bounds of cell k + 2 (loads),
        // layout + copy of cell k + 1, pairs of cell k (one call site each)
        int px = c0 % ncx, py = (c0 / ncx) % ncy, pz = c0 / (ncx * ncy);   // cell being planned
        int pb = 0, pe = 0;                    // planned run of this lane, one cell ahead
        int ni_c = 0, tot_c = 0, mode_c = 0;
        for (int cell = c0 - 2; cell < c1; ++cell) {
            int nb = 0, ne = 0;
            if (cell + 2 < c1) {
                plan(cell + 2, px, py, pz, nb, ne);
                if (++px == ncx) { px = 0; if (++py == ncy) { py = 0; ++pz; } }
            }
            int ni_n = 0, tot_n = 0, mode_n = 0;
            const int slot = (cell - c0) & 1;
            if (cell + 1 >= c0 && cell + 1 < c1) mode_n = launch(slot ^ 1, pb, pe, ni_n, tot_n);
            pb = nb; pe = ne;
            if (mode_c == 1 || mode_c == 2) {
                int r = HALF ? 1 : 1, o = 0;   // run 0 is the own cell (copied with segment 1)
                bool first = true;
                for (;;) {
                    int je = tot_c;
                    if (mode_c == 2) je = ni_c + fill_segment(slot, ni_c, r, o, first);
                    cp_mbar_wait(bar32 + 8u * slot, (phase >> slot) & 1u);
                    phase ^= 1u << slot;
                    compute(slot, ni_c, je, first);
                    first = false;
                    if (mode_c == 1 || r >= kCpRanges) break;
                }
            } else if (mode_c == 3) {
                // more particles in one cell than a warp should take on: the fp64 kernel
                // (one thread per particle) does this cell's pairs
                if (lane == 0) {
                    P.cellflag[(int64_t)frame * P.cstride + cell] = 1;
                    atomicAdd(&P.nflag[frame], 1);
                }
            }
            if (mode_c != 0 && mode_c != 3 && lane == 0) {
                my_evals += (unsigned long long)ni_c *
                            (unsigned long long)(HALF ? tot_c : tot_c - ni_c);
                if (count_self)
                    red_shared(hist32 + 4u * ((unsigned)slot_zero << fc.sb), (unsigned)ni_c);
            }
            ni_c = ni_n; tot_c = tot_n; mode_c = mode_n;
        }
    }
    __syncthreads();

    // merge into the global int64 histogram (sum of the warps' words modulo 2^32 first)
    for (int k = tid; k < n_bins; k += kCpThreads) {
        unsigned sum = 0;
        for (int w = 0; w < kCpWarps; ++w)
            for (int q = 0; q < (1 << fc.sb); ++q)
                sum += sH[w * hwords + ((k + 1) << fc.sb) + q];
        if (sum) atomicAdd(&P.counts[k], (unsigned long long)sum);
    }
    if (lane == 0 && my_evals) atomicAdd(P.evals, my_evals);
    n_inline = __reduce_add_sync(0xffffffffu, n_inline);
    if (lane == 0) {
        // n_deferred is warp-uniform (every lane added n_list), n_inline is per lane
        if (n_deferred) atomicAdd(&P.fstats[0], (unsigned long long)n_deferred);
        if (n_inline) atomicAdd(&P.fstats[1], (unsigned long long)n_inline);
    }
    if (AUDIT) {
        if (audit_bad) atomicAdd(&P.fstats[2], audit_bad);
        if (audit_unc) atomicAdd(&P.fstats[3], audit_unc);
    }
}

template <bool HALF, bool EXCL, bool LOWER, bool AUDIT, int IPT>
int launch_cellpair_t(mdh_ctx *c, const CellPairParams &P)
{
    const size_t smem = cp_smem_bytes(P.n_bins, P.fc.sb, P.cap);
    auto kern = rdf_cellpair_kernel<HALF, EXCL, LOWER, AUDIT, IPT>;
    // attribute and occupancy are looked up once per shared-memory size and device (these
    // calls cost more host time than the launch itself)
    static thread_local size_t cached_smem = 0;
    static thread_local int cached_dev = -1, cached_per_sm = 0;
    if (cached_smem != smem || cached_dev != c->device) {
        MDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      (int)smem));
        MDH_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cached_per_sm, kern, kCpThreads,
                                                               smem));
        cached_smem = smem;
        cached_dev = c->device;
    }
    const int per_sm = cached_per_sm;
    MDH_REQUIRE(per_sm >= 1, MDH_EINVAL, "rdf: cell-pair kernel does not fit on an SM");
    const int items = (P.max_ncell + P.chunk_cells - 1) / P.chunk_cells * P.n_frames;
    const int blocks = std::max(1, std::min(c->sm_count * per_sm, (items + kCpWarps - 1) / kCpWarps));
    kern<<<blocks, kCpThreads, smem, c->stream>>>(P);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    return MDH_OK;
}

template <bool HALF, bool EXCL>
int launch_cellpair_he(mdh_ctx *c, const CellPairParams &P, bool audit, int ipt)
{
    if (audit)
        return P.fc.lower ? launch_cellpair_t<HALF, EXCL, true, true, 4>(c, P)
                          : launch_cellpair_t<HALF, EXCL, false, true, 4>(c, P);
    if (ipt == 2)
        return P.fc.lower ? launch_cellpair_t<HALF, EXCL, true, false, 2>(c, P)
                          : launch_cellpair_t<HALF, EXCL, false, false, 2>(c, P);
    return P.fc.lower ? launch_cellpair_t<HALF, EXCL, true, false, 4>(c, P)
                      : launch_cellpair_t<HALF, EXCL, false, false, 4>(c, P);
}

int launch_cellpair(mdh_ctx *c, const CellPairParams &P, bool half, bool excl, bool audit,
                    int ipt)
{
    if (half)
        return excl ? launch_cellpair_he<true, true>(c, P, audit, ipt)
                    : launch_cellpair_he<true, false>(c, P, audit, ipt);
    return excl ? launch_cellpair_he<false, true>(c, P, audit, ipt)
                : launch_cellpair_he<false, false>(c, P, audit, ipt);
}

// Largest number of sub-bins (log2) <= sb_max whose histograms leave room for two
// resident blocks; -1 if not even sb = 0 fits a single block.
int cellpair_sub_bins(int n_bins, int sb_max, int cap)
{
    for (int sb = sb_max; sb >= 0; --sb)
        if (cp_smem_bytes(n_bins, sb, cap) <= (size_t)(224 * 1024 / MDH_CP_BLOCKS)) return sb;
    return cp_smem_bytes(n_bins, 0, cap) <= 224 * 1024 ? 0 : -1;
}

}  // namespace

// Grid of the orthorhombic cell list for one frame, per PHYSICAL axis: cells of edge at least
// r_cut = r_hi * (1 + 1e-5), at least 3 and at most 160 per kept axis, a single cell along a
// dropped axis (drop_axis 0/1/2, or -1), and no more cells than keep about 2 particles per
// cell (n_max: the larger group) while every kept axis has more than 3.  Returns the first
// kept axis on which fewer than 3 cells fit (nc is then incomplete), or -1.
int rdf_ortho_grid_plan(const double box[3], double r_hi, int64_t n_max, int drop_axis,
                        int nc[3])
{
    const double r_cut = r_hi * 1.00001;
    double ncell = 1;
    for (int k = 0; k < 3; ++k) {
        if (k == drop_axis) {
            nc[k] = 1;
            continue;
        }
        const double fit = std::floor(box[k] / r_cut);
        if (!(fit >= 3.0)) return k;
        nc[k] = (int)std::min(fit, 160.0);
        ncell *= nc[k];
    }
    // keep at least ~2 particles per cell on average
    const double want = std::max(drop_axis < 0 ? 27.0 : 9.0, (double)n_max / 2.0);
    while (ncell > want) {
        int kmax = 0;
        for (int k = 1; k < 3; ++k) if (nc[k] > nc[kmax]) kmax = k;
        if (nc[kmax] <= 3) break;
        ncell = ncell / nc[kmax] * (nc[kmax] - 1);
        nc[kmax]--;
    }
    return -1;
}

// Device layout of the cell-list scratch (RdfState::cell):
//   cell[0] CellGrid[F]            cell[1] int cnt[2][G][cstride] | unsigned ext[2][G][6] | work
//   cell[2] int start[2][G][cstride]   cell[3] int2 keyrank[G][n1]   cell[4] float4 sorted1[G][n1]
//   cell[7] int2 keyrank[G][n2]    cell[8] float4 sorted2[G][n2]     cell[9] evals (+ selfcheck word)
// G = frames per group.
int rdf_cells_accumulate(mdh_ctx *c, const float *raw1, int64_t stride1, const float *raw2,
                         int64_t stride2, int f0, int n_frames, bool use_filter, double sqrt_err)
{
    RdfState &R = c->rdf;
    MDH_REQUIRE(R.n1 <= (1ll << 25) && R.n2 <= (1ll << 25), MDH_EINVAL,
                "rdf: cell-list mode takes at most 2^25 particles per group");
    // grid axis k <- physical axis: a dropped axis goes last (see CellGrid)
    static const int kAxes[4][3] = {{0, 1, 2}, {1, 2, 0}, {0, 2, 1}, {0, 1, 2}};
    const int *axes = kAxes[R.drop_axis + 1];
    const bool flat = R.drop_axis >= 0;
    std::vector<CellGrid> grids(n_frames);
    int ncell_max = 0;
    for (int f = 0; f < n_frames; ++f) {
        CellGrid &g = grids[f];
        int nc[3];
        const int short_axis = rdf_ortho_grid_plan(R.h_boxes[f0 + f].box, sqrt(R.thr_hi),
                                                   std::max(R.n1, R.n2), R.drop_axis, nc);
        MDH_REQUIRE(short_axis < 0, MDH_EINVAL,
                    "rdf: cell-list mode needs box edge >= 3*r_max (frame %d axis %d)", f,
                    short_axis);
        for (int k = 0; k < 3; ++k) {
            g.axis[k] = axes[k];
            g.box[k] = R.h_boxes[f0 + f].box[axes[k]];
            g.nc[k] = nc[axes[k]];
            g.inv_w[k] = g.nc[k] / g.box[k];
        }
        g.ncell = g.nc[0] * g.nc[1] * g.nc[2];
        ncell_max = std::max(ncell_max, g.ncell);
    }
    MDH_TRACE("cells: %d frames, %d cells", n_frames, ncell_max);
    const int cstride = ncell_max + 1;
    DevBuf &d_grids = R.cell[0];
    if (int rc = d_grids.reserve(sizeof(CellGrid) * n_frames)) return rc;
    // pageable source: the runtime stages it before returning, so the local vector
    // may go out of scope while the copy is still queued
    MDH_CUDA(cudaMemcpyAsync(d_grids.p, grids.data(), sizeof(CellGrid) * n_frames,
                             cudaMemcpyHostToDevice, c->stream));

    MDH_TRACE("cells: grids uploaded");
    // frames per group: the sorted copies, the (cell, rank) words and the raw floats of a
    // group should stay in L2 between the passes (R.cells_ws_mb, default 48 MB)
    const int n_groups = R.same ? 1 : 2;
    const double per_frame = 36.0 * (double)(R.n1 + (R.same ? 0 : R.n2)) + 8.0 * cstride * n_groups;
    int G = (int)std::max(1.0, std::min(64.0, floor(R.cells_ws_mb * 1048576.0 / per_frame)));
    G = std::min(G, n_frames);

    const size_t cnt_words = (size_t)2 * G * cstride;
    const size_t ext_off = cnt_words, work_off = ext_off + (size_t)2 * G * 6;
    const size_t nflag_off = work_off + 4, flag_off = nflag_off + G;
    const size_t reset_words = flag_off + (size_t)G * cstride;
    if (int rc = R.cell[1].reserve(sizeof(int) * reset_words)) return rc;
    if (int rc = R.cell[2].reserve(sizeof(int) * cnt_words)) return rc;
    if (int rc = R.cell[3].reserve(sizeof(int2) * (size_t)R.n1 * G)) return rc;
    if (int rc = R.cell[4].reserve(sizeof(float4) * (size_t)R.n1 * G)) return rc;
    if (!R.same) {
        if (int rc = R.cell[7].reserve(sizeof(int2) * (size_t)R.n2 * G)) return rc;
        if (int rc = R.cell[8].reserve(sizeof(float4) * (size_t)R.n2 * G)) return rc;
    }
    if (use_filter)
        if (int rc = R.filt.reserve(sizeof(FrameFilter) * G)) return rc;

    MDH_TRACE("cells: buffers reserved, groups of %d", G);
    int *d_cnt = R.cell[1].as<int>();
    unsigned *d_ext = R.cell[1].as<unsigned>() + ext_off;
    unsigned *d_work = R.cell[1].as<unsigned>() + work_off;
    int *d_nflag = R.cell[1].as<int>() + nflag_off, *d_cellflag = R.cell[1].as<int>() + flag_off;
    int *d_start = R.cell[2].as<int>();

    // candidates per cell the buffers are sized for: mean + 6 sigma (Poisson) + slack
    const double per_cell1 = (double)R.n1 / ncell_max, per_cell2 = (double)R.n2 / ncell_max;
    const double expect = per_cell1 + (flat ? (R.same ? 4.0 : 9.0) : (R.same ? 13.0 : 27.0)) *
                                          per_cell2;
    int cap = (int)(expect + 6.0 * sqrt(expect) + 24.0);
    cap = std::min(1024, std::max(96, (cap + 31) / 32 * 32));
    int sb_c = use_filter ? cellpair_sub_bins(R.n_bins, R.fc.sb, cap) : -1;
    while (use_filter && sb_c < 0 && cap > 96) {      // many bins: smaller buffers
        cap = std::max(96, cap / 2 / 32 * 32);
        sb_c = cellpair_sub_bins(R.n_bins, R.fc.sb, cap);
    }
    use_filter = use_filter && sb_c >= 0;

    const bool excl = R.excl1 > 0, fast = R.fast_bins;
    // MDH_TUNE="cdbg=1": device time of every stage, printed per call (tuning aid;
    // synchronises)
    std::vector<cudaEvent_t> dbg;
    auto mark = [&]() {
        if (!R.cells_debug) return;
        cudaEvent_t e;
        cudaEventCreate(&e);
        cudaEventRecord(e, c->stream);
        dbg.push_back(e);
    };
    for (int g0 = 0; g0 < n_frames; g0 += G) {
        const int ng = std::min(G, n_frames - g0);
        mark();
        // counters, extents and the work counter: one contiguous region, one zero fill
        MDH_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(int) * reset_words, c->stream));
        const CellGrid *gg = d_grids.as<CellGrid>() + g0;
        for (int grp = 0; grp < n_groups; ++grp) {
            const float *raw = (grp ? raw2 : raw1) + (int64_t)g0 * (grp ? stride2 : stride1);
            const int n = (int)(grp ? R.n2 : R.n1);
            dim3 grid((unsigned)std::min((n + 255) / 256, 4096), ng);
            cells_bin_kernel<<<grid, 256, 0, c->stream>>>(
                raw, grp ? stride2 : stride1, n, gg, d_cnt + (size_t)grp * G * cstride, cstride,
                R.cell[grp ? 7 : 3].as<int2>(), use_filter ? d_ext + (size_t)grp * G * 6 : nullptr,
                R.boxes.as<FrameBox>() + f0 + g0, R.drop_axis);
            MDH_CUDA(cudaGetLastError());
            c->launches++;
        }
        mark();
        ScanFilter F{};
        F.out = nullptr;
        if (use_filter) {
            F.boxes = R.boxes.as<FrameBox>() + f0 + g0;
            F.ext1 = d_ext;
            F.ext2 = R.same ? d_ext : d_ext + (size_t)G * 6;
            F.out = R.filt.as<FrameFilter>();
            F.prep = rdf_filter_prep(R, sqrt_err);
        }
        const size_t scan_smem = sizeof(int) * (kScanTile + kScanTile / 32);
        static thread_local int scan_attr_dev = -1;
        if (scan_attr_dev != c->device) {
            MDH_CUDA(cudaFuncSetAttribute(cells_scan_kernel<CellGrid>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize,
                                          (int)scan_smem));
            scan_attr_dev = c->device;
        }
        cells_scan_kernel<CellGrid><<<dim3(ng, n_groups), 1024, scan_smem, c->stream>>>(
            d_cnt, d_start, cstride, G, gg, F);
        MDH_CUDA(cudaGetLastError());
        c->launches++;
        mark();
        for (int grp = 0; grp < n_groups; ++grp) {
            const float *raw = (grp ? raw2 : raw1) + (int64_t)g0 * (grp ? stride2 : stride1);
            const int n = (int)(grp ? R.n2 : R.n1);
            dim3 grid((unsigned)std::min((n + 255) / 256, 4096), ng);
            cells_scatter_kernel<<<grid, 256, 0, c->stream>>>(
                raw, grp ? stride2 : stride1, n, grp ? R.excl2 : R.excl1,
                d_start + (size_t)grp * G * cstride, cstride, R.cell[grp ? 7 : 3].as<int2>(),
                R.cell[grp ? 8 : 4].as<float4>(), R.boxes.as<FrameBox>() + f0 + g0,
                R.drop_axis);
            MDH_CUDA(cudaGetLastError());
            c->launches++;
        }

        mark();
        const float4 *s1 = R.cell[4].as<float4>();
        const float4 *s2 = R.same ? s1 : R.cell[8].as<float4>();
        const int *start1 = d_start, *start2 = R.same ? d_start : d_start + (size_t)G * cstride;
        if (use_filter) {
            CellPairParams Q;
            Q.s1 = s1; Q.s2 = s2;
            Q.n1 = (int)R.n1; Q.n2 = (int)R.n2;
            Q.start1 = start1; Q.start2 = start2;
            Q.cstride = cstride;
            Q.grids = gg;
            Q.boxes = R.boxes.as<FrameBox>() + f0 + g0;
            Q.filt = R.filt.as<FrameFilter>();
            Q.thr = R.thr.as<double>();
            Q.n_bins = R.n_bins;
            Q.guess = rdf_bin_guess(R);
            Q.fc = R.fc;
            Q.fc.sb = sb_c;
            Q.fast_bins = R.fast_bins ? 1 : 0;
            Q.counts = R.counts.as<unsigned long long>();
            Q.evals = R.cell[9].as<unsigned long long>();
            Q.fstats = R.fstats.as<unsigned long long>();
            Q.work = d_work;
            Q.cellflag = d_cellflag;
            Q.nflag = d_nflag;
            Q.n_frames = ng;
            Q.max_ncell = ncell_max;
            Q.chunk_cells = R.cells_chunk;
            Q.cap = cap;
            Q.sign2 = 0x8000000080000000ull;
            if (int rc = launch_cellpair(c, Q, R.same != 0, excl,
                                         R.filter_mode == MDH_FILTER_AUDIT, R.cells_ipt))
                return rc;
        }
        mark();
        // the fp64 kernel: every frame without the filter, else the frames it declined
        CellParams P;
        P.s1 = s1; P.s2 = s2;
        P.n1 = (int)R.n1; P.n2 = (int)R.n2;
        P.start2 = start2;
        P.cstride = cstride;
        P.grids = gg;
        P.boxes = R.boxes.as<FrameBox>() + f0 + g0;
        P.thr = R.thr.as<double>();
        P.n_bins = R.n_bins;
        P.guess = rdf_bin_guess(R);
        P.counts = R.counts.as<unsigned long long>();
        P.evals = R.cell[9].as<unsigned long long>();
        P.half = R.same;
        P.filt = use_filter ? R.filt.as<FrameFilter>() : nullptr;
        P.cellflag = d_cellflag;
        P.nflag = d_nflag;
        dim3 grid((unsigned)((R.n1 + kThreads - 1) / kThreads), (unsigned)ng);
        int rc;
        if (R.hist == MDH_HIST_LANE_PRIVATE) {
            if (excl)
                rc = fast ? launch_cells<MDH_HIST_LANE_PRIVATE, true, true>(c, P, grid)
                          : launch_cells<MDH_HIST_LANE_PRIVATE, true, false>(c, P, grid);
            else
                rc = fast ? launch_cells<MDH_HIST_LANE_PRIVATE, false, true>(c, P, grid)
                          : launch_cells<MDH_HIST_LANE_PRIVATE, false, false>(c, P, grid);
        } else if (excl) {
            rc = fast ? launch_cells<MDH_HIST_WARP_ATOMIC, true, true>(c, P, grid)
                      : launch_cells<MDH_HIST_WARP_ATOMIC, true, false>(c, P, grid);
        } else {
            rc = fast ? launch_cells<MDH_HIST_WARP_ATOMIC, false, true>(c, P, grid)
                      : launch_cells<MDH_HIST_WARP_ATOMIC, false, false>(c, P, grid);
        }
        if (rc) return rc;
        mark();
    }
    if (R.cells_debug && !dbg.empty()) {
        cudaStreamSynchronize(c->stream);
        double t[5] = {0, 0, 0, 0, 0};            // six marks, five stages per group
        for (size_t k = 0; k + 5 < dbg.size(); k += 6)
            for (int q = 0; q < 5; ++q) {
                float ms = 0;
                cudaEventElapsedTime(&ms, dbg[k + q], dbg[k + q + 1]);
                t[q] += ms;
            }
        float whole = 0;
        cudaEventElapsedTime(&whole, dbg.front(), dbg.back());
        fprintf(stderr, "cells: %d frames (groups of %d): reset+bin %.1f scan %.1f scatter %.1f "
                        "pair %.1f fp64 %.1f | whole %.1f us per frame\n", n_frames, G,
                1e3 * t[0] / n_frames, 1e3 * t[1] / n_frames, 1e3 * t[2] / n_frames,
                1e3 * t[3] / n_frames, 1e3 * t[4] / n_frames, 1e3 * whole / n_frames);
        for (cudaEvent_t e : dbg) cudaEventDestroy(e);
    }
    return MDH_OK;
}
