// rdf_filter.cu -- all-pairs histogram with an fp32 filter in front of the exact
// fp64 arithmetic (seam #1, /root/reference/src/mdhelper/analysis/structure.py:32-104).
//
// The counts are the reference's, bit for bit: a pair is binned from fp32 arithmetic
// only when a rigorous error bound proves that the reference's fp64 distance falls in
// the same bin; every other pair ("uncertain": within the bound of a bin edge, about
// 1 in 1,000 for the benchmark configurations) is re-evaluated with the exact
// arithmetic of rdf_device.cuh::pair_d2 and corrected.  The fp32 path costs ~15
// issue slots per pair (6.5 packed f32x2 instructions on the FMA pipe in the half-box
// form, 8 in the rint form, ~5 on the ALU pipe, one MUFU, one RED) instead of 21 FP64-pipe instructions plus conversions (46
// in total) -- it removes the FP64 pipe as the bound.
//
// fp32 evaluation (rdf_device.cuh::filter_eval2, two pairs per instruction), per axis
// one of two forms of the minimum image, chosen per frame (FrameFilter::halfbox):
//     df = xj - xi                      the reference's own float32 difference (exact copy)
//   half-box form, when every |df| of the frame is <= 1.5 box (h = box/2, exact):
//     e  = |df| - h                     FADD2 with an |x| operand
//     m  = |e| - h                      FADD2; |m| is the minimum-image distance
//   rint form, all other frames (unwrapped trajectories):
//     t  = fma(df, inv, 1.5*2^23)       -> 1.5*2^23 + rint(df * inv), one rounding
//     r  = t - 1.5*2^23                 exact
//     m  = fma(-box, r, df)             minimum image, one rounding
// then d2 = mx*mx + my*my + mz*mz (fma chain), s = sqrt.approx(d2), and the bin
// coordinate as a fixed-point number in the mantissa of one more fma:
//     bits(fma(s, scale, 1.5*2^(23-k) + off)) - bits(1.5*2^(23-k)) = slot * 2^k + frac
// slot = bin + 1 + lo (filter_plan: lo = ceil(r_lo * scale) when the histogram is sized
// for the unclamped body, so that no coordinate is negative; else lo = 0).  The slots
// outside [lo + 1, lo + n_bins] are scratch words, never read.  The coordinate is
// additionally shifted up by the window half-width m, so that "within m of a bin
// edge" reads "fraction bits <= 2m" (one AND + one MIN per pair on the ALU pipe).
//
// Three bodies, chosen per frame (one branch per block): half-box unclamped -- the block
// histogram has a word for every slot the frame's fp32 arithmetic can reach
// (rdf_device.cuh::filter_reach; cfg2: 353 slots), so a pair's word address is one SHF
// and one LOP3 --, half-box clamped and rint clamped (one more MIN sends everything
// beyond the histogram to its last slot).
//
// Error bound (rdf_filter_prepare_kernel, per frame, in bin units) -- see DESIGN.md
// section 4.1b for the derivation.  With eps_b = |box*inv - 1| (the reference's
// float32 inverse box makes its minimum image differ from df - box*r by eps_b*df),
// D_k the largest |df| of the frame (coordinate extents from the pack kernel):
//     | |m_f| - |m_ref| |  <=  a_k = 2^-24 (box_k/2 + eps_b D_k + 2^-24 D_k) + eps_b D_k
//                                (half-box form: 2^-24 box_k/2 when D_k <= box_k, else
//                                 2^-23 box_k/2, + eps_b D_k; at most one FADD rounds)
//     | |m_f|_2 - d_ref |  <=  |a|_2                          (reverse triangle inequality)
//     fp32 sum of squares: relative 3*2^-24 on d2 -> 1.5*2^-24 on d
//     sqrt.approx: relative error measured exhaustively at start-up (<= 2^-22 required)
//     scale rounding 2^-24, off rounding 2^-(k+1), fma rounding 2^-(k+1)
// The window half-width is ceil(1.25 * bound * 2^k) + 1 units of 2^-k.  Frames whose
// bound is not small against a bin (coordinates many boxes away, non-finite values)
// are left to the exact kernel of rdf.cu.

#include <algorithm>
#include <type_traits>

#include "rdf_device.cuh"

using namespace rdfdev;

namespace {

#ifndef MDH_FILTER_ROWS
#define MDH_FILTER_ROWS 2
#endif

constexpr int kListCap = 3072;           // deferred entries per block and tile
constexpr int kTilePad = 4;              // rows behind each j-tile: the main loop fetches
                                         // rows up to 4 ahead without a bound

// shared memory of a block: histogram (hslots slots x 2^cb columns, first, so that its
// address is the kernel's shared-memory base + an offset), thresholds, two j-tiles, the
// deferred list
__host__ __device__ inline size_t filter_hist_bytes(int hslots, int cb)
{
    return align16(sizeof(unsigned) * ((size_t)hslots << cb));
}
template <int IPT>
__host__ __device__ inline size_t filter_smem_bytes(int n_bins, int hslots, int cb)
{
    return filter_hist_bytes(hslots, cb) + align16(sizeof(double) * (n_bins + 1)) +
           2 * (kThreads * IPT + kTilePad) * sizeof(float4) + sizeof(unsigned) * (kListCap + 4);
}

// Exact re-evaluation of the IPT pairs behind one deferred entry (thread te of the
// block, tile row jj): every pair the main loop saw as uncertain has been added to
// the slot the fp32 arithmetic suggested -- unclamped: its coordinate's slot, which
// lies below fc.hslots --; move it if the fp64 arithmetic disagrees.  CX: the tile pair is
// x-clean with the shift of form (filter_cleanx_form): the i-coordinates take the same
// shift as in the main loop, and the j-row's x is restored for the fp64 arithmetic.
template <bool EXCL, bool LOWER, int IPT, bool HALF, bool CX = false>
__device__ __noinline__ void filter_fix(const PairParams &P, int frame, int it, unsigned entry,
                                        const float4 *tile, const double *sT, unsigned hist32,
                                        unsigned weight, int form = 0)
{
    constexpr int TILE = kThreads * IPT;
    const FrameFilter ff = P.filt[frame];
    const FrameBox fb = P.boxes[frame];
    const FilterConst fc = P.fc;
    const int te = (int)(entry >> 16), jj = (int)(entry & 0xffffu);
    const float4 pj = tile[jj];
    const float4 *f1 = P.p1 + (int64_t)frame * P.pad1;
    const unsigned span_l = LOWER ? fc.span : fc.cbits + fc.span;
    const float L = -ff.nbox[0];
    float4 pjx = pj;                      // the j-row as the reference sees it
    if (CX && form == 2) pjx.x = __fadd_rn(pj.x, L);
    for (int ip = 0; ip < IPT; ip += 2) {
        // the same particle pairing as the main loop (rows past the end of the group
        // repeat the last particle there; they carry weight 0 and are skipped here)
        const int i0 = it * TILE + ip * kThreads + te, i1 = i0 + kThreads;
        const float4 a0 = f1[min(i0, P.n1 - 1)], a1 = f1[min(i1, P.n1 - 1)];
        f32x2 ax = pk2(-a0.x, -a1.x);
        if (CX && form == 3) ax = add2(ax, pk2(L, L));
        unsigned uu[2];
        filter_eval2<LOWER, HALF, CX>(ax, pk2(-a0.y, -a1.y), pk2(-a0.z, -a1.z),
                                      pk2(pj.x, pj.x), pk2(pj.y, pj.y), pk2(pj.z, pj.z), ff,
                                      fc.scale, ff.offm, fc.cbits, uu[0], uu[1]);
        for (int h = 0; h < 2; ++h) {
            const int i = h ? i1 : i0;
            const float4 a = h ? a1 : a0;
            const unsigned u = uu[h];
            if (i >= P.n1) continue;
            if (!(u < span_l)) continue;
            if (!((u & ((1u << fc.k) - 1u)) < ff.wlim)) continue;
            if (EXCL && __float_as_int(a.w) == __float_as_int(pj.w)) continue;
            // the main loop added the pair to (slot it saw, column of thread te's lane);
            // u < span_l: that slot is a word of the histogram, below fc.hslots
            const unsigned seen = (LOWER ? u : u - fc.cbits) >> fc.k;
            const unsigned col = (unsigned)te & ((1u << fc.cb) - 1u);
            const double d2 = pair_d2(a.x, a.y, a.z, pjx, fb);
            const int slot = (P.fast_bins ? slot_fast(d2, sT, P.n_bins, P.guess)
                                          : slot_search(d2, sT, P.n_bins)) + fc.lo;
            if (seen == (unsigned)slot) continue;
            // slots outside [lo + 1, lo + n_bins] are scratch words, so no range test is
            // needed (a count may move between bin n_bins - 1 and a slot above lo + n_bins)
            red_shared(hist32 + 4u * ((seen << fc.cb) + col), 0u - weight);
            red_shared(hist32 + 4u * (((unsigned)slot << fc.cb) + col), weight);
        }
    }
}

// One block of rdf_filter_kernel with the frame's form of the minimum image; CLAMP =
// false for frames whose every reachable slot is a histogram word (FrameFilter::unclamped).
template <bool EXCL, bool LOWER, bool AUDIT, int IPT, bool HALF, bool CLAMP>
__device__ __forceinline__ void filter_block(const PairParams &P, const FrameFilter &ff)
{
    constexpr int TILE = kThreads * IPT;
    constexpr int TSTRIDE = TILE + kTilePad;
    const int frame = blockIdx.y;

    extern __shared__ __align__(16) unsigned char smem[];
    const int n_bins = P.n_bins;
    const FilterConst fc = P.fc;
    // ONE histogram per block: hslots slots x 2^cb columns, a lane updates column lane mod
    // 2^cb -- with 32 columns the 32 updates of a warp instruction fall in 32 different
    // banks whatever the bins are (per-warp histograms with sub-bins took 3.8 wavefronts
    // per instruction on random bins).  Only slots lo + 1 .. lo + n_bins are read; the
    // others take the pairs outside the range.
    const int hwords = fc.hslots << fc.cb;
    unsigned *sH = reinterpret_cast<unsigned *>(smem);
    double *sT = reinterpret_cast<double *>(smem + filter_hist_bytes(fc.hslots, fc.cb));
    float4 *sJ = reinterpret_cast<float4 *>(reinterpret_cast<unsigned char *>(sT) +
                                            align16(sizeof(double) * (n_bins + 1)));
    unsigned *sList = reinterpret_cast<unsigned *>(sJ + 2 * TSTRIDE);
    unsigned *sCount = sList + kListCap;

    const int tid = threadIdx.x, lane = tid & 31;
    const int it = blockIdx.x / P.n_jchunks;
    const int jc = blockIdx.x - it * P.n_jchunks;
    int jt0 = jc * P.jtiles_per_chunk;
    const int jt1 = min(P.n_jtiles, jt0 + P.jtiles_per_chunk);
    if (P.same) jt0 = max(jt0, it);       // upper triangle of tile pairs
    if (jt0 >= jt1) return;

    for (int k = tid; k <= n_bins; k += kThreads) sT[k] = P.thr[k];
    for (int k = tid; k < hwords; k += kThreads) sH[k] = 0;
    if (tid == 0) *sCount = 0;

    const float4 *f1 = P.p1 + (int64_t)frame * P.pad1;
    const float4 *f2 = P.same ? f1 : P.p2 + (int64_t)frame * P.pad2;

    static_assert(IPT % 2 == 0, "particles are processed in packed pairs");
    float xi[IPT], yi[IPT], zi[IPT];
    int gi[IPT];
    // rows of this thread below the end of the group: ii * kThreads < nv (one register
    // across the tile loop rather than one per row)
    const int nv = P.n1 - it * TILE - tid;
#pragma unroll
    for (int ii = 0; ii < IPT; ++ii) {
        const int i = it * TILE + ii * kThreads + tid;
        // rows past the end of the group repeat the last particle with weight 0
        const float4 a = f1[min(i, P.n1 - 1)];
        xi[ii] = a.x; yi[ii] = a.y; zi[ii] = a.z; gi[ii] = __float_as_int(a.w);
    }
    // negated coordinates of particle pairs (0,1), (2,3), ... for the packed arithmetic
    f32x2 nx[IPT / 2], ny[IPT / 2], nz[IPT / 2];
#pragma unroll
    for (int ip = 0; ip < IPT / 2; ++ip) {
        nx[ip] = pk2(-xi[2 * ip], -xi[2 * ip + 1]);
        ny[ip] = pk2(-yi[2 * ip], -yi[2 * ip + 1]);
        nz[ip] = pk2(-zi[2 * ip], -zi[2 * ip + 1]);
    }

    const unsigned hist32 = (unsigned)__cvta_generic_to_shared(sH);
    // Byte offset of a pair's word without touching the FMA pipe (an IMAD per pair there
    // costs as much as a packed FP32 instruction): t = u >> (k - cb - 2) holds the slot in
    // bits [cb + 2, cb + 2 + lg) -- above them, for !LOWER, the bits of 1.5*2^(23-k), which
    // start at bit 24 - k + cb >= cb + 2 + lg --, fraction bits below.  CLAMP: one MIN
    // sends everything beyond the histogram to its last slot (a scratch word); without
    // it the slot is below hslots already.  One LOP3 keeps the slot field and inserts the
    // lane's column; the base is the kernel's shared-memory base, an immediate.
    const int tshift = fc.k - fc.cb - 2;
    const unsigned low = (4u << fc.cb) - 1u;
    const unsigned tmask = ((4u << (fc.cb + fc.lg)) - 1u) & ~low;
    const unsigned tmax = ((((LOWER ? 0u : fc.cbits) >> fc.k) + (unsigned)(fc.hslots - 1))
                           << (fc.cb + 2)) | low;
    const unsigned colbits = ((unsigned)lane & ((1u << fc.cb) - 1u)) << 2;
    const unsigned span_l = LOWER ? fc.span : fc.cbits + fc.span;
    const unsigned fmask = (1u << fc.k) - 1u;      // fraction bits of the bin coordinate
    const float scale = fc.scale, offm = ff.offm;

    auto stage_tile = [&](int jt, int buf) {
        const float4 *src = f2 + (int64_t)jt * TILE;
        float4 *dst = sJ + buf * TSTRIDE;
#pragma unroll
        for (int q = 0; q < IPT; ++q)
            __pipeline_memcpy_async(dst + q * kThreads + tid, src + q * kThreads + tid,
                                    sizeof(float4));
        __pipeline_commit();
    };
    stage_tile(jt0, 0);

    // x-clean tile pairs (filter_cleanx_form) in the half-box unclamped body of x-sorted
    // groups.  The tile pair's form is kept in a shared word (sCount[1]) and the box edge
    // L is reread where it is needed: no register stays live across the hot loop for them.
    // Not with exclusions: the tag compare leaves no room for a second body without
    // spills in the hot loop (ptxas -v; those launches keep the dirty form).
    constexpr bool CXOK = HALF && !CLAMP && !EXCL;
    unsigned *sForm = sCount + 1;

    unsigned long long audit_bad = 0, audit_unc = 0;
    int buf = 0;
    for (int jt = jt0; jt < jt1; ++jt) {
        if (jt + 1 < jt1) {
            stage_tile(jt + 1, buf ^ 1);
            __pipeline_wait_prior(1);
        } else {
            __pipeline_wait_prior(0);
        }
        // the tile pair's x form (uniform over the block); S = +L moves this thread's own
        // rows of the j-tile (their copies have landed), S = -L the thread's i-coordinates
        if constexpr (CXOK) {
            if (P.xform != nullptr) {
                const float L = -ff.nbox[0];
                const int form =
                    P.xform[((int64_t)frame * (P.pad1 / TILE) + it) * P.n_jtiles + jt];
                if (tid == 0) *sForm = (unsigned)form;
                if (form == 2) {
                    float4 *rows = sJ + buf * TSTRIDE;
#pragma unroll
                    for (int q = 0; q < IPT; ++q)
                        rows[q * kThreads + tid].x = __fsub_rn(rows[q * kThreads + tid].x, L);
                }
                if (form == 3) {
#pragma unroll
                    for (int ip = 0; ip < IPT / 2; ++ip) nx[ip] = add2(nx[ip], pk2(L, L));
                }
            } else if (tid == 0) {
                *sForm = 0u;
            }
        }
        __syncthreads();

        const unsigned weight = (P.same && jt > it) ? 2u : 1u;
        unsigned wi[IPT];
#pragma unroll
        for (int ii = 0; ii < IPT; ++ii) wi[ii] = ii * kThreads < nv ? weight : 0u;
        const int jn = min(TILE, P.n2 - jt * TILE);
        const float4 *tile = sJ + buf * TSTRIDE;

        // the tile's pipeline and deferred entries, in the x-clean form (CX) or not
        auto body = [&](auto cx_tag) {
        constexpr bool CX = decltype(cx_tag)::value;
        // Stage A1: packed squared distances of NR tile rows against the IPT particles of
        // this thread (FMA pipe only).
        auto stage_a1 = [&](const float4 *pj, f32x2 (*dd)[IPT / 2], auto nr_tag) {
            constexpr int NR = decltype(nr_tag)::value;
#pragma unroll
            for (int r = 0; r < NR; ++r)
#pragma unroll
                for (int ip = 0; ip < IPT / 2; ++ip)
                    dd[r][ip] = filter_d2<HALF, CX>(nx[ip], ny[ip], nz[ip], pk2(pj[r].x, pj[r].x),
                                          pk2(pj[r].y, pj[r].y), pk2(pj[r].z, pj[r].z), ff);
        };
        // Stage A2: square roots (MUFU) and fixed-point bin coordinates.
        auto stage_a2 = [&](const f32x2 (*dd)[IPT / 2], unsigned (*uu)[IPT], auto nr_tag) {
            constexpr int NR = decltype(nr_tag)::value;
#pragma unroll
            for (int r = 0; r < NR; ++r)
#pragma unroll
                for (int ip = 0; ip < IPT / 2; ++ip)
                    filter_bin2<LOWER>(dd[r][ip], scale, offm, fc.cbits, uu[r][2 * ip],
                                       uu[r][2 * ip + 1]);
        };
        // Stage B: histogram updates and the uncertainty test of NR rows (ALU pipe,
        // LSU), then one rarely taken branch for the uncertain pairs of the group.
        auto stage_hist = [&](const float4 *pj, const unsigned (*uu)[IPT], unsigned *vmin,
                              auto nr_tag) {
            constexpr int NR = decltype(nr_tag)::value;
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                vmin[r] = 0xffffffffu;
#pragma unroll
                for (int ii = 0; ii < IPT; ++ii) {
                    const unsigned u = uu[r][ii];
                    // uncertain iff the fraction bits are below wlim; keep the smallest
                    vmin[r] = min(vmin[r], u & fmask);
                    unsigned t = u >> tshift;
                    if (CLAMP) t = min(t, tmax);
                    if (EXCL && gi[ii] == __float_as_int(pj[r].w)) t = tmax;
                    red_shared_hot(hist32 + lop3_and_or(t, tmask, colbits), wi[ii]);
                    if (AUDIT) {
                        const bool unc = (u & fmask) < ff.wlim;
                        const bool in = u < span_l;
                        // an unclamped frame must never leave the histogram
                        if (!CLAMP && !in) ++audit_bad;
                        float4 pr = pj[r];       // the j-row as the reference sees it
                        if (CX && *sForm == 2u) pr.x = __fadd_rn(pr.x, -ff.nbox[0]);
                        const double d2 = pair_d2(xi[ii], yi[ii], zi[ii], pr, P.boxes[frame]);
                        const int slot = slot_search(d2, sT, n_bins);
                        // the slot the pair was added to, and the exact one
                        const unsigned fs = in ? ((LOWER ? u : u - fc.cbits) >> fc.k)
                                               : (unsigned)(fc.hslots - 1);
                        const unsigned xs = (unsigned)(slot + fc.lo);
                        const bool counted = slot >= 1 && slot <= n_bins;
                        if (in && unc) ++audit_unc;
                        // certain pairs must agree with the exact arithmetic wherever
                        // a count is at stake
                        if (!(in && unc) && xs != fs &&
                            (counted || (fs >= (unsigned)fc.lo + 1u &&
                                         fs <= (unsigned)(fc.lo + n_bins))))
                            ++audit_bad;
                    }
                }
            }
        };
        // the rarely taken branch: rows with an uncertain pair go on the block's list
        auto stage_push = [&](const unsigned *vmin, int jj, auto nr_tag) {
            constexpr int NR = decltype(nr_tag)::value;
            unsigned vall = vmin[0];
#pragma unroll
            for (int r = 1; r < NR; ++r) vall = min(vall, vmin[r]);
            if (vall < ff.wlim) {
#pragma unroll
                for (int r = 0; r < NR; ++r) {
                    if (vmin[r] < ff.wlim) {
                        const unsigned entry = ((unsigned)tid << 16) | (unsigned)(jj + r);
                        const unsigned idx = atomicAdd(sCount, 1u);
                        if (idx < (unsigned)kListCap) sList[idx] = entry;
                        else
                            filter_fix<EXCL, LOWER, IPT, HALF, CX>(P, frame, it, entry, tile,
                                                                   sT, hist32, weight,
                                                                   CX ? (int)*sForm : 0);
                    }
                }
            }
        };
        auto stage_b = [&](const float4 *pj, const unsigned (*uu)[IPT], int jj, auto nr_tag) {
            constexpr int NR = decltype(nr_tag)::value;
            unsigned vmin[NR];
            stage_hist(pj, uu, vmin, nr_tag);
            stage_push(vmin, jj, nr_tag);
        };
        // Software pipeline over pairs of rows.  What crosses the iteration boundary are the
        // squared distances of rows (jj, jj+1): an iteration starts with their square roots
        // (MUFU latency) and runs bin coordinates -> histogram updates (ALU pipe, LSU) next
        // to the independent squared distances of rows (jj+2, jj+3) (FMA pipe), so that
        // every warp offers both pipes work from its first to its last instruction; the
        // rows after those are fetched from shared memory one more iteration ahead.  Rows
        // up to TILE - 1 always exist (the packed arrays are padded), so the last
        // iteration may evaluate two rows nobody uses; the rows fetched past the end of the
        // tile are its kTilePad padding rows.
        using two = std::integral_constant<int, 2>;
        const int jn2 = jn & ~1;
        f32x2 da[2][IPT / 2], db[2][IPT / 2];
        float4 cur[2] = {tile[0], tile[1]};
        float4 nxt[2] = {tile[2], tile[3]};
        if (jn2 > 0) stage_a1(cur, da, two());
        // one step of the pipeline: rows (jj, jj+1) leave it (their squared distances in
        // din), rows (jj+2, jj+3) enter it (into dout).  The steps alternate da and db,
        // so no register is copied from one step to the next.
        auto step = [&](int jj, const f32x2 (*din)[IPT / 2], f32x2 (*dout)[IPT / 2],
                        unsigned *vmin) {
            unsigned ua[2][IPT];
            const float4 nn[2] = {nxt[0], nxt[1]};
            nxt[0] = tile[jj + 4];
            nxt[1] = tile[jj + 5];
            stage_a2(din, ua, two());
            stage_a1(nn, dout, two());
            stage_hist(cur, ua, vmin, two());
            cur[0] = nn[0]; cur[1] = nn[1];
        };
        int jj = 0;
#if MDH_FILTER_ROWS == 4
        // two steps per trip, ONE test for uncertain pairs behind them: no branch between
        // the steps, so the second step's arithmetic overlaps the first step's updates
        for (; jj + 4 <= jn2; jj += 4) {
            unsigned vmin[4];
            step(jj, da, db, vmin);
            step(jj + 2, db, da, vmin + 2);
            stage_push(vmin, jj, std::integral_constant<int, 4>());
        }
#else
        // two steps per trip, each with its own test for uncertain pairs: one loop
        // counter, compare and branch per 2 steps, one row address per 2 steps
        for (; jj + 4 <= jn2; jj += 4) {
            unsigned vmin[2];
            step(jj, da, db, vmin);
            stage_push(vmin, jj, two());
            step(jj + 2, db, da, vmin);
            stage_push(vmin, jj + 2, two());
        }
#endif
        if (jj < jn2) {
            unsigned vmin[2];
            step(jj, da, db, vmin);
            stage_push(vmin, jj, two());
        }
        if (jn2 < jn) {
            f32x2 d1[1][IPT / 2];
            unsigned u1[1][IPT];
            stage_a1(tile + jn2, d1, std::integral_constant<int, 1>());
            stage_a2(d1, u1, std::integral_constant<int, 1>());
            stage_b(tile + jn2, u1, jn2, std::integral_constant<int, 1>());
        }
        __syncthreads();

        // drain the deferred entries of this tile while it is still in shared memory
        const unsigned n_push = *sCount;
        const unsigned n_list = min(n_push, (unsigned)kListCap);
        for (unsigned e = tid; e < n_list; e += kThreads)
            filter_fix<EXCL, LOWER, IPT, HALF, CX>(P, frame, it, sList[e], tile, sT, hist32,
                                                   weight, CX ? (int)*sForm : 0);
        if (tid == 0 && n_push) {
            atomicAdd(&P.fstats[0], (unsigned long long)n_list);
            if (n_push > n_list) atomicAdd(&P.fstats[1], (unsigned long long)(n_push - n_list));
        }
        };
        if constexpr (CXOK) {
            if (*sForm) {
                body(std::true_type());
                if (tid == 0)     // nv of thread 0: the rows of the i-tile below n1
                    atomicAdd(&P.fstats[8], (unsigned long long)min(TILE, nv) *
                                                (unsigned long long)jn);
                if (*sForm == 3u) {
                    const float L = -ff.nbox[0];
#pragma unroll
                    for (int ip = 0; ip < IPT / 2; ++ip) nx[ip] = add2(nx[ip], pk2(-L, -L));
                }
            } else {
                body(std::false_type());
            }
        } else {
            body(std::false_type());
        }
        __syncthreads();
        if (tid == 0) *sCount = 0;
        buf ^= 1;
    }

    // merge into the global int64 histogram.  The columns are summed modulo 2^32 first
    // (a correction is subtracted from the column that was incremented, but the block
    // total is what stays below 2^32, not every word).
    for (int k = tid; k < n_bins; k += kThreads) {
        unsigned s = 0;
        for (int q = 0; q < (1 << fc.cb); ++q)
            s += sH[((k + 1 + fc.lo) << fc.cb) + ((q + tid) & ((1 << fc.cb) - 1))];
        if (s) atomicAdd(&P.counts[k], (unsigned long long)s);
    }
    if (AUDIT) {
        if (audit_bad) atomicAdd(&P.fstats[2], audit_bad);
        if (audit_unc) atomicAdd(&P.fstats[3], audit_unc);
    }
}

template <bool EXCL, bool LOWER, bool AUDIT, int IPT, int OCC>
__global__ void __launch_bounds__(kThreads, OCC)
    rdf_filter_kernel(const __grid_constant__ PairParams P)
{
    const FrameFilter ff = P.filt[blockIdx.y];
    if (ff.wlim == 0u) {                  // left to the exact kernel (whole block)
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&P.fstats[4], 1ull);
        return;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(&P.fstats[ff.halfbox ? 5 : 6], 1ull);
    // the frame's flags are uniform over the block: one branch, then straight-line code.
    // A launch whose coordinates may be negative (LOWER) never has unclamped frames.
    if (ff.halfbox) {
        if constexpr (!LOWER) {
            if (ff.unclamped) {
                filter_block<EXCL, LOWER, AUDIT, IPT, true, false>(P, ff);
                return;
            }
        }
        filter_block<EXCL, LOWER, AUDIT, IPT, true, true>(P, ff);
    } else {
        filter_block<EXCL, LOWER, AUDIT, IPT, false, true>(P, ff);
    }
}

// Largest relative error of sqrt.approx.ftz.f32 over two binades [1, 4) -- all 2^24
// inputs; the instruction works on the mantissa and the exponent parity, so this
// covers every normal input.  Stored as the bits of a non-negative double.
__global__ void sqrt_error_kernel(unsigned long long *out)
{
    const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;     // < 2^24
    const float x = __uint_as_float(0x3f800000u + i);
    float s;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(x));
    const double t = sqrt((double)x);
    double err = fabs((double)s - t) / t;
    for (int o = 16; o; o >>= 1) err = fmax(err, __shfl_xor_sync(0xffffffffu, err, o));
    if ((threadIdx.x & 31) == 0 && err > 0.0)
        atomicMax(out, (unsigned long long)__double_as_longlong(err));
}

struct PrepareParams {
    const FrameBox *boxes;
    const unsigned *ext1, *ext2;     // [F][6] keys
    FrameFilter *out;
    unsigned long long *fstats;      // [7]: frames the filter kernel will run unclamped
    int n_frames;
    FilterPrep prep;
};

__global__ void rdf_filter_prepare_kernel(const PrepareParams Q)
{
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= Q.n_frames) return;
    const FrameFilter ff =
        filter_prepare_frame<true>(Q.boxes[f], Q.ext1 + f * 6, Q.ext2 + f * 6, Q.prep);
    Q.out[f] = ff;
    // counted here rather than in the filter kernel, whose register allocation is at its
    // limit; rdf_filter_kernel takes the unclamped body exactly for these frames (the
    // flag is only set when the launch's layout has no negative coordinates, !LOWER)
    if (ff.unclamped) atomicAdd(&Q.fstats[7], 1ull);
}

template <bool EXCL, bool LOWER, bool AUDIT, int IPT, int OCC>
int launch_filter_o(mdh_ctx *c, const PairParams &P, dim3 grid)
{
    const size_t smem = filter_smem_bytes<IPT>(P.n_bins, P.fc.hslots, P.fc.cb);
    auto kern = rdf_filter_kernel<EXCL, LOWER, AUDIT, IPT, OCC>;
    MDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)smem));
    kern<<<grid, kThreads, smem, c->stream>>>(P);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    return MDH_OK;
}

template <bool EXCL, bool LOWER>
int launch_filter_a(mdh_ctx *c, const PairParams &P, dim3 grid, bool audit)
{
    const int occ = c->rdf.filter_occ;
    if (c->rdf.ipt == 2) {
        if (audit) return launch_filter_o<EXCL, LOWER, true, 2, 2>(c, P, grid);
        return occ == 4   ? launch_filter_o<EXCL, LOWER, false, 2, 4>(c, P, grid)
               : occ == 3 ? launch_filter_o<EXCL, LOWER, false, 2, 3>(c, P, grid)
                          : launch_filter_o<EXCL, LOWER, false, 2, 2>(c, P, grid);
    }
    if (audit) return launch_filter_o<EXCL, LOWER, true, 4, 2>(c, P, grid);
    return occ == 3 ? launch_filter_o<EXCL, LOWER, false, 4, 3>(c, P, grid)
                    : launch_filter_o<EXCL, LOWER, false, 4, 2>(c, P, grid);
}

}  // namespace

// Measured once per process (thread-safe enough: a race recomputes the same number).
static double g_sqrt_err = -1.0;

int rdf_filter_sqrt_error(mdh_ctx *c, double *err)
{
    if (g_sqrt_err < 0.0) {
        unsigned long long *d = nullptr, h = 0;
        MDH_CUDA(cudaMalloc(&d, sizeof(h)));
        MDH_CUDA(cudaMemsetAsync(d, 0, sizeof(h), c->stream));
        sqrt_error_kernel<<<(1u << 24) / 256, 256, 0, c->stream>>>(d);
        MDH_CUDA(cudaGetLastError());
        c->launches++;
        MDH_CUDA(cudaMemcpyAsync(&h, d, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
        MDH_CUDA(cudaStreamSynchronize(c->stream));
        MDH_CUDA(cudaFree(d));
        double e;
        memcpy(&e, &h, sizeof(e));
        g_sqrt_err = e;
    }
    *err = g_sqrt_err;
    return MDH_OK;
}

// shared memory of one block of the all-pairs filter kernel
static size_t filter_need(const RdfState &R, int hslots, int cb)
{
    return R.ipt == 2 ? filter_smem_bytes<2>(R.n_bins, hslots, cb)
                      : filter_smem_bytes<4>(R.n_bins, hslots, cb);
}

// histogram columns: as many (up to one per lane) as the shared memory of R.filter_occ
// resident blocks allows
static int filter_columns(const RdfState &R, int hslots, int k)
{
    const size_t budget = (size_t)(224 * 1024) / R.filter_occ - 1024;
    int cb = 5;
    while (cb > 0 && filter_need(R, hslots, cb) > budget) --cb;
    return std::min(cb, k - 2);
}

// Decides whether a configuration can use the filter and fills R.fc.
bool rdf_filter_configure(RdfState &R, const double *thr, double sqrt_err)
{
    R.filter_ok = false;
    const int n_bins = R.n_bins;
    int lg = 0;
    while ((1 << lg) < n_bins + 2) ++lg;
    const int k = std::min(16, 22 - lg);
    if (k < 9) return false;
    if (!(sqrt_err >= 0.0 && sqrt_err <= 1.0 / 4194304.0)) return false;   // 2^-22
    const double scale = n_bins / (R.r_hi - R.r_lo);
    // the thresholds must be the uniform edges the bound assumes (to 1e-9 of a bin)
    for (int i = 0; i <= n_bins; ++i) {
        const double e = R.r_lo + i / scale;
        if (!(fabs(sqrt(thr[i]) - e) * scale <= 1e-9)) return false;
    }
    FilterConst fc;
    fc.k = k;
    fc.scale = (float)scale;
    const double two_k = (double)(1 << k);
    const double magic = 1.5 * (double)(1 << (23 - k));
    // slot = bin + 1: one scratch slot below the range
    const double off = nearbyint((1.0 - R.r_lo * scale) * two_k) / two_k;
    fc.offbase = magic + off;
    // representable with the largest shift added, and still below the next binade
    if ((double)(float)fc.offbase != fc.offbase ||
        (double)(float)(fc.offbase + 0.125) != fc.offbase + 0.125) return false;
    const float mf = (float)magic;
    memcpy(&fc.cbits, &mf, 4);
    fc.span = (unsigned)(n_bins + 2) << k;
    fc.lower = R.r_lo > 0.0;
    fc.lg = lg;
    fc.lo = 0;
    fc.hslots = n_bins + 2;
    fc.unclamped = 0;
    fc.cb = filter_columns(R, fc.hslots, k);
    if (filter_need(R, fc.hslots, fc.cb) > 200 * 1024) return false;
    // the cell-pair kernel keeps one histogram per warp with 2^sb sub-bins per bin
    fc.sb = std::min(2, k);
    R.fc = fc;
    R.filter_ok = true;
    return true;
}

FilterPrep rdf_filter_prep(const RdfState &R, double sqrt_err)
{
    FilterPrep q;
    q.k = R.fc.k;
    q.halfbox = 0;
    q.scale = R.n_bins / (R.r_hi - R.r_lo);
    q.d_max = R.r_hi + 2.0 / q.scale;
    q.sqrt_err = sqrt_err;
    q.offbase = R.fc.offbase;
    q.fscale = (double)R.fc.scale;
    q.hslots = 0;
    return q;
}

// The all-pairs filter kernel's histogram layout for a batch of frames.  Sized so that
// every slot a half-box frame of the batch can reach is a word (rdf_device.cuh::
// filter_reach with the largest |m| of the form, |m_k| <= box_k / 2), with the offset
// shifted by lo = ceil(r_lo * scale) slots so that no coordinate is negative.  When that
// histogram does not fit the shared memory of R.filter_occ blocks at the clamped layout's
// column count, or would leave fewer than 9 fraction bits or more than one fewer than the
// clamped layout (each lost bit about doubles the uncertain pairs; one bit is what the
// measured trade covers: cfg2, 1.6x deferred entries for a 7 % faster kernel), it is the
// clamped layout R.fc.
static FilterConst filter_plan(const RdfState &R, const FrameBox *boxes, int n_frames,
                               double sqrt_err)
{
    FilterConst fc = R.fc;
    const int n_bins = R.n_bins;
    const double scale = n_bins / (R.r_hi - R.r_lo);
    const int lo = (int)ceil(R.r_lo * scale);
    // offset coordinate: 1 + lo - r_lo * scale rounded to 2^-k, plus the window (< 1/16 by
    // filter_prepare_frame's 2m + 1 < 2^k / 8)
    auto top = [&](const FrameBox &b, int k) {
        double mb[3];
        for (int a = 0; a < 3; ++a) {
            const double h = 0.5 * b.box[a];
            mb[a] = filter_halfbox_mbound(a == R.drop_axis ? 0.0 : h, h);  // dropped: df = 0
        }
        const double c0 = 1.0 + lo - R.r_lo * scale + 1.0 / 16.0 + 1.0 / (double)(2u << k);
        return floor(filter_reach(mb, (double)fc.scale, c0, sqrt_err, k));
    };
    // the frames' reachable slots at k = 9, the coarsest rounding; the histogram covers the
    // largest of them that fits (frames beyond it keep the clamped body)
    std::vector<double> t9(n_frames);
    for (int f = 0; f < n_frames; ++f) t9[f] = top(boxes[f], 9);
    std::sort(t9.begin(), t9.end());
    t9.erase(std::unique(t9.begin(), t9.end()), t9.end());
    int hslots = 0, k = 0, cb = 0;
    for (int q = (int)t9.size() - 1; q >= 0 && hslots == 0; --q) {
        if (!(t9[q] < 65536.0)) continue;
        const int hs = std::max((int)t9[q] + 1, n_bins + lo + 2);
        int lg = 0;
        while ((1 << lg) < hs) ++lg;
        k = std::min(16, 22 - lg);
        if (k < 9 || k < R.fc.k - 1) continue;
        cb = filter_columns(R, hs, k);
        if (cb < R.fc.cb || filter_need(R, hs, cb) > 200 * 1024) continue;
        hslots = hs;
    }
    if (hslots == 0) return fc;
    int lg = 0;
    while ((1 << lg) < hslots) ++lg;
    const double two_k = (double)(1 << k);
    const double magic = 1.5 * (double)(1 << (23 - k));
    const double offbase = magic + nearbyint((1.0 + lo - R.r_lo * scale) * two_k) / two_k;
    // representable with the largest shift added, and still below the next binade
    if ((double)(float)offbase != offbase || (double)(float)(offbase + 0.125) != offbase + 0.125)
        return fc;
    fc.k = k;
    fc.offbase = offbase;
    const float mf = (float)magic;
    memcpy(&fc.cbits, &mf, 4);
    fc.span = (unsigned)hslots << k;
    fc.lg = lg;
    fc.cb = cb;
    fc.lower = 0;
    fc.lo = lo;
    fc.hslots = hslots;
    fc.unclamped = 1;
    return fc;
}

// The per-frame preparation of the all-pairs filter kernel for the batch layout fca
static FilterPrep filter_prep_allpairs(const RdfState &R, const FilterConst &fca, double sqrt_err)
{
    FilterPrep q = rdf_filter_prep(R, sqrt_err);
    q.halfbox = 1;                 // the all-pairs kernel evaluates both forms
    q.k = fca.k;
    q.offbase = fca.offbase;
    q.hslots = fca.unclamped ? fca.hslots : 0;
    return q;
}

// Builds the per-frame filter parameters of a batch (device side, asynchronous) and the
// all-pairs kernel's layout for it (R.fca).
int rdf_filter_prepare(mdh_ctx *c, int f0, int n_frames, double sqrt_err)
{
    RdfState &R = c->rdf;
    if (int rc = R.filt.reserve(sizeof(FrameFilter) * n_frames)) return rc;
    R.fca = filter_plan(R, R.h_boxes.data() + f0, n_frames, sqrt_err);
    PrepareParams Q;
    Q.boxes = R.boxes.as<FrameBox>() + f0;
    Q.ext1 = R.ext1.as<unsigned>();
    Q.ext2 = R.same ? Q.ext1 : R.ext2.as<unsigned>();
    Q.out = R.filt.as<FrameFilter>();
    Q.fstats = R.fstats.as<unsigned long long>();
    Q.n_frames = n_frames;
    Q.prep = filter_prep_allpairs(R, R.fca, sqrt_err);
    rdf_filter_prepare_kernel<<<(n_frames + 127) / 128, 128, 0, c->stream>>>(Q);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    return MDH_OK;
}

int rdf_filter_launch(mdh_ctx *c, const PairParams &P, dim3 grid, bool excl, bool audit)
{
    if (excl)
        return P.fc.lower ? launch_filter_a<true, true>(c, P, grid, audit)
                          : launch_filter_a<true, false>(c, P, grid, audit);
    return P.fc.lower ? launch_filter_a<false, true>(c, P, grid, audit)
                      : launch_filter_a<false, false>(c, P, grid, audit);
}

// Device-free: the layouts and per-frame windows the filter would use (mdh_rdf_filter_window).
int rdf_filter_window_impl(int n_bins, double r_lo, double r_hi, int drop_axis, int ipt,
                           int filter_occ, double sqrt_err, int n_frames, const float *box,
                           const float *ext1, const float *ext2, double *layout, double *frames)
{
    MDH_REQUIRE(n_bins >= 1 && n_bins <= 65536, MDH_EINVAL, "filter_window: n_bins must be in [1, 65536]");
    MDH_REQUIRE(r_hi > r_lo && r_lo >= 0, MDH_EINVAL, "filter_window: invalid range");
    MDH_REQUIRE(drop_axis >= -1 && drop_axis <= 2, MDH_EINVAL, "filter_window: invalid drop_axis");
    MDH_REQUIRE(ipt == 2 || ipt == 4, MDH_EINVAL, "filter_window: ipt must be 2 or 4");
    MDH_REQUIRE(filter_occ >= 2 && filter_occ <= 4, MDH_EINVAL,
                "filter_window: filter_occ must be in [2, 4]");
    MDH_REQUIRE(n_frames >= 1 && box != nullptr && ext1 != nullptr && layout != nullptr &&
                    frames != nullptr, MDH_EINVAL, "filter_window: NULL argument");
    if (ext2 == nullptr) ext2 = ext1;
    RdfState R;                    // host fields only: no device buffer is touched
    R.n_bins = n_bins;
    R.r_lo = r_lo;
    R.r_hi = r_hi;
    R.drop_axis = drop_axis;
    R.ipt = ipt;
    R.filter_occ = filter_occ;
    // uniform edges (rdf_filter_configure only checks that the thresholds are these)
    std::vector<double> thr(n_bins + 1);
    for (int i = 0; i <= n_bins; ++i) {
        const double e = r_lo + i * ((r_hi - r_lo) / n_bins);
        thr[i] = e * e;
    }
    MDH_REQUIRE(rdf_filter_configure(R, thr.data(), sqrt_err), MDH_EINVAL,
                "filter_window: the configuration is not eligible for the fp32 filter");
    // per-frame boxes as mdh_rdf_accumulate builds them
    std::vector<FrameBox> boxes(n_frames);
    for (int f = 0; f < n_frames; ++f)
        for (int k = 0; k < 3; ++k) {
            const float b = box[3 * f + k];
            MDH_REQUIRE(b > FLT_EPSILON && std::isfinite(b), MDH_EINVAL,
                        "filter_window: box edge %d of frame %d is not a positive length", k, f);
            boxes[f].box[k] = (double)b;
            boxes[f].inv[k] = (double)(float)(1.0 / (double)b);
        }
    const FilterConst fca = filter_plan(R, boxes.data(), n_frames, sqrt_err);
    for (int q = 0; q < 2; ++q) {
        const FilterConst &fc = q ? fca : R.fc;
        const double v[12] = {(double)fc.k,  (double)fc.scale, fc.offbase,          (double)fc.cbits,
                              (double)fc.span, (double)fc.lg,  (double)fc.cb,       (double)fc.hslots,
                              (double)fc.lo, (double)fc.unclamped, (double)fc.sb, (double)fc.lower};
        for (int i = 0; i < 12; ++i) layout[12 * q + i] = v[i];
    }
    const FilterPrep qa = filter_prep_allpairs(R, fca, sqrt_err);
    const FilterPrep qc = rdf_filter_prep(R, sqrt_err);     // cell lists: rint form, clamped
    for (int f = 0; f < n_frames; ++f) {
        unsigned k1[6], k2[6];
        for (int i = 0; i < 6; ++i) {
            const unsigned b1 = f32_bits(ext1[6 * f + i]), b2 = f32_bits(ext2[6 * f + i]);
            k1[i] = (b1 & 0x80000000u) ? ~b1 : (b1 | 0x80000000u);   // rdf_device.cuh::ext_key
            k2[i] = (b2 & 0x80000000u) ? ~b2 : (b2 | 0x80000000u);
        }
        for (int q = 0; q < 2; ++q) {
            double mu = 0.0;
            const FrameFilter ff = q ? filter_prepare_frame(boxes[f], k1, k2, qc, &mu)
                                     : filter_prepare_frame<true>(boxes[f], k1, k2, qa, &mu);
            double *o = frames + 10 * f + 5 * q;
            o[0] = (double)ff.offm;
            o[1] = (double)ff.wlim;
            o[2] = (double)ff.halfbox;
            o[3] = (double)ff.unclamped;
            o[4] = mu;
        }
    }
    return MDH_OK;
}
