// rdf_tri.cu -- pair histogram for TRICLINIC cells (seam #1 with a non-orthogonal box).
//
// The reference hands the full `dims` (lengths and angles) to capped_distance
// (/root/reference/src/mdhelper/analysis/structure.py:93-96); for a triclinic cell the
// third-party MDAnalysis code then (restated from its published algorithm, SURVEY.md
// Appendix A; NOT pinned against MDAnalysis itself, which is not installable here):
//   1. wraps both coordinate sets into the primary cell (lib/include/calc_distances.h
//      `_triclinic_pbc`).  Restated mathematically: along c, then b, then a,
//      s = floor(x_k / h_kk), r -= s * h_k, in double, rounded back to float32.  For
//      coordinates that already lie in the cell this is the identity, as in MDAnalysis;
//      for the others its float rounding details are not reproduced.
//   2. per pair: dx = (double)(float)(r_j - r_i), then `minimum_image_triclinic`: the
//      shortest of the 27 images dx + ix a + iy b + iz c, ix, iy, iz in {-1, 0, 1}
//      (loop order ix, iy, iz; strict "<"), every sum in double in the order
//      ((dx0 + a_x ix) + b_x iy) + c_x iz, (dx1 + b_y iy) + c_y iz, dx2 + c_z iz,
//      and d^2 = (rx rx + ry ry) + rz rz.
// Binning is the squared-threshold comparison of the orthorhombic kernels (rdf.cu).
//
// Three pair kernels give the same counts:
//   rdf_triclinic_kernel   all pairs, every pair evaluates the 27 images (fp64);
//   rdf_tri_filter_kernel  all pairs, ONE image per pair in fp32 behind an error bound,
//                          the 27 images for pairs near a bin edge (DESIGN.md 4.8b);
//   rdf_tri_cells_kernel   cut-off runs: a cell list in fractional coordinates, and for
//                          every candidate only the ONE image that can be in range
//                          (argument and margin: tri_grid_plan below, DESIGN.md 4.8).

#include <algorithm>

#include "rdf_cells.cuh"
#include "rdf_device.cuh"

using namespace rdfdev;

namespace {

// in place on the packed float4 array
__global__ void tri_wrap_kernel(float4 *__restrict__ p, int64_t npad, int n,
                                const TriBox *__restrict__ boxes)
{
    const int frame = blockIdx.y;
    const TriBox h = boxes[frame];
    float4 *pf = p + (int64_t)frame * npad;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float4 v = pf[i];
        double x = v.x, y = v.y, z = v.z;
        double s = floor(z / h.cz);
        if (s != 0.0) { x -= s * h.cx; y -= s * h.cy; z -= s * h.cz; }
        s = floor(y / h.by);
        if (s != 0.0) { x -= s * h.bx; y -= s * h.by; }
        s = floor(x / h.ax);
        if (s != 0.0) x -= s * h.ax;
        v.x = (float)x; v.y = (float)y; v.z = (float)z;
        pf[i] = v;
    }
}

// d^2 of ONE image of dx = (double)(float)(r_j - r_i), in the reference's operation order;
// s.. are the image's shift terms h_k * i (i in {-1, 0, 1}: exact products).  tri_d2 (all
// 27 images) and the cell-list kernel (the one image that can be in range) both go
// through it, so the two cannot drift apart.
__device__ __forceinline__ double tri_image_d2(double dx0, double dx1, double dx2, double sax,
                                               double sbx, double sby, double scx, double scy,
                                               double scz)
{
    const double rx = __dadd_rn(__dadd_rn(__dadd_rn(dx0, sax), sbx), scx);
    const double ry = __dadd_rn(__dadd_rn(dx1, sby), scy);
    const double rz = __dadd_rn(dx2, scz);
    return __dadd_rn(__dadd_rn(__dmul_rn(rx, rx), __dmul_rn(ry, ry)), __dmul_rn(rz, rz));
}

__device__ __forceinline__ double tri_d2(float xi, float yi, float zi, const float4 &pj,
                                         const TriBox &h)
{
    const double dx0 = (double)__fsub_rn(pj.x, xi);
    const double dx1 = (double)__fsub_rn(pj.y, yi);
    const double dx2 = (double)__fsub_rn(pj.z, zi);
    double best = (double)FLT_MAX;
#pragma unroll
    for (int ix = -1; ix <= 1; ++ix)
#pragma unroll
        for (int iy = -1; iy <= 1; ++iy)
#pragma unroll
            for (int iz = -1; iz <= 1; ++iz) {
                const double dsq = tri_image_d2(dx0, dx1, dx2, h.ax * ix, h.bx * iy, h.by * iy,
                                                h.cx * iz, h.cy * iz, h.cz * iz);
                if (dsq < best) best = dsq;
            }
    return best;
}

struct TriParams {
    const float4 *p1, *p2;
    int64_t pad1, pad2;
    int n1, n2;
    const TriBox *boxes;
    const double *thr;
    int n_bins;
    unsigned long long *counts;
    int jchunk;                    // j particles per block (multiple of 256)
};

template <bool EXCL>
__global__ void __launch_bounds__(256) rdf_triclinic_kernel(const TriParams P)
{
    extern __shared__ __align__(16) unsigned char smem[];
    double *sT = reinterpret_cast<double *>(smem);
    float4 *sJ = reinterpret_cast<float4 *>(smem + align16(sizeof(double) * (P.n_bins + 1)));
    unsigned *sH = reinterpret_cast<unsigned *>(sJ + 256);

    const int tid = threadIdx.x, warp = tid >> 5;
    const int frame = blockIdx.z;
    const int n_bins = P.n_bins;
    for (int k = tid; k <= n_bins; k += 256) sT[k] = P.thr[k];
    for (int k = tid; k < kWarps * n_bins; k += 256) sH[k] = 0;

    const float4 *f1 = P.p1 + (int64_t)frame * P.pad1;
    const float4 *f2 = P.p2 + (int64_t)frame * P.pad2;
    const TriBox h = P.boxes[frame];
    const int i = blockIdx.x * 256 + tid;
    const bool valid = i < P.n1;
    const float4 a = f1[min(i, P.n1 - 1)];
    unsigned *myhist = sH + warp * n_bins;

    const int j0 = blockIdx.y * P.jchunk, j1 = min(P.n2, j0 + P.jchunk);
    for (int jt = j0; jt < j1; jt += 256) {
        __syncthreads();
        if (jt + tid < j1) sJ[tid] = f2[jt + tid];
        __syncthreads();
        const int jn = min(256, j1 - jt);
        if (!valid) continue;
        for (int jj = 0; jj < jn; ++jj) {
            const float4 pj = sJ[jj];
            if (EXCL && __float_as_int(a.w) == __float_as_int(pj.w)) continue;
            const double d2 = tri_d2(a.x, a.y, a.z, pj, h);
            const int slot = slot_search(d2, sT, n_bins);
            if ((unsigned)(slot - 1) < (unsigned)n_bins) atomicAdd(&myhist[slot - 1], 1u);
        }
    }
    __syncthreads();
    for (int k = tid; k < n_bins; k += 256) {
        unsigned long long s = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) s += sH[w * n_bins + k];
        if (s) atomicAdd(&P.counts[k], s);
    }
}

// ---- fp32 filter of the all-pairs path (DESIGN.md 4.8b) -------------------------------
//
// Per pair ONE image in fp32, from the sequential fold the lower-triangular cell allows
// (tri_fold2): n_c = rint(df_z / c_z), then n_b from the remaining y, then n_a from the
// remaining x, u = df - n_c c - n_b b - n_a a.  Let B be the open brick of half-widths
// a_x / 2, b_y / 2, c_z / 2 and R = min(a_x, b_y, c_z) / 2.  Two points of B never differ by
// a lattice vector (compare z, then y, then x), so if the exact value of u has |u| < R it
// lies in B and every other image is at least R long.  The computed n are rint of rounded
// arguments, so the exact u lies within delta of B (tri_filter_prepare_frame bounds delta)
// and the true minimum is at least min(|u|, R - delta).  A frame is filtered when every
// pair the filter can bin lies well inside R - delta; then
//   - n in {-1, 0, 1}^3 (u is one of the reference's 27 images): the reference's minimum
//     is its fp64 d^2 of u, and the window of 4.1b decides the bin from the fp32 d^2;
//   - some |n_k| >= 2: u is not among the reference's images, its minimum is at least
//     R - delta - (fp64 error) > r_hi, and the pair goes to the above-range slot.  This is
//     the reference's quirk (its 27 images miss the shortest one), reproduced.
// Pairs inside the window are re-evaluated with tri_d2 (rdf_triclinic_kernel's bits).

struct TriFilter {         // per frame (tri_filter_prepare_frame)
    float nh[6];           // -a_x, -b_x, -b_y, -c_x, -c_y, -c_z
    float inv[3];          // (float)(1 / a_x), (float)(1 / b_y), (float)(1 / c_z)
    float offm;            // as FrameFilter::offm
    unsigned wlim;         // as FrameFilter::wlim; 0 = declined (rdf_triclinic_kernel's arithmetic)
};

// The fold of two pairs, d = b + a per axis (a: the negated group-1 coordinates).  Returns
// the packed fp32 |u|^2; w0 / w1 are the bits of n_a | n_b | n_c of each pair, whose bit
// 30 is set iff some |n_k| >= 2 (the n are small integers in float32).  Odd-symmetric bit
// for bit: (j, i) gives -df, -n, -u.
__device__ __forceinline__ f32x2 tri_fold2(f32x2 ax, f32x2 ay, f32x2 az, f32x2 bx, f32x2 by,
                                           f32x2 bz, const TriFilter &tf, unsigned &w0,
                                           unsigned &w1)
{
    const f32x2 magic = pk2(kMagicF, kMagicF), nmagic = pk2(-kMagicF, -kMagicF);
    const f32x2 dx = add2(bx, ax), dy = add2(by, ay), dz = add2(bz, az);
    const f32x2 nc = add2(fma2(dz, pk2(tf.inv[2], tf.inv[2]), magic), nmagic);
    const f32x2 uz = fma2(nc, pk2(tf.nh[5], tf.nh[5]), dz);
    const f32x2 y1 = fma2(nc, pk2(tf.nh[4], tf.nh[4]), dy);
    const f32x2 x1 = fma2(nc, pk2(tf.nh[3], tf.nh[3]), dx);
    const f32x2 nb = add2(fma2(y1, pk2(tf.inv[1], tf.inv[1]), magic), nmagic);
    const f32x2 uy = fma2(nb, pk2(tf.nh[2], tf.nh[2]), y1);
    const f32x2 x2 = fma2(nb, pk2(tf.nh[1], tf.nh[1]), x1);
    const f32x2 na = add2(fma2(x2, pk2(tf.inv[0], tf.inv[0]), magic), nmagic);
    const f32x2 ux = fma2(na, pk2(tf.nh[0], tf.nh[0]), x2);
    float a0, a1, b0, b1, c0, c1;
    upk2(na, a0, a1);
    upk2(nb, b0, b1);
    upk2(nc, c0, c1);
    w0 = __float_as_uint(a0) | __float_as_uint(b0) | __float_as_uint(c0);
    w1 = __float_as_uint(a1) | __float_as_uint(b1) | __float_as_uint(c1);
    return fma2(uz, uz, fma2(uy, uy, mul2(ux, ux)));
}

// Per-frame parameters from the cell and the extent keys of the WRAPPED coordinates
// (e1 / e2: {min x, y, z, max x, y, z} of the two groups).  info (optional): {R, delta, mu
// (the bound in bins, before the 1.25 margin of the window), reach}.  Bound, per axis, of
// the fp32 |u| against the reference's fp64 d of the same image:
//   fold: one rounding per FMA, on results bounded by the extents D and the tilts:
//         x: 2^-24 (X1 + X2 + H_x), y: 2^-24 (Y1 + H_y), z: 2^-24 H_z (H_k = half-width
//         + delta_k bounds |u_k|; X1, X2, Y1 bound the intermediate x', x'', y');
//   reference: its image sums in fp64, 3 / 2 / 1 roundings of terms below D_k + the
//         row of the cell (no eps_b term: the triclinic reference has no float32 inverse);
// then, as filter_prepare_frame: the 2-norm of those, the fp32 sum of squares, the measured
// sqrt.approx error, scale / offset / fma roundings, and the fp64 squares of the reference.
// delta_k: the rint argument's rounding, |arg| |inv_k h_kk - 1| h_kk, plus the fold's
// roundings before it.  The frame is filtered when reach = d_max + 1.25 mu / scale + 2 (fp64
// error of any image) + delta < R.
__host__ __device__ inline TriFilter tri_filter_prepare_frame(const TriBox &h, const unsigned *e1,
                                                              const unsigned *e2,
                                                              const FilterPrep &Q,
                                                              double *info = nullptr)
{
    const double e24 = 1.0 / 16777216.0, u53 = 1.0 / 9007199254740992.0;
    bool ok = true;
    double D[3];
    for (int k = 0; k < 3; ++k) {
        const float e4[4] = {ext_unkey(e1[k]), ext_unkey(e1[3 + k]), ext_unkey(e2[k]),
                             ext_unkey(e2[3 + k])};
        for (int q = 0; q < 4; ++q)
            if ((f32_bits(e4[q]) & 0x7f800000u) == 0x7f800000u) ok = false;
        D[k] = fmax(fmax((double)e4[3] - (double)e4[0], (double)e4[1] - (double)e4[2]), 0.0) *
               (1.0 + 2.0 * e24);
    }
    TriFilter tf;
    const float ia = (float)(1.0 / h.ax), ib = (float)(1.0 / h.by), ic = (float)(1.0 / h.cz);
    const double ea = fabs((double)ia * h.ax - 1.0), eb = fabs((double)ib * h.by - 1.0),
                 ec = fabs((double)ic * h.cz - 1.0);              // exact: 24 x 24 bits
    const double Nc = floor(D[2] * ic * (1.0 + 1e-12) + 0.5);
    const double Y1 = (D[1] + Nc * fabs(h.cy)) * (1.0 + e24);
    const double Nb = floor(Y1 * ib * (1.0 + 1e-12) + 0.5);
    const double X1 = (D[0] + Nc * fabs(h.cx)) * (1.0 + e24);
    const double X2 = (X1 + Nb * fabs(h.bx)) * (1.0 + e24);
    // the magic-number rint needs its arguments well inside 2^22
    if (!(D[2] * ic < 1048576.0 && Y1 * ib < 1048576.0 && X2 * ia < 1048576.0)) ok = false;
    const double dz = D[2] * ec, dy = Y1 * (eb + e24), dx = X2 * ea + e24 * (X1 + X2);
    const double delta = fmax(dx, fmax(dy, dz)) * (1.0 + 1e-6);
    const double Hx = 0.5 * h.ax + dx, Hy = 0.5 * h.by + dy, Hz = 0.5 * h.cz + dz;
    const double fx = e24 * (X1 + X2 + Hx) * (1.0 + 1e-6), fy = e24 * (Y1 + Hy) * (1.0 + 1e-6),
                 fz = e24 * Hz * (1.0 + 1e-6);
    const double rx = 3.0 * u53 * (D[0] + h.ax + fabs(h.bx) + fabs(h.cx)),
                 ry = 2.0 * u53 * (D[1] + h.by + fabs(h.cy)), rz = u53 * (D[2] + h.cz);
    const double a = sqrt((fx + rx) * (fx + rx) + (fy + ry) * (fy + ry) + (fz + rz) * (fz + rz));
    const double e_ref = sqrt(rx * rx + ry * ry + rz * rz);
    const double R = 0.5 * fmin(h.ax, fmin(h.by, h.cz));
    const double two_k = (double)(1u << Q.k);
    const double mu = Q.scale * (a + Q.d_max * (1.5 * e24 * 1.001 + Q.sqrt_err + 4.0 * u53)) +
                      e24 * Q.scale * Q.d_max * 1.001 + 1.0 / two_k + 1e-9;
    const double m = ceil(1.25 * mu * two_k) + 1.0;
    if (!(m >= 1.0) || !(2.0 * m + 1.0 < two_k / 8.0)) ok = false;
    const double reach = Q.d_max + 1.25 * mu / Q.scale + 2.0 * (e_ref + 4.0 * u53 * R) + delta;
    if (!(reach * (1.0 + 1e-9) < R)) ok = false;
    if (info) { info[0] = R; info[1] = delta; info[2] = mu; info[3] = reach; }
    tf.nh[0] = -(float)h.ax; tf.nh[1] = -(float)h.bx; tf.nh[2] = -(float)h.by;
    tf.nh[3] = -(float)h.cx; tf.nh[4] = -(float)h.cy; tf.nh[5] = -(float)h.cz;
    tf.inv[0] = ia; tf.inv[1] = ib; tf.inv[2] = ic;
    tf.offm = ok ? (float)(Q.offbase + m / two_k) : 0.f;
    tf.wlim = ok ? 2u * (unsigned)m + 1u : 0u;
    return tf;
}

// per frame {min x, y, z, max x, y, z} keys of the wrapped packed coordinates (ext set
// up by rdf_ext_init_kernel)
__global__ void __launch_bounds__(256)
    tri_extent_kernel(const float4 *__restrict__ p, int64_t npad, int n, unsigned *__restrict__ ext)
{
    __shared__ unsigned red[8][6];
    const int frame = blockIdx.y, tid = threadIdx.x;
    unsigned lo[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, hi[3] = {0u, 0u, 0u};
    for (int i = blockIdx.x * 256 + tid; i < n; i += gridDim.x * 256) {
        const float4 v = p[(int64_t)frame * npad + i];
        const unsigned k[3] = {ext_key(v.x), ext_key(v.y), ext_key(v.z)};
        for (int a = 0; a < 3; ++a) { lo[a] = min(lo[a], k[a]); hi[a] = max(hi[a], k[a]); }
    }
    for (int a = 0; a < 3; ++a) {
        const unsigned l = __reduce_min_sync(0xffffffffu, lo[a]);
        const unsigned h = __reduce_max_sync(0xffffffffu, hi[a]);
        if ((tid & 31) == 0) { red[tid >> 5][a] = l; red[tid >> 5][3 + a] = h; }
    }
    __syncthreads();
    if (tid < 6) {
        unsigned v = red[0][tid];
        for (int w = 1; w < 8; ++w) v = tid < 3 ? min(v, red[w][tid]) : max(v, red[w][tid]);
        if (tid < 3) { if (v != 0xffffffffu) atomicMin(&ext[frame * 6 + tid], v); }
        else if (v != 0u) atomicMax(&ext[frame * 6 + tid], v);
    }
}

constexpr int kTriIpt = 4;                       // i-particles per thread
constexpr int kTriTile = kThreads * kTriIpt;     // rows of an i-tile and of a j-tile
constexpr int kTriListCap = 2048;                // deferred rows per block and tile

struct TriFilterParams {
    const float4 *p1, *p2;
    int64_t pad1, pad2;            // multiples of kTriTile
    int n1, n2;
    const TriBox *boxes;
    const TriFilter *filt;
    const double *thr;
    int n_bins;
    BinGuess guess;
    int fast_bins;
    int same;
    int n_jchunks, jtiles_per_chunk, n_jtiles;
    FilterConst fc;                // the clamped layout (rdf_filter_configure)
    unsigned long long *counts;
    unsigned long long *fstats;    // PairParams::fstats; [9] frames filtered, [10] pairs
                                   // re-evaluated with the 27-image arithmetic
    unsigned long long *evals;
};

__host__ __device__ inline size_t tri_filter_smem_bytes(int n_bins, int hslots, int cb)
{
    return align16(sizeof(unsigned) * ((size_t)hslots << cb)) +
           align16(sizeof(double) * (n_bins + 1)) + 2 * kTriTile * sizeof(float4) +
           sizeof(unsigned) * (kTriListCap + 4);
}

// Exact re-evaluation of the kTriIpt pairs of one deferred row (thread te, tile row jj):
// every in-window pair of the row was added to the slot its fp32 coordinate gave; move it
// where tri_d2 puts it.  Pairs that are not one of the reference's images (|n_k| >= 2) went
// to the above-range slot, which is where the reference puts them too.  *n_exact (shared)
// counts the pairs evaluated with tri_d2.
template <bool EXCL, bool LOWER>
__device__ __noinline__ void tri_filter_fix(const TriFilterParams &P, int frame, int it,
                                                unsigned entry, const float4 *tile,
                                            const double *sT, unsigned hist32, unsigned weight,
                                            unsigned *n_exact)
{
    const TriFilter tf = P.filt[frame];
    const TriBox h = P.boxes[frame];
    const FilterConst fc = P.fc;
    const int te = (int)(entry >> 16), jj = (int)(entry & 0xffffu);
    const float4 pj = tile[jj];
    const float4 *f1 = P.p1 + (int64_t)frame * P.pad1;
    const unsigned span_l = LOWER ? fc.span : fc.cbits + fc.span;
    for (int ip = 0; ip < kTriIpt; ip += 2) {
        const int i0 = it * kTriTile + ip * kThreads + te, i1 = i0 + kThreads;
        const float4 a0 = f1[min(i0, P.n1 - 1)], a1 = f1[min(i1, P.n1 - 1)];
        unsigned w[2], uu[2];
        const f32x2 d2 = tri_fold2(pk2(-a0.x, -a1.x), pk2(-a0.y, -a1.y), pk2(-a0.z, -a1.z),
                                   pk2(pj.x, pj.x), pk2(pj.y, pj.y), pk2(pj.z, pj.z), tf, w[0],
                                   w[1]);
        filter_bin2<LOWER>(d2, fc.scale, tf.offm, fc.cbits, uu[0], uu[1]);
        for (int q = 0; q < 2; ++q) {
            const int i = q ? i1 : i0;
            const float4 a = q ? a1 : a0;
            const unsigned u = uu[q];
            if (i >= P.n1 || (w[q] & 0x40000000u)) continue;
            if (!(u < span_l) || !((u & ((1u << fc.k) - 1u)) < tf.wlim)) continue;
            if (EXCL && __float_as_int(a.w) == __float_as_int(pj.w)) continue;
            const unsigned seen = (LOWER ? u : u - fc.cbits) >> fc.k;
            const unsigned col = (unsigned)te & ((1u << fc.cb) - 1u);
            const double d2r = tri_d2(a.x, a.y, a.z, pj, h);
            const int slot = P.fast_bins ? slot_fast(d2r, sT, P.n_bins, P.guess)
                                         : slot_search(d2r, sT, P.n_bins);
            atomicAdd(n_exact, 1u);
            if (seen == (unsigned)slot) continue;
            red_shared(hist32 + 4u * ((seen << fc.cb) + col), 0u - weight);
            red_shared(hist32 + 4u * (((unsigned)slot << fc.cb) + col), weight);
        }
    }
}

// All pairs of tile pairs (i-tile, j-tile) in the fp32 fold; same group: the upper triangle
// of tile pairs, weight 2 off the diagonal (fold and reference are odd-symmetric), the
// diagonal tiles with every ordered pair, the self pairs included.  Tiles are staged with
// cp.async into two buffers; one block histogram of hslots x 2^cb columns (as
// rdf_filter_kernel); rows with an in-window pair go on the block's list, drained after each
// tile by tri_filter_fix (all rows of the tile if the list overflowed).  AUDIT: every pair also through tri_d2, disagreements among the
// certified pairs counted in fstats[2].
// (exclusion tags and the audit do not fit 128 registers: those instances take one block
// per SM's register file share, 255 registers)
template <bool EXCL, bool LOWER, bool AUDIT>
__global__ void __launch_bounds__(kThreads, EXCL || AUDIT ? 1 : 2)
    rdf_tri_filter_kernel(const __grid_constant__ TriFilterParams P)
{
    const int frame = blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const TriFilter tf = P.filt[frame];
    if (tf.wlim == 0u) {                  // declined: rdf_triclinic_kernel takes the frame
        if (blockIdx.x == 0 && tid == 0) atomicAdd(&P.fstats[4], 1ull);
        return;
    }
    if (blockIdx.x == 0 && tid == 0) atomicAdd(&P.fstats[9], 1ull);
    const int it = blockIdx.x / P.n_jchunks;
    const int jc = blockIdx.x - it * P.n_jchunks;
    int jt0 = jc * P.jtiles_per_chunk;
    const int jt1 = min(P.n_jtiles, jt0 + P.jtiles_per_chunk);
    if (P.same) jt0 = max(jt0, it);
    if (jt0 >= jt1) return;

    extern __shared__ __align__(16) unsigned char smem[];
    const int n_bins = P.n_bins;
    const FilterConst fc = P.fc;
    const int hwords = fc.hslots << fc.cb;
    unsigned *sH = reinterpret_cast<unsigned *>(smem);
    double *sT = reinterpret_cast<double *>(smem + align16(sizeof(unsigned) * hwords));
    float4 *sJ = reinterpret_cast<float4 *>(reinterpret_cast<unsigned char *>(sT) +
                                            align16(sizeof(double) * (n_bins + 1)));
    unsigned *sList = reinterpret_cast<unsigned *>(sJ + 2 * kTriTile);
    unsigned *sCount = sList + kTriListCap;
    for (int k = tid; k <= n_bins; k += kThreads) sT[k] = P.thr[k];
    for (int k = tid; k < hwords; k += kThreads) sH[k] = 0;
    if (tid == 0) { sCount[0] = 0; sCount[1] = 0; }

    const float4 *f1 = P.p1 + (int64_t)frame * P.pad1;
    const float4 *f2 = P.same ? f1 : P.p2 + (int64_t)frame * P.pad2;
    float xi[kTriIpt], yi[kTriIpt], zi[kTriIpt];
    int gi[kTriIpt];
    const int nv = P.n1 - it * kTriTile - tid;
#pragma unroll
    for (int ii = 0; ii < kTriIpt; ++ii) {
        // rows past the end of the group repeat the last particle with weight 0
        const float4 a = f1[min(it * kTriTile + ii * kThreads + tid, P.n1 - 1)];
        xi[ii] = a.x; yi[ii] = a.y; zi[ii] = a.z; gi[ii] = __float_as_int(a.w);
    }
    f32x2 nx[kTriIpt / 2], ny[kTriIpt / 2], nz[kTriIpt / 2];
#pragma unroll
    for (int ip = 0; ip < kTriIpt / 2; ++ip) {
        nx[ip] = pk2(-xi[2 * ip], -xi[2 * ip + 1]);
        ny[ip] = pk2(-yi[2 * ip], -yi[2 * ip + 1]);
        nz[ip] = pk2(-zi[2 * ip], -zi[2 * ip + 1]);
    }

    // word address of a slot as in rdf_filter_kernel (clamped body); a pair that is not one
    // of the reference's images gets bit 30 in t, which the clamp sends to the last slot
    const unsigned hist32 = (unsigned)__cvta_generic_to_shared(sH);
    const int tshift = fc.k - fc.cb - 2;
    const unsigned low = (4u << fc.cb) - 1u;
    const unsigned tmask = ((4u << (fc.cb + fc.lg)) - 1u) & ~low;
    const unsigned tmax = ((((LOWER ? 0u : fc.cbits) >> fc.k) + (unsigned)(fc.hslots - 1))
                           << (fc.cb + 2)) | low;
    const unsigned colbits = ((unsigned)lane & ((1u << fc.cb) - 1u)) << 2;
    const unsigned span_l = LOWER ? fc.span : fc.cbits + fc.span;
    const unsigned fmask = (1u << fc.k) - 1u;
    const float scale = fc.scale, offm = tf.offm;
    const unsigned wlim = tf.wlim;

    auto stage_tile = [&](int jt, int buf) {
        const float4 *src = f2 + (int64_t)jt * kTriTile;
        float4 *dst = sJ + buf * kTriTile;
#pragma unroll
        for (int q = 0; q < kTriIpt; ++q)
            __pipeline_memcpy_async(dst + q * kThreads + tid, src + q * kThreads + tid,
                                    sizeof(float4));
        __pipeline_commit();
    };
    stage_tile(jt0, 0);

    unsigned long long audit_bad = 0, audit_unc = 0;
    int buf = 0;
    for (int jt = jt0; jt < jt1; ++jt) {
        if (jt + 1 < jt1) {
            stage_tile(jt + 1, buf ^ 1);
            __pipeline_wait_prior(1);
        } else {
            __pipeline_wait_prior(0);
        }
        __syncthreads();
        const unsigned weight = (P.same && jt > it) ? 2u : 1u;
        unsigned wi[kTriIpt];
#pragma unroll
        for (int ii = 0; ii < kTriIpt; ++ii) wi[ii] = ii * kThreads < nv ? weight : 0u;
        const int jn = min(kTriTile, P.n2 - jt * kTriTile);
        const float4 *tile = sJ + buf * kTriTile;

        // two rows per trip where the registers allow it (ptxas -v: no spills)
        constexpr int kRows = 2;
#pragma unroll kRows
        for (int jj = 0; jj < jn; ++jj) {
            const float4 pj = tile[jj];
            unsigned vmin = 0xffffffffu;
#pragma unroll
            for (int ip = 0; ip < kTriIpt / 2; ++ip) {
                unsigned w[2], uu[2];
                const f32x2 d2 = tri_fold2(nx[ip], ny[ip], nz[ip], pk2(pj.x, pj.x),
                                           pk2(pj.y, pj.y), pk2(pj.z, pj.z), tf, w[0], w[1]);
                filter_bin2<LOWER>(d2, scale, offm, fc.cbits, uu[0], uu[1]);
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    const int ii = 2 * ip + q;
                    const unsigned u = uu[q];
                    vmin = min(vmin, u & fmask);
                    unsigned t = min(lop3_and_or(w[q], 0x40000000u, u >> tshift), tmax);
                    if (EXCL && gi[ii] == __float_as_int(pj.w)) t = tmax;
                    red_shared_hot(hist32 + lop3_and_or(t, tmask, colbits), wi[ii]);
                    if (AUDIT && wi[ii] && !(EXCL && gi[ii] == __float_as_int(pj.w))) {
                        const bool bad = (w[q] & 0x40000000u) != 0u;
                        const bool in = u < span_l && !bad;
                        const bool unc = in && (u & fmask) < wlim;
                        const double d2r = tri_d2(xi[ii], yi[ii], zi[ii], pj, P.boxes[frame]);
                        const int slot = slot_search(d2r, sT, n_bins);
                        // the slot the pair was added to, and the exact one
                        const unsigned fs = in ? ((LOWER ? u : u - fc.cbits) >> fc.k)
                                               : (unsigned)(fc.hslots - 1);
                        const bool counted = slot >= 1 && slot <= n_bins;
                        const bool fcounted = fs >= 1u && fs <= (unsigned)n_bins;
                        if (unc) ++audit_unc;
                        else if (fs != (unsigned)slot && (counted || fcounted)) ++audit_bad;
                    }
                }
            }
            if (vmin < wlim) {
                const unsigned entry = ((unsigned)tid << 16) | (unsigned)jj;
                const unsigned idx = atomicAdd(sCount, 1u);
                if (idx < (unsigned)kTriListCap) sList[idx] = entry;
            }
        }
        __syncthreads();
        const unsigned n_push = *sCount;
        const unsigned n_list = min(n_push, (unsigned)kTriListCap);
        if (n_push <= (unsigned)kTriListCap) {
            for (unsigned e = tid; e < n_list; e += kThreads)
                tri_filter_fix<EXCL, LOWER>(P, frame, it, sList[e], tile, sT, hist32, weight,
                                            sCount + 1);
        } else {
            // the list overflowed (rare): every thread re-evaluates all its rows of the tile,
            // tri_filter_fix acts on the in-window pairs only
            for (int jj = 0; jj < jn; ++jj)
                tri_filter_fix<EXCL, LOWER>(P, frame, it, ((unsigned)tid << 16) | (unsigned)jj,
                                            tile, sT, hist32, weight, sCount + 1);
        }
        if (tid == 0) {
            if (n_push) {
                atomicAdd(&P.fstats[0], (unsigned long long)n_list);
                if (n_push > n_list)
                    atomicAdd(&P.fstats[1], (unsigned long long)(n_push - n_list));
            }
            // pairs evaluated: the rows of the i-tile below n1 (nv of thread 0) x jn
            atomicAdd(P.evals, (unsigned long long)min(kTriTile, nv) * (unsigned long long)jn);
        }
        __syncthreads();
        if (tid == 0) *sCount = 0;
        buf ^= 1;
    }

    for (int k = tid; k < n_bins; k += kThreads) {
        unsigned s = 0;
        for (int q = 0; q < (1 << fc.cb); ++q)
            s += sH[((k + 1) << fc.cb) + ((q + tid) & ((1 << fc.cb) - 1))];
        if (s) atomicAdd(&P.counts[k], (unsigned long long)s);
    }
    if (tid == 0 && sCount[1]) atomicAdd(&P.fstats[10], (unsigned long long)sCount[1]);
    if (AUDIT) {
        if (audit_bad) atomicAdd(&P.fstats[2], audit_bad);
        if (audit_unc) atomicAdd(&P.fstats[3], audit_unc);
    }
}

template <bool EXCL, bool LOWER, bool AUDIT>
int launch_tri_filter(mdh_ctx *c, const TriFilterParams &P, dim3 grid)
{
    const size_t smem = tri_filter_smem_bytes(P.n_bins, P.fc.hslots, P.fc.cb);
    auto kern = rdf_tri_filter_kernel<EXCL, LOWER, AUDIT>;
    MDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kThreads, smem, c->stream>>>(P);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    return MDH_OK;
}

template <bool EXCL>
int launch_tri_filter_e(mdh_ctx *c, const TriFilterParams &P, dim3 grid, bool audit)
{
    if (P.fc.lower)
        return audit ? launch_tri_filter<EXCL, true, true>(c, P, grid)
                     : launch_tri_filter<EXCL, true, false>(c, P, grid);
    return audit ? launch_tri_filter<EXCL, false, true>(c, P, grid)
                 : launch_tri_filter<EXCL, false, false>(c, P, grid);
}

// ---- cell list in fractional coordinates ---------------------------------------------

constexpr int kTriShiftMax = 60;   // |k| per axis: k_j - k_i + wrap stays inside a signed byte

struct TriGrid {           // per frame
    TriBox h;
    int nc[3];
    int ncell;
};

// Fractional coordinates of a wrapped particle, s = r H^-1 (H lower triangular; the
// operation order is the one tri_grid_plan bounds), its cell in [0, n_k) per axis
// (clamped) and its lattice shift k = -floor(s): p = r + k H lies in the cell.  k is
// returned as packed signed bytes (axis a in byte 0).  A NaN coordinate lands in some
// cell; its pairs are NaN and binned nowhere.
__device__ __forceinline__ int tri_cell(const float4 &p, const TriGrid &g, unsigned &kcode)
{
    double sa, sb, sc;
    tri_frac(p.x, p.y, p.z, g.h, sa, sb, sc);
    const double s[3] = {sa, sb, sc};
    int c[3];
    kcode = 0u;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const double f = floor(s[k]);
        c[k] = min(max((int)__dmul_rn(__dsub_rn(s[k], f), (double)g.nc[k]), 0), g.nc[k] - 1);
        const int kk = (int)fmin(fmax(-f, (double)-kTriShiftMax), (double)kTriShiftMax);
        kcode |= ((unsigned)kk & 0xffu) << (8 * k);
    }
    return (c[2] * g.nc[1] + c[1]) * g.nc[0] + c[0];
}

// Coordinates outside the wrapped cell's brick widened by half its edges on either side:
// there the margin of tri_grid_plan does not bound the float32 rounding of dx (only
// finite coordinates a long way out of the cell, which tri_wrap_kernel cannot move in
// exactly, get here).  NaN is not "far".
__device__ __forceinline__ bool tri_far(const float4 &p, const TriBox &h)
{
    const double x = p.x, y = p.y, z = p.z;
    return x < -0.5 * h.ax || x > 1.5 * h.ax || y < -0.5 * h.by || y > 1.5 * h.by ||
           z < -0.5 * h.cz || z > 1.5 * h.cz;
}

// pass 1: cell and rank in the cell of every particle of the packed, wrapped array;
// far[frame] = 1 if the frame has a far coordinate
__global__ void __launch_bounds__(256)
    tri_bin_kernel(const float4 *__restrict__ pk, int64_t npad, int n,
                   const TriGrid *__restrict__ grids, int *__restrict__ cnt, int cstride,
                   int2 *__restrict__ keyrank, int *__restrict__ far)
{
    const int frame = blockIdx.y, tid = threadIdx.x;
    const TriGrid g = grids[frame];
    const float4 *src = pk + (int64_t)frame * npad;
    bool is_far = false;
    for (int64_t i0 = (int64_t)blockIdx.x * 256; i0 < n; i0 += (int64_t)gridDim.x * 256) {
        const int64_t i = i0 + tid;
        const unsigned active = __ballot_sync(0xffffffffu, i < n);
        if (i < n) {
            const float4 p = src[i];
            unsigned kc;
            const int cell = tri_cell(p, g, kc);
            is_far = is_far || tri_far(p, g.h);
            // warp-aggregated counter update, as cells_bin_kernel (rdf_cells.cu)
            const unsigned peers = __match_any_sync(active, cell);
            const int leader = __ffs(peers) - 1, lane = tid & 31;
            int base = 0;
            if (lane == leader)
                base = atomicAdd(&cnt[(int64_t)frame * cstride + cell], __popc(peers));
            base = __shfl_sync(peers, base, leader);
            keyrank[(int64_t)frame * n + i] =
                make_int2(cell, base + __popc(peers & ((1u << lane) - 1u)));
        }
    }
    if (__syncthreads_or(is_far) && tid == 0) far[frame] = 1;
}

// pass 3: packed -> cell-sorted float4 (x, y, z, exclusion block id) and shift codes
__global__ void __launch_bounds__(256)
    tri_scatter_kernel(const float4 *__restrict__ pk, int64_t npad, int n,
                       const TriGrid *__restrict__ grids, const int *__restrict__ start,
                       int cstride, const int2 *__restrict__ keyrank,
                       float4 *__restrict__ sorted, int *__restrict__ kcode)
{
    const int frame = blockIdx.y;
    const TriGrid g = grids[frame];
    const float4 *src = pk + (int64_t)frame * npad;
    const int *st = start + (int64_t)frame * cstride;
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * 256) {
        const float4 p = src[i];
        unsigned kc;
        tri_cell(p, g, kc);
        const int2 kr = keyrank[(int64_t)frame * n + i];
        const int64_t o = (int64_t)frame * n + st[kr.x] + kr.y;
        sorted[o] = p;
        kcode[o] = (int)kc;
    }
}

struct TriCellParams {
    const float4 *s1, *s2;        // cell-sorted particles, [G][n1], [G][n2]
    const int *k2;                // shift codes of s2 (tri_cell), [G][n2]
    int n1, n2;
    const int *start2;            // [G][cstride]
    int cstride;
    const TriGrid *grids;
    const int *far;               // [G]
    const double *thr;
    int n_bins;
    BinGuess guess;
    unsigned long long *counts;
    unsigned long long *evals;
    int half;                     // same group: half stencil, weight 2
};

__host__ inline size_t tri_cells_smem_bytes(int n_bins)
{
    return align16(sizeof(double) * (n_bins + 1)) +
           sizeof(unsigned) * kWarps * warp_hist_words(n_bins);
}

// One thread per particle i of the cell-sorted group 1, candidates from the 27 (same
// group: 13 forward + own) cells around i's cell.  A candidate j of the run that starts
// at neighbour cell index c_i + d (wrapped: c_i + d = c_j + w n, w in {-1, 0, 1}) is at
// the image m' = k_j - k_i + w of the reference's dx; if m' is not one of the reference's
// 27 images, the pair is out of range for both (tri_grid_plan).  The per-byte arithmetic
// of the packed shift codes gives m' with one VADD4.
template <bool EXCL, bool FAST>
__global__ void __launch_bounds__(kThreads, 2) rdf_tri_cells_kernel(const TriCellParams P)
{
    extern __shared__ __align__(16) unsigned char smem[];
    double *sT = reinterpret_cast<double *>(smem);
    unsigned *sH =
        reinterpret_cast<unsigned *>(smem + align16(sizeof(double) * (P.n_bins + 1)));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int frame = blockIdx.y;
    const int n_bins = P.n_bins;
    for (int k = tid; k <= n_bins; k += kThreads) sT[k] = P.thr[k];
    for (int k = tid; k < kWarps * warp_hist_words(n_bins); k += kThreads) sH[k] = 0;
    __syncthreads();

    unsigned *myhist = sH + warp * warp_hist_words(n_bins) + 1;
    const unsigned hist32 = (unsigned)__cvta_generic_to_shared(myhist);
    const unsigned trash32 = hist32 + 4u * (unsigned)(n_bins + lane);
    const BinGuess guess = P.guess;

    const TriGrid g = P.grids[frame];
    const TriBox h = g.h;
    const float4 *s1 = P.s1 + (int64_t)frame * P.n1;
    const float4 *s2 = P.s2 + (int64_t)frame * P.n2;
    const int *k2 = P.k2 + (int64_t)frame * P.n2;
    const int *start = P.start2 + (int64_t)frame * P.cstride;

    const int i = blockIdx.x * kThreads + tid;
    const bool valid = i < P.n1;
    const float4 pi = s1[min(i, P.n1 - 1)];
    const int gi = __float_as_int(pi.w);
    unsigned ki;
    const int my_cell = tri_cell(pi, g, ki);
    const int cx = my_cell % g.nc[0], cy = (my_cell / g.nc[0]) % g.nc[1],
              cz = my_cell / (g.nc[0] * g.nc[1]);
    const unsigned kneg = __vsub4(0u, ki);          // -k_i per byte
    unsigned long long my_evals = 0;

    auto bin = [&](double d2, bool keep, unsigned w) {
        if (FAST) {
            bool below;
            const int j = slot_fast_parts(d2, sT, n_bins, guess, below);
            unsigned a = (below ? hist32 - 4u : hist32) + 4u * (unsigned)j;
            if ((!below && j == n_bins) || !keep) a = trash32;
            red_shared(a, w);
        } else {
            const int slot = slot_search(d2, sT, n_bins);
            if (keep && (unsigned)(slot - 1) < (unsigned)n_bins) atomicAdd(&myhist[slot - 1], w);
        }
    };

    if (P.far[frame]) {
        // the margin does not hold for this frame: every ordered pair, all 27 images
        if (valid) {
            for (int j = 0; j < P.n2; ++j) {
                const float4 pj = s2[j];
                bin(tri_d2(pi.x, pi.y, pi.z, pj, h), !(EXCL && gi == __float_as_int(pj.w)),
                    1u);
            }
            my_evals += P.n2;
        }
    } else {
        // candidates s2[b, b + len); base = (w - k_i) per byte: m' = k_j + base
        auto sweep = [&](int b, int len, unsigned base, unsigned w_first, unsigned w_rest) {
            if (!valid) return;
            my_evals += len;
            for (int t = 0; t < len; ++t) {
                const float4 pj = __ldg(s2 + b + t);
                const unsigned m = __vadd4((unsigned)__ldg(k2 + b + t), base);
                // every byte in {-1, 0, 1} (byte 3 is 0)
                const bool ref_image = __vcmpleu4(__vadd4(m, 0x00010101u), 0x00020202u) ==
                                       0xffffffffu;
                const int ix = (int)(signed char)(m & 0xffu);
                const int iy = (int)(signed char)((m >> 8) & 0xffu);
                const int iz = (int)(signed char)((m >> 16) & 0xffu);
                auto sh = [](double v, int s) { return s == 0 ? 0.0 : (s > 0 ? v : -v); };
                const double d2 = tri_image_d2(
                    (double)__fsub_rn(pj.x, pi.x), (double)__fsub_rn(pj.y, pi.y),
                    (double)__fsub_rn(pj.z, pi.z), sh(h.ax, ix), sh(h.bx, iy), sh(h.by, iy),
                    sh(h.cx, iz), sh(h.cy, iz), sh(h.cz, iz));
                bin(d2, ref_image && !(EXCL && gi == __float_as_int(pj.w)),
                    t == 0 ? w_first : w_rest);
            }
        };
        auto wrap = [](int v, int n, int &w) {
            w = v < 0 ? -1 : (v >= n ? 1 : 0);
            return v - w * n;
        };
        auto code = [](int wa, int wb, int wc) {
            return ((unsigned)wa & 0xffu) | (((unsigned)wb & 0xffu) << 8) |
                   (((unsigned)wc & 0xffu) << 16);
        };
        // the three x-adjacent cells of row (cy + dy, cz + dz) are one contiguous range of
        // the sorted array, plus one more cell when the x stencil wraps around the cell
        auto sweep_row = [&](int dy, int dz, unsigned w) {
            int wb, wc;
            const int y = wrap(cy + dy, g.nc[1], wb), z = wrap(cz + dz, g.nc[2], wc);
            const int row = (z * g.nc[1] + y) * g.nc[0];
            const int xa = max(cx - 1, 0), xb = min(cx + 1, g.nc[0] - 1);
            const int b0 = start[row + xa];
            sweep(b0, start[row + xb + 1] - b0, __vadd4(code(0, wb, wc), kneg), w, w);
            if (cx == 0 || cx == g.nc[0] - 1) {
                const int wa = cx == 0 ? -1 : 1, xw = cx == 0 ? g.nc[0] - 1 : 0;
                const int bw = start[row + xw];
                sweep(bw, start[row + xw + 1] - bw, __vadd4(code(wa, wb, wc), kneg), w, w);
            }
        };
        // one cell along c (drop_axis = 2, tri_grid_plan_flat): the 9 cells (half: 4 + own)
        // of the (a, b) plane; the c component of every m' is 0
        const int dz_max = g.nc[2] > 1 ? 1 : 0;
        if (!P.half) {
            for (int dz = -dz_max; dz <= dz_max; ++dz)
                for (int dy = -1; dy <= 1; ++dy) sweep_row(dy, dz, 1u);
        } else {
            // forward offsets (dz, dy, dx) > 0 in lexicographic order, weight 2 for both
            // orders ((i, j) and (j, i) have the same 27-image minimum: float rounding is
            // odd-symmetric); the own cell from j = i: the self pair once
            if (dz_max)
                for (int dy = -1; dy <= 1; ++dy) sweep_row(dy, 1, 2u);
            sweep_row(1, 0, 2u);
            const int row = (cz * g.nc[1] + cy) * g.nc[0];
            int wa;
            const int xr = wrap(cx + 1, g.nc[0], wa);
            const int br = start[row + xr];
            sweep(br, start[row + xr + 1] - br, __vadd4(code(wa, 0, 0), kneg), 2u, 2u);
            sweep(i, start[row + cx + 1] - i, kneg, 1u, 2u);
        }
    }
    __syncthreads();
    for (int k = tid; k < n_bins; k += kThreads) {
        unsigned long long s = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) s += sH[w * warp_hist_words(n_bins) + 1 + k];
        if (s) atomicAdd(&P.counts[k], s);
    }
    for (int o = 16; o; o >>= 1) my_evals += __shfl_xor_sync(0xffffffffu, my_evals, o);
    if (lane == 0 && my_evals) atomicAdd(P.evals, my_evals);
}

template <bool EXCL, bool FAST>
int launch_tri_cells(mdh_ctx *c, const TriCellParams &P, dim3 grid)
{
    const size_t smem = tri_cells_smem_bytes(P.n_bins);
    auto kern = rdf_tri_cells_kernel<EXCL, FAST>;
    MDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kThreads, smem, c->stream>>>(P);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    return MDH_OK;
}

// ---- fp32 filter of the cell list (DESIGN.md 4.8c) -------------------------------------
//
// The cell list evaluates one image per candidate, m' = k_j - k_i + w (tri_grid_plan).
// With q = r + k H, the particle's position inside its cell (tri_cellq_kernel stores it
// rounded to float32), that image is q_j + (w H - q_i) exactly.  Per run the thread holds
// v = (float)(w H - q_i), so a candidate costs u = q_j + v (3 FADD), the fp32 sum of
// squares, sqrt.approx and the fixed-point bin coordinate of 4.1b.  A candidate with its
// coordinate inside the window (tri_cells_filter_prepare bounds its error against the
// reference's fp64 d^2 of the same image) is re-evaluated on the spot with the bits of
// rdf_tri_cells_kernel: tri_image_d2 of m' from the wrapped r, and the same slot lookup.

struct TriCellFilter {     // per frame, from the cell matrix alone (tri_cells_filter_prepare)
    float offm;            // as FrameFilter::offm
    unsigned wlim;         // as FrameFilter::wlim; 0 = declined
};

// q = r + k H of every cell-sorted particle, (q_x, q_y, q_z, shift code); bad[frame] = 1 if
// a q is not finite.  The sums in fp64 (the products k h are exact), one float32 rounding.
__global__ void __launch_bounds__(256)
    tri_cellq_kernel(const float4 *__restrict__ sorted, const int *__restrict__ kcode, int n,
                     const TriGrid *__restrict__ grids, float4 *__restrict__ q,
                     int *__restrict__ bad)
{
    const int frame = blockIdx.y;
    const TriBox h = grids[frame].h;
    bool nonfinite = false;
    for (int64_t i0 = (int64_t)blockIdx.x * 256; i0 < n; i0 += (int64_t)gridDim.x * 256) {
        const int64_t i = i0 + threadIdx.x;
        if (i < n) {
            const int64_t o = (int64_t)frame * n + i;
            const float4 p = sorted[o];
            const unsigned kc = (unsigned)kcode[o];
            const double ka = (signed char)(kc & 0xffu), kb = (signed char)((kc >> 8) & 0xffu),
                         kk = (signed char)((kc >> 16) & 0xffu);
            const float qx = (float)__dadd_rn(__dadd_rn(__dadd_rn((double)p.x, ka * h.ax),
                                                        kb * h.bx), kk * h.cx);
            const float qy = (float)__dadd_rn(__dadd_rn((double)p.y, kb * h.by), kk * h.cy);
            const float qz = (float)__dadd_rn((double)p.z, kk * h.cz);
            nonfinite = nonfinite || !isfinite(qx) || !isfinite(qy) || !isfinite(qz);
            q[o] = make_float4(qx, qy, qz, __uint_as_float(kc));
        }
    }
    if (__syncthreads_or(nonfinite) && threadIdx.x == 0) bad[frame] = 1;
}

struct TriCellFilterParams {
    TriCellParams c;              // the fp64 kernel's parameters (s1, s2: the wrapped r)
    const float4 *q1, *q2;        // (q, shift code) of the cell-sorted groups
    const int *bad;               // [G] (tri_cellq_kernel)
    const TriCellFilter *filt;    // [G]
    FilterConst fc;
    int fast_bins;
    unsigned long long *fstats;   // [4] declined frames, [9] frames filtered, [10] candidates
                                  // re-evaluated exactly, [2] / [3] audit
};

// rdf_tri_cells_kernel with the fp32 filter: one thread per particle i of the cell-sorted
// group 1, the same runs in the same order.  A frame the filter cannot certify (TriCellFilter
// wlim 0, a "far" coordinate, a non-finite q) is declined: every candidate then takes the
// exact arithmetic (far: every ordered pair with all 27 images), as in rdf_tri_cells_kernel.
// AUDIT: every certain candidate of a filtered frame is also evaluated exactly;
// disagreements in fstats[2], uncertain candidates in fstats[3].
template <bool EXCL, bool LOWER, bool AUDIT>
__global__ void __launch_bounds__(kThreads, 2)
    rdf_tri_cells_filter_kernel(const __grid_constant__ TriCellFilterParams F)
{
    const TriCellParams &P = F.c;
    extern __shared__ __align__(16) unsigned char smem[];
    double *sT = reinterpret_cast<double *>(smem);
    unsigned *sH =
        reinterpret_cast<unsigned *>(smem + align16(sizeof(double) * (P.n_bins + 1)));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int frame = blockIdx.y;
    const int n_bins = P.n_bins;
    for (int k = tid; k <= n_bins; k += kThreads) sT[k] = P.thr[k];
    for (int k = tid; k < kWarps * warp_hist_words(n_bins); k += kThreads) sH[k] = 0;
    __syncthreads();

    // word 0 of the warp's histogram: slot 0 (below the range); slot s: word s; words from
    // n_bins + 1 on: scratch, one per lane
    unsigned *myhist = sH + warp * warp_hist_words(n_bins) + 1;
    const unsigned hist32 = (unsigned)__cvta_generic_to_shared(myhist);
    const unsigned slot32 = hist32 - 4u;
    const unsigned trash32 = hist32 + 4u * (unsigned)(n_bins + lane);
    const BinGuess guess = P.guess;
    const bool fast = F.fast_bins != 0;

    const TriGrid g = P.grids[frame];
    const TriBox h = g.h;
    const TriCellFilter tf = F.filt[frame];
    const bool far = P.far[frame] != 0;
    const bool filtered = tf.wlim != 0u && !far && !F.bad[frame];
    if (blockIdx.x == 0 && tid == 0) atomicAdd(&F.fstats[filtered ? 9 : 4], 1ull);
    const float4 *s1 = P.s1 + (int64_t)frame * P.n1;
    const float4 *s2 = P.s2 + (int64_t)frame * P.n2;
    const float4 *q2 = F.q2 + (int64_t)frame * P.n2;
    const int *start = P.start2 + (int64_t)frame * P.cstride;

    const int i = blockIdx.x * kThreads + tid;
    const bool valid = i < P.n1;
    const int ic = min(i, P.n1 - 1);
    const float4 pi = s1[ic];
    const float4 qi = F.q1[(int64_t)frame * P.n1 + ic];
    const int gi = __float_as_int(pi.w);
    unsigned ki;
    const int my_cell = tri_cell(pi, g, ki);
    const int cx = my_cell % g.nc[0], cy = (my_cell / g.nc[0]) % g.nc[1],
              cz = my_cell / (g.nc[0] * g.nc[1]);
    const unsigned kneg = __vsub4(0u, ki);          // -k_i per byte
    unsigned long long my_evals = 0;
    unsigned n_exact = 0;
    unsigned long long audit_bad = 0, audit_unc = 0;

    const FilterConst fc = F.fc;
    const unsigned span_l = LOWER ? fc.span : fc.cbits + fc.span;
    const unsigned fmask = (1u << fc.k) - 1u;
    const float scale = fc.scale, offm = tf.offm;
    const unsigned wlim = tf.wlim;

    // the slot of an exact d^2 and its histogram word, as rdf_tri_cells_kernel bins
    auto exact_word = [&](double d2, bool keep, int &slot) -> unsigned {
        if (fast) {
            bool below;
            const int j = slot_fast_parts(d2, sT, n_bins, guess, below);
            slot = below ? j : j + 1;
            return ((!below && j == n_bins) || !keep) ? trash32 : slot32 + 4u * (unsigned)slot;
        }
        slot = slot_search(d2, sT, n_bins);
        return (keep && (unsigned)(slot - 1) < (unsigned)n_bins) ? slot32 + 4u * (unsigned)slot
                                                                  : trash32;
    };

    if (far) {
        // the margin does not hold for this frame: every ordered pair, all 27 images
        if (valid) {
            for (int j = 0; j < P.n2; ++j) {
                const float4 pj = s2[j];
                int slot;
                red_shared(exact_word(tri_d2(pi.x, pi.y, pi.z, pj, h), !(EXCL && gi ==
                                      __float_as_int(pj.w)), slot), 1u);
            }
            my_evals += P.n2;
        }
    } else {
        // candidates [b, b + len) of a run with wrap code wc; base = (w - k_i) per byte
        auto sweep = [&](int b, int len, unsigned wc, unsigned w_first, unsigned w_rest) {
            if (!valid) return;
            my_evals += len;
            const unsigned base = __vadd4(wc, kneg);
            const double wa = (signed char)(wc & 0xffu), wb = (signed char)((wc >> 8) & 0xffu),
                         ww = (signed char)((wc >> 16) & 0xffu);
            // v = (float)(w H - q_i): the lattice vector w H in fp64, one float32 rounding
            const float vx = (float)__dsub_rn(
                __dadd_rn(__dadd_rn(wa * h.ax, wb * h.bx), ww * h.cx), (double)qi.x);
            const float vy = (float)__dsub_rn(__dadd_rn(wb * h.by, ww * h.cy), (double)qi.y);
            const float vz = (float)__dsub_rn(ww * h.cz, (double)qi.z);
            for (int t = 0; t < len; ++t) {
                const float4 qj = __ldg(q2 + b + t);
                const unsigned m = __vadd4(__float_as_uint(qj.w), base);
                // every byte in {-1, 0, 1} (byte 3 is 0)
                const bool ref_image = __vcmpleu4(__vadd4(m, 0x00010101u), 0x00020202u) ==
                                       0xffffffffu;
                const bool keep =
                    ref_image &&
                    !(EXCL && gi == __ldg(reinterpret_cast<const int *>(s2 + b + t) + 3));
                const float ux = __fadd_rn(qj.x, vx), uy = __fadd_rn(qj.y, vy),
                            uz = __fadd_rn(qj.z, vz);
                const float d2 = __fmaf_rn(uz, uz, __fmaf_rn(uy, uy, __fmul_rn(ux, ux)));
                float s;
                asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s) : "f"(d2));
                const unsigned u = __float_as_uint(__fmaf_rn(s, scale, offm)) -
                                   (LOWER ? fc.cbits : 0u);
                const bool in = u < span_l && keep;
                const unsigned fs = (LOWER ? u : u - fc.cbits) >> fc.k;
                const unsigned wgt = t == 0 ? w_first : w_rest;
                // declined frame: every candidate exact
                const bool unc = !filtered || (in && (u & fmask) < wlim);
                if (unc || (AUDIT && filtered && keep)) {
                    // exact: the image m' of the reference's dx, rdf_tri_cells_kernel's bits
                    const float4 pj = __ldg(s2 + b + t);
                    const int ix = (int)(signed char)(m & 0xffu);
                    const int iy = (int)(signed char)((m >> 8) & 0xffu);
                    const int iz = (int)(signed char)((m >> 16) & 0xffu);
                    auto sh = [](double v, int q) { return q == 0 ? 0.0 : (q > 0 ? v : -v); };
                    const double d2r = tri_image_d2(
                        (double)__fsub_rn(pj.x, pi.x), (double)__fsub_rn(pj.y, pi.y),
                        (double)__fsub_rn(pj.z, pi.z), sh(h.ax, ix), sh(h.bx, iy),
                        sh(h.by, iy), sh(h.cx, iz), sh(h.cy, iz), sh(h.cz, iz));
                    int slot;
                    const unsigned a = exact_word(d2r, keep, slot);
                    if (unc) {
                        red_shared(a, wgt);
                        ++n_exact;
                        if (AUDIT && filtered) ++audit_unc;
                        continue;
                    }
                    if (AUDIT) {
                        const bool counted = keep && slot >= 1 && slot <= n_bins;
                        const bool fcounted = in && fs >= 1u && fs <= (unsigned)n_bins;
                        if ((counted || fcounted) && (!counted || !fcounted || fs != (unsigned)slot))
                            ++audit_bad;
                    }
                }
                red_shared(in && fs <= (unsigned)n_bins ? slot32 + 4u * fs : trash32, wgt);
            }
        };
        auto wrap = [](int v, int n, int &w) {
            w = v < 0 ? -1 : (v >= n ? 1 : 0);
            return v - w * n;
        };
        auto code = [](int wa, int wb, int wc) {
            return ((unsigned)wa & 0xffu) | (((unsigned)wb & 0xffu) << 8) |
                   (((unsigned)wc & 0xffu) << 16);
        };
        auto sweep_row = [&](int dy, int dz, unsigned w) {
            int wb, wc;
            const int y = wrap(cy + dy, g.nc[1], wb), z = wrap(cz + dz, g.nc[2], wc);
            const int row = (z * g.nc[1] + y) * g.nc[0];
            const int xa = max(cx - 1, 0), xb = min(cx + 1, g.nc[0] - 1);
            const int b0 = start[row + xa];
            sweep(b0, start[row + xb + 1] - b0, code(0, wb, wc), w, w);
            if (cx == 0 || cx == g.nc[0] - 1) {
                const int wa = cx == 0 ? -1 : 1, xw = cx == 0 ? g.nc[0] - 1 : 0;
                const int bw = start[row + xw];
                sweep(bw, start[row + xw + 1] - bw, code(wa, wb, wc), w, w);
            }
        };
        const int dz_max = g.nc[2] > 1 ? 1 : 0;
        if (!P.half) {
            for (int dz = -dz_max; dz <= dz_max; ++dz)
                for (int dy = -1; dy <= 1; ++dy) sweep_row(dy, dz, 1u);
        } else {
            if (dz_max)
                for (int dy = -1; dy <= 1; ++dy) sweep_row(dy, 1, 2u);
            sweep_row(1, 0, 2u);
            const int row = (cz * g.nc[1] + cy) * g.nc[0];
            int wa;
            const int xr = wrap(cx + 1, g.nc[0], wa);
            const int br = start[row + xr];
            sweep(br, start[row + xr + 1] - br, code(wa, 0, 0), 2u, 2u);
            sweep(i, start[row + cx + 1] - i, 0u, 1u, 2u);
        }
    }
    __syncthreads();
    for (int k = tid; k < n_bins; k += kThreads) {
        unsigned long long s = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) s += sH[w * warp_hist_words(n_bins) + 1 + k];
        if (s) atomicAdd(&P.counts[k], s);
    }
    for (int o = 16; o; o >>= 1) my_evals += __shfl_xor_sync(0xffffffffu, my_evals, o);
    if (lane == 0 && my_evals) atomicAdd(P.evals, my_evals);
    if (filtered) {
        n_exact = __reduce_add_sync(0xffffffffu, n_exact);
        if (lane == 0 && n_exact) atomicAdd(&F.fstats[10], (unsigned long long)n_exact);
    }
    if (AUDIT) {
        if (audit_bad) atomicAdd(&F.fstats[2], audit_bad);
        if (audit_unc) atomicAdd(&F.fstats[3], audit_unc);
    }
}

template <bool EXCL, bool LOWER, bool AUDIT>
int launch_tri_cells_filter(mdh_ctx *c, const TriCellFilterParams &F, dim3 grid)
{
    const size_t smem = tri_cells_smem_bytes(F.c.n_bins);
    auto kern = rdf_tri_cells_filter_kernel<EXCL, LOWER, AUDIT>;
    MDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, kThreads, smem, c->stream>>>(F);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    return MDH_OK;
}

template <bool EXCL>
int launch_tri_cells_filter_e(mdh_ctx *c, const TriCellFilterParams &F, dim3 grid, bool audit)
{
    if (F.fc.lower)
        return audit ? launch_tri_cells_filter<EXCL, true, true>(c, F, grid)
                     : launch_tri_cells_filter<EXCL, true, false>(c, F, grid);
    return audit ? launch_tri_cells_filter<EXCL, false, true>(c, F, grid)
                 : launch_tri_cells_filter<EXCL, false, false>(c, F, grid);
}

// ---- grid planner (host, no device) ------------------------------------------------------
//
// Why one image per candidate gives the reference's counts.  Cells are cut in fractional
// coordinates, n_k >= 3 per axis, and every cell's perpendicular width w_k / n_k is at least
// r + M (r = sqrt(U), U the last squared threshold).  Let p_i = r_i + k_i H be particle i's
// position in the cell (tri_cell).  The 3x3x3 block of cells around p_i's cell spans less
// than one period per axis (n_k >= 3), so exactly one lattice image of j lies in it,
// p_j + w H = r_j + m' H, m' = k_j - k_i + w; every other image of j -- and every image of
// a j whose cell is not in the block -- differs from p_i in some fractional coordinate k by
// at least 1 / n_k - 2 eps_k (eps_k: error of the computed fractional coordinates), i.e. is
// at least w_k / n_k - 2 eps_k w_k >= r + M - 2 eps_k w_k away.  The reference computes
// d^2 from dx~ = (float)(r_j - r_i) instead of the exact difference, and rounds the image
// sums and squares in fp64.  With
//   M = max_k 2 eps_k w_k            (cell assignment)
//     + e_f                          (dx~: |dx~ - dx| <= 2^-24 |dx| per component)
//     + e_d                          (fp64 image sums)
//     + 1e-5 r                       (fp64 squares and sums of d^2, r = sqrt(U) rounding)
// every image but m' has a computed d^2 above U, so min27 <= U implies min27 = d^2(m') and
// m' in {-1, 0, 1}^3; otherwise both are above U and neither is counted.  The kernel
// computes d^2(m') with tri_image_d2 (same operations, same bits).
//
// Bounds.  Unless a frame is "far" (tri_far; such frames take the 27-image arithmetic for
// every pair), wrapped coordinates lie within [-E_k / 2, 3 E_k / 2], E = (a_x, b_y, c_z),
// so |dx_k| <= 2 E_k and e_f = 2^-24 * 2 |E|.  Image sums: three fp64 additions of terms
// below 2 E_k + sum_k' |H_k'k| per component: e_d = 4 * 2^-53 |that vector|.  eps_k follows
// the operations of tri_cell step by step (every rounding: 2^-53 of the bound on its
// result), doubled to absorb second-order terms; fractional part and product with n_k add
// 2^-53.  The shifts k are bounded by the magnitude bounds of s (|k| <= |s| + 1); a cell
// whose bound exceeds kTriShiftMax gets no grid.
struct TriPlan {
    int nc[3];        // cells per axis (0: fewer than 3 fit)
    int fit[3];       // cells per axis before the cap and the occupancy rule
    double margin;    // M
    bool c_ok;        // flat grid (tri_grid_plan_flat): c_z >= r + M
};

int tri_check_matrix(const float *m9, double r_hi)
{
    MDH_REQUIRE(m9 != nullptr, MDH_EINVAL, "rdf: cell matrix is NULL");
    MDH_REQUIRE(m9[1] == 0.f && m9[2] == 0.f && m9[5] == 0.f, MDH_EINVAL,
                "rdf: the cell matrix is not lower triangular");
    for (int k = 0; k < 9; ++k)
        MDH_REQUIRE(std::isfinite(m9[k]), MDH_EINVAL, "rdf: the cell matrix is not finite");
    MDH_REQUIRE(m9[0] > 0.f && m9[4] > 0.f && m9[8] > 0.f, MDH_EINVAL,
                "rdf: the cell matrix is not a valid cell");
    MDH_REQUIRE(r_hi >= 0.0 && std::isfinite(r_hi), MDH_EINVAL, "rdf: invalid r_max");
    return MDH_OK;
}

// cells per axis from the (lower bounds of the) widths w: w_k / n_k >= width exactly, at
// most 160, then fewer until about 2 particles per cell remain or the axes are down to 3;
// `axes` axes are cut (3, or 2 with one cell along c)
void tri_cells_per_axis(const double *w, double width, int64_t n_max, int axes, TriPlan &out)
{
    double ncell = 1;
    for (int k = 0; k < axes; ++k) {
        double f = std::floor(w[k] / width);
        while (f >= 1.0 && w[k] / f < width) f -= 1.0;     // w_k / n_k >= r + M exactly
        out.fit[k] = (int)std::min(f, 1e6);
        out.nc[k] = std::min(out.fit[k], 160);
        ncell *= out.nc[k];
    }
    for (int k = axes; k < 3; ++k) out.fit[k] = out.nc[k] = 1;
    if (std::min({out.nc[0], out.nc[1], axes == 3 ? out.nc[2] : 3}) < 3) {
        for (int k = 0; k < 3; ++k) out.nc[k] = 0;
        return;
    }
    // keep at least ~2 particles per cell on average
    const double want = std::max(axes == 3 ? 27.0 : 9.0, (double)n_max / 2.0);
    while (ncell > want) {
        int kmax = 0;
        for (int k = 1; k < axes; ++k) if (out.nc[k] > out.nc[kmax]) kmax = k;
        if (out.nc[kmax] <= 3) break;
        ncell = ncell / out.nc[kmax] * (out.nc[kmax] - 1);
        out.nc[kmax]--;
    }
}

int tri_grid_plan(const float *m9, double r_hi, int64_t n_max, TriPlan &out)
{
    if (int rc = tri_check_matrix(m9, r_hi)) return rc;
    out.c_ok = true;
    const double ax = m9[0], bx = m9[3], by = m9[4], cx = m9[6], cy = m9[7], cz = m9[8];
    const double u = 1.0 / 9007199254740992.0;           // 2^-53
    // magnitude bounds (B) and absolute errors (e) of the steps of tri_cell
    const double X = 1.5 * ax, Y = 1.5 * by, Z = 1.5 * cz;
    const double Bc = Z / cz * (1 + u), ec = u * Bc;                     // s_c = z / c_z
    const double Bp1 = Bc * std::fabs(cy) * (1 + u), ep1 = std::fabs(cy) * ec + u * Bp1;
    const double Bt = (Y + Bp1) * (1 + u), et = ep1 + u * Bt;            // y - s_c c_y
    const double Bb = Bt / by * (1 + u), eb = et / by + u * Bb;          // s_b
    const double Bq1 = Bb * std::fabs(bx) * (1 + u), eq1 = std::fabs(bx) * eb + u * Bq1;
    const double Br1 = (X + Bq1) * (1 + u), er1 = eq1 + u * Br1;         // x - s_b b_x
    const double Bq2 = Bc * std::fabs(cx) * (1 + u), eq2 = std::fabs(cx) * ec + u * Bq2;
    const double Br2 = (Br1 + Bq2) * (1 + u), er2 = er1 + eq2 + u * Br2; // ... - s_c c_x
    const double Ba = Br2 / ax * (1 + u), ea = er2 / ax + u * Ba;        // s_a
    const double eps[3] = {2 * ea + u, 2 * eb + u, 2 * ec + u};
    const double B[3] = {Ba, Bb, Bc};
    // perpendicular widths V / |b x c|, V / |c x a|, c_z (lower bounds)
    const double w[3] = {
        ax * by * cz / std::sqrt(by * cz * by * cz + bx * cz * bx * cz +
                                 (bx * cy - by * cx) * (bx * cy - by * cx)) * (1 - 1e-12),
        by * cz / std::sqrt(cy * cy + cz * cz) * (1 - 1e-12), cz};
    const double E = std::sqrt(ax * ax + by * by + cz * cz);
    const double rows[3] = {2 * ax + ax + std::fabs(bx) + std::fabs(cx),
                            2 * by + by + std::fabs(cy), 2 * cz + cz};
    const double e_f = 2.0 * E / 16777216.0;
    const double e_d = 4 * u * std::sqrt(rows[0] * rows[0] + rows[1] * rows[1] + rows[2] * rows[2]);
    double e_a = 0.0;
    for (int k = 0; k < 3; ++k) e_a = std::max(e_a, 2.0 * eps[k] * w[k]);
    out.margin = e_a + e_f + e_d + 1e-5 * r_hi;
    const double width = r_hi + out.margin;
    bool shifts_ok = true;
    for (int k = 0; k < 3; ++k) shifts_ok = shifts_ok && B[k] + 1.0 <= kTriShiftMax;
    tri_cells_per_axis(w, width, n_max, 3, out);
    if (!shifts_ok)
        for (int k = 0; k < 3; ++k) out.nc[k] = 0;
    return MDH_OK;
}

// ---- the flat grid of drop_axis = 2 ------------------------------------------------------
//
// The zeroed z stays exactly 0 through tri_wrap_kernel (s = floor(0 / c_z) = 0, and the a
// and b rows have no z component), so every wrapped particle lies in the plane z = 0, has
// s_c = 0 exactly in tri_cell and the shift k_c = 0.  The grid has one cell along c and the
// stencil is the 9 cells of the (a, b) plane, so every m' has m'_c = 0.
//
// Images with a c shift iz != 0.  dx_2 = (float)(0 - 0) = 0, so the reference's
// r_z = dx_2 + c_z iz = +-c_z exactly, c_z^2 is exact in fp64 (24-bit x 24-bit), and the
// computed d^2 = fl(fl(r_x^2 + r_y^2) + c_z^2) >= c_z^2 (rounding is monotone, the other
// terms are >= 0).  With c_z >= r + M > r such an image is above U: never counted, and
// never the 27-image minimum when that is in range.
//
// Images with iz = 0.  These and p_i all lie in the plane, so the argument of tri_grid_plan
// holds in two dimensions with the in-plane widths of the (a, b) lattice, w_a = a_x b_y / |b|
// and w_b = b_y (at least the three-dimensional perpendicular widths): per axis a, b the
// 3 x 3 block of cells around p_i's cell spans less than one period (n_k >= 3), every image
// but m' differs from p_i in s_a or s_b by at least 1 / n_k - 2 eps_k, i.e. lies at least
// r + M - 2 eps_k w_k away.  The terms of M, for z = 0 and (not "far") x in
// [-a_x / 2, 3 a_x / 2], y in [-b_y / 2, 3 b_y / 2]:
//   eps_b, eps_a   tri_cell with s_c = 0 exactly: s_b = y / b_y (one rounding) and
//                  s_a = (x - s_b b_x) / a_x (the term s_c c_x is 0, exact); each rounding
//                  2^-53 of the bound on its result, doubled, plus 2^-53 for the
//                  fractional part and the product with n_k (as tri_grid_plan);
//   e_f            2^-24 |dx| with |dx_k| <= 2 E_k, E = (a_x, b_y): 2^-23 |E| (dx_2 = 0);
//   e_d            the image sums (dx_0 + a_x ia) + b_x ib (+ 0, exact) and dx_1 + b_y ib:
//                  4 * 2^-53 |(3 a_x + |b_x|, 3 b_y)|;
//   1e-5 r         fp64 squares and sums of d^2, as tri_grid_plan.
// M = max(2 eps_a w_a, 2 eps_b w_b) + e_f + e_d + 1e-5 r; cells of width >= r + M per kept
// axis, and c_ok = (c_z >= r + M).  (c_z > r alone would do by the argument above; the plan
// asks the same width of all three axes.)  drop_axis 0 or 1 gets no grid: the wrap then
// moves the zeroed coordinate again, and the particles do not lie in a lattice plane.
int tri_grid_plan_flat(const float *m9, double r_hi, int64_t n_max, TriPlan &out)
{
    if (int rc = tri_check_matrix(m9, r_hi)) return rc;
    const double ax = m9[0], bx = m9[3], by = m9[4], cz = m9[8];
    const double u = 1.0 / 9007199254740992.0;           // 2^-53
    const double X = 1.5 * ax, Y = 1.5 * by;
    const double Bb = Y / by * (1 + u), eb = u * Bb;                     // s_b = y / b_y
    const double Bq1 = Bb * std::fabs(bx) * (1 + u), eq1 = std::fabs(bx) * eb + u * Bq1;
    const double Br1 = (X + Bq1) * (1 + u), er1 = eq1 + u * Br1;         // x - s_b b_x
    const double Ba = Br1 / ax * (1 + u), ea = er1 / ax + u * Ba;        // s_a
    const double eps[2] = {2 * ea + u, 2 * eb + u};
    const double B[2] = {Ba, Bb};
    const double w[2] = {ax * by / std::sqrt(bx * bx + by * by) * (1 - 1e-12), by};
    const double e_f = 2.0 * std::sqrt(ax * ax + by * by) / 16777216.0;
    const double rx = 3 * ax + std::fabs(bx), ry = 3 * by;
    const double e_d = 4 * u * std::sqrt(rx * rx + ry * ry);
    const double e_a = std::max(2.0 * eps[0] * w[0], 2.0 * eps[1] * w[1]);
    out.margin = e_a + e_f + e_d + 1e-5 * r_hi;
    const double width = r_hi + out.margin;
    out.c_ok = cz >= width;
    tri_cells_per_axis(w, width, n_max, 2, out);
    if (!(B[0] + 1.0 <= kTriShiftMax && B[1] + 1.0 <= kTriShiftMax))
        for (int k = 0; k < 3; ++k) out.nc[k] = 0;
    return MDH_OK;
}

// Per-frame parameters of the cell-list filter (rdf_tri_cells_filter_kernel) from the cell
// matrix alone: no extent pass, valid for every frame that is not "far" (tri_far; those
// are declined on the device).  info (optional): {A, a, mu} (A: the fp32 evaluation's
// absolute error, a: A + e_f + e_d, mu: the bound in bins before the 1.25 margin).
//
// Rows of the cell: R_x = a_x + |b_x| + |c_x|, R_y = b_y + |c_y|, R_z = c_z.  The fractional
// coordinates of q = r + k H are s + k = s - floor(s~) in [-eps, 1 + eps] (s~ the computed
// s, eps < 1e-12 whenever the plan gives a grid), so |q_k| <= Q_k = R_k (1 + 1e-9).  Per
// axis, against the exact image dx + m' H = q_j + w H - q_i:
//   q      tri_cellq_kernel: three fp64 sums of terms below 1.5 E_k + 60 R_k (non-far r,
//          |k| <= kTriShiftMax), one float32 rounding: e_q = 2^-24 Q_k + 3 u (1.5 E_k + 60 R_k);
//   v      (float)(w H - q~_i): three fp64 sums below R_k + Q_k, one float32 rounding of a
//          result below R_k + Q_k (1 + 2^-24): e_v = 2^-24 (R_k + Q_k) (1 + 2^-23) +
//          3 u (R_k + Q_k);
//   A_k = 2 e_q + e_v (q_i and q_j are both rounded);
//   u      the FADD q~_j + v~ rounds once: 2^-24 |u_k|, relative, in the d_max term below.
// Reference side (as tri_grid_plan): e_f = 2^-23 |E| for its float32 dx, e_d = 4 u |rows|
// for its fp64 image sums, 4 u relative for its fp64 squares.  Then as
// tri_filter_prepare_frame: the fp32 sum of squares (1.5 2^-24 relative on d), the final
// add (2^-24), the measured sqrt.approx error, the scale / offset FMA (2^-24 d_max scale),
// the fixed-point resolution 2^-k.  u = 2^-53, E = (a_x, b_y, c_z).
TriCellFilter tri_cells_filter_prepare(const float *m9, const FilterPrep &Q,
                                       double *info = nullptr)
{
    const double e24 = 1.0 / 16777216.0, u = 1.0 / 9007199254740992.0;
    const double ax = m9[0], bx = m9[3], by = m9[4], cx = m9[6], cy = m9[7], cz = m9[8];
    const double R[3] = {ax + std::fabs(bx) + std::fabs(cx), by + std::fabs(cy), cz};
    const double E[3] = {ax, by, cz};
    double A2 = 0.0;
    for (int k = 0; k < 3; ++k) {
        const double Qk = R[k] * (1.0 + 1e-9);
        const double eq = e24 * Qk + 3.0 * u * (1.5 * E[k] + kTriShiftMax * R[k]);
        const double ev = e24 * (R[k] + Qk) * (1.0 + 2.0 * e24) + 3.0 * u * (R[k] + Qk);
        const double A = 2.0 * eq + ev;
        A2 += A * A;
    }
    const double A = std::sqrt(A2) * (1.0 + 1e-9);
    const double rows[3] = {2 * ax + ax + std::fabs(bx) + std::fabs(cx),
                            2 * by + by + std::fabs(cy), 2 * cz + cz};
    const double e_f = 2.0 * std::sqrt(ax * ax + by * by + cz * cz) * e24;
    const double e_d = 4 * u * std::sqrt(rows[0] * rows[0] + rows[1] * rows[1] + rows[2] * rows[2]);
    const double a = (A + e_f + e_d) * (1.0 + 1e-9);
    const double two_k = (double)(1u << Q.k);
    const double mu = Q.scale * (a + Q.d_max * (2.5 * e24 * 1.001 + Q.sqrt_err + 4.0 * u)) +
                      e24 * Q.scale * Q.d_max * 1.001 + 1.0 / two_k + 1e-9;
    const double m = std::ceil(1.25 * mu * two_k) + 1.0;
    const bool ok = m >= 1.0 && 2.0 * m + 1.0 < two_k / 8.0;
    if (info) { info[0] = A; info[1] = a; info[2] = mu; }
    TriCellFilter tf;
    tf.offm = ok ? (float)(Q.offbase + m / two_k) : 0.f;
    tf.wlim = ok ? 2u * (unsigned)m + 1u : 0u;
    return tf;
}

}  // namespace

int rdf_triclinic_grid_impl(const float *cell9, double r_hi, int64_t n_max, int32_t *nc,
                            double *margin)
{
    MDH_REQUIRE(nc != nullptr && margin != nullptr, MDH_EINVAL, "triclinic_grid: NULL output");
    TriPlan pl;
    if (int rc = tri_grid_plan(cell9, r_hi, n_max, pl)) return rc;
    for (int k = 0; k < 3; ++k) nc[k] = pl.nc[k];
    *margin = pl.margin;
    return MDH_OK;
}

int rdf_ortho_grid_plan(const double box[3], double r_hi, int64_t n_max, int drop_axis,
                        int nc[3]);                           // rdf_cells.cu

int rdf_cells_grid_impl(const float *cell9, double r_hi, int64_t n_max, int drop_axis,
                        int32_t *nc, double *margin)
{
    MDH_REQUIRE(nc != nullptr && margin != nullptr, MDH_EINVAL, "cells_grid: NULL output");
    MDH_REQUIRE(drop_axis >= -1 && drop_axis <= 2, MDH_EINVAL, "rdf: invalid drop_axis");
    if (int rc = tri_check_matrix(cell9, r_hi)) return rc;
    if (cell9[3] == 0.f && cell9[6] == 0.f && cell9[7] == 0.f) {
        // orthorhombic: the grid of mdh_rdf_accumulate (rdf_cells_accumulate)
        const double box[3] = {cell9[0], cell9[4], cell9[8]};
        int g[3];
        const bool ok = rdf_ortho_grid_plan(box, r_hi, n_max, drop_axis, g) < 0;
        for (int k = 0; k < 3; ++k) nc[k] = ok ? g[k] : 0;
        *margin = r_hi * 1.00001 - r_hi;
        return MDH_OK;
    }
    MDH_REQUIRE(drop_axis < 0 || drop_axis == 2, MDH_EINVAL,
                "rdf: the triclinic cell list takes drop_axis 2 (z) only; drop_axis %d runs "
                "through all pairs", drop_axis);
    TriPlan pl;
    if (int rc = drop_axis == 2 ? tri_grid_plan_flat(cell9, r_hi, n_max, pl)
                                : tri_grid_plan(cell9, r_hi, n_max, pl))
        return rc;
    MDH_REQUIRE(pl.c_ok, MDH_EINVAL,
                "rdf: the triclinic cell list with drop_axis 2 needs c_z >= r_max + %g "
                "(c_z = %g)", pl.margin, (double)cell9[8]);
    for (int k = 0; k < 3; ++k) nc[k] = pl.nc[k];
    *margin = pl.margin;
    return MDH_OK;
}

namespace {

// Device layout of the scratch (RdfState::cell) on this path:
//   cell[0] TriBox[F]   cell[5] TriGrid[F]   cell[1] int cnt[2][G][cstride] | far[G]
//   cell[2] int start[2][G][cstride]   cell[3] int2 keyrank[G][n1]   cell[4] float4 sorted1
//   cell[6] int kcode[G][n1] | [G][n2]   cell[7] keyrank2   cell[8] sorted2   cell[9] evals
//   fp32 filter (filt not empty): cell[1] also bad[G] after far[G], cell[10] float4 q1[G][n1],
//   cell[11] float4 q2[G][n2], R.filt TriCellFilter[F]
int tri_cells_accumulate(mdh_ctx *c, const std::vector<TriGrid> &grids, int64_t pad1,
                         int64_t pad2, const std::vector<TriCellFilter> &filt, bool audit)
{
    RdfState &R = c->rdf;
    const int n_frames = (int)grids.size();
    int ncell_max = 0;
    for (const TriGrid &g : grids) ncell_max = std::max(ncell_max, g.ncell);
    const int cstride = ncell_max + 1;
    DevBuf &d_grids = R.cell[5];
    if (int rc = d_grids.reserve(sizeof(TriGrid) * n_frames)) return rc;
    // pageable source: the runtime stages it before returning
    MDH_CUDA(cudaMemcpyAsync(d_grids.p, grids.data(), sizeof(TriGrid) * n_frames,
                             cudaMemcpyHostToDevice, c->stream));
    const bool use_filter = !filt.empty();
    if (use_filter) {
        if (int rc = R.filt.reserve(sizeof(TriCellFilter) * n_frames)) return rc;
        MDH_CUDA(cudaMemcpyAsync(R.filt.p, filt.data(), sizeof(TriCellFilter) * n_frames,
                                 cudaMemcpyHostToDevice, c->stream));
    }
    // frames per group: what one group reads and writes between the passes should stay
    // in L2 (the rule of rdf_cells_accumulate; 44 bytes per particle here)
    const int n_groups = R.same ? 1 : 2;
    const int64_t n1 = R.n1, n2 = R.n2;
    const double per_frame = (use_filter ? 60.0 : 44.0) * (double)(n1 + (R.same ? 0 : n2)) +
                             8.0 * cstride * n_groups;
    int G = (int)std::max(1.0, std::min(64.0, floor(R.cells_ws_mb * 1048576.0 / per_frame)));
    G = std::min(G, n_frames);
    const size_t cnt_words = (size_t)2 * G * cstride,
                 reset_words = cnt_words + (use_filter ? 2 : 1) * (size_t)G;
    if (int rc = R.cell[1].reserve(sizeof(int) * reset_words)) return rc;
    if (int rc = R.cell[2].reserve(sizeof(int) * cnt_words)) return rc;
    if (int rc = R.cell[3].reserve(sizeof(int2) * (size_t)n1 * G)) return rc;
    if (int rc = R.cell[4].reserve(sizeof(float4) * (size_t)n1 * G)) return rc;
    if (int rc = R.cell[6].reserve(sizeof(int) * (size_t)(n1 + (R.same ? 0 : n2)) * G))
        return rc;
    if (!R.same) {
        if (int rc = R.cell[7].reserve(sizeof(int2) * (size_t)n2 * G)) return rc;
        if (int rc = R.cell[8].reserve(sizeof(float4) * (size_t)n2 * G)) return rc;
    }
    if (use_filter) {
        if (int rc = R.cell[10].reserve(sizeof(float4) * (size_t)n1 * G)) return rc;
        if (!R.same)
            if (int rc = R.cell[11].reserve(sizeof(float4) * (size_t)n2 * G)) return rc;
    }
    int *d_cnt = R.cell[1].as<int>(), *d_far = d_cnt + cnt_words, *d_bad = d_far + G;
    int *d_start = R.cell[2].as<int>();
    int *d_k1 = R.cell[6].as<int>(), *d_k2 = R.same ? d_k1 : d_k1 + (size_t)n1 * G;
    const size_t scan_smem = sizeof(int) * (kScanTile + kScanTile / 32);
    MDH_CUDA(cudaFuncSetAttribute(cells_scan_kernel<TriGrid>,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)scan_smem));
    const bool excl = R.excl1 > 0, fast = R.fast_bins;
    for (int g0 = 0; g0 < n_frames; g0 += G) {
        const int ng = std::min(G, n_frames - g0);
        MDH_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(int) * reset_words, c->stream));
        const TriGrid *gg = d_grids.as<TriGrid>() + g0;
        for (int grp = 0; grp < n_groups; ++grp) {
            const float4 *pk = (grp ? R.pk2 : R.pk1).as<float4>() + (int64_t)g0 * (grp ? pad2 : pad1);
            const int n = (int)(grp ? n2 : n1);
            dim3 grid((unsigned)std::min((n + 255) / 256, 4096), ng);
            tri_bin_kernel<<<grid, 256, 0, c->stream>>>(
                pk, grp ? pad2 : pad1, n, gg, d_cnt + (size_t)grp * G * cstride, cstride,
                R.cell[grp ? 7 : 3].as<int2>(), d_far);
            MDH_CUDA(cudaGetLastError());
            c->launches++;
        }
        ScanFilter F{};
        F.out = nullptr;
        cells_scan_kernel<TriGrid><<<dim3(ng, n_groups), 1024, scan_smem, c->stream>>>(
            d_cnt, d_start, cstride, G, gg, F);
        MDH_CUDA(cudaGetLastError());
        c->launches++;
        for (int grp = 0; grp < n_groups; ++grp) {
            const float4 *pk = (grp ? R.pk2 : R.pk1).as<float4>() + (int64_t)g0 * (grp ? pad2 : pad1);
            const int n = (int)(grp ? n2 : n1);
            dim3 grid((unsigned)std::min((n + 255) / 256, 4096), ng);
            tri_scatter_kernel<<<grid, 256, 0, c->stream>>>(
                pk, grp ? pad2 : pad1, n, gg, d_start + (size_t)grp * G * cstride, cstride,
                R.cell[grp ? 7 : 3].as<int2>(), R.cell[grp ? 8 : 4].as<float4>(),
                grp ? d_k2 : d_k1);
            MDH_CUDA(cudaGetLastError());
            c->launches++;
            if (use_filter) {
                tri_cellq_kernel<<<grid, 256, 0, c->stream>>>(
                    R.cell[grp ? 8 : 4].as<float4>(), grp ? d_k2 : d_k1, n, gg,
                    R.cell[grp ? 11 : 10].as<float4>(), d_bad);
                MDH_CUDA(cudaGetLastError());
                c->launches++;
            }
        }
        TriCellParams P;
        P.s1 = R.cell[4].as<float4>();
        P.s2 = R.same ? P.s1 : R.cell[8].as<float4>();
        P.k2 = d_k2;
        P.n1 = (int)n1; P.n2 = (int)n2;
        P.start2 = R.same ? d_start : d_start + (size_t)G * cstride;
        P.cstride = cstride;
        P.grids = gg;
        P.far = d_far;
        P.thr = R.thr.as<double>();
        P.n_bins = R.n_bins;
        P.guess = rdf_bin_guess(R);
        P.counts = R.counts.as<unsigned long long>();
        P.evals = R.cell[9].as<unsigned long long>();
        P.half = R.same;
        dim3 grid((unsigned)((n1 + kThreads - 1) / kThreads), (unsigned)ng);
        int rc;
        if (use_filter) {
            TriCellFilterParams F;
            F.c = P;
            F.q1 = R.cell[10].as<float4>();
            F.q2 = R.same ? F.q1 : R.cell[11].as<float4>();
            F.bad = d_bad;
            F.filt = R.filt.as<TriCellFilter>() + g0;
            F.fc = R.fc;
            F.fast_bins = fast ? 1 : 0;
            F.fstats = R.fstats.as<unsigned long long>();
            rc = excl ? launch_tri_cells_filter_e<true>(c, F, grid, audit)
                      : launch_tri_cells_filter_e<false>(c, F, grid, audit);
        } else if (excl) {
            rc = fast ? launch_tri_cells<true, true>(c, P, grid)
                      : launch_tri_cells<true, false>(c, P, grid);
        } else {
            rc = fast ? launch_tri_cells<false, true>(c, P, grid)
                      : launch_tri_cells<false, false>(c, P, grid);
        }
        if (rc) return rc;
    }
    return MDH_OK;
}

}  // namespace

int rdf_filter_sqrt_error(mdh_ctx *c, double *err);        // rdf_filter.cu

// Device-free: the per-frame parameters of the triclinic filter (mdh_rdf_triclinic_filter_window)
int rdf_triclinic_filter_window_impl(int n_bins, double r_lo, double r_hi, double sqrt_err,
                                     int n_frames, const float *cell, const float *ext1,
                                     const float *ext2, double *frames)
{
    MDH_REQUIRE(n_bins >= 1 && n_bins <= 65536, MDH_EINVAL,
                "triclinic_filter_window: n_bins must be in [1, 65536]");
    MDH_REQUIRE(r_hi > r_lo && r_lo >= 0, MDH_EINVAL, "triclinic_filter_window: invalid range");
    MDH_REQUIRE(n_frames >= 1 && cell != nullptr && ext1 != nullptr && frames != nullptr,
                MDH_EINVAL, "triclinic_filter_window: NULL argument");
    if (ext2 == nullptr) ext2 = ext1;
    RdfState R;                    // host fields only: no device buffer is touched
    R.n_bins = n_bins;
    R.r_lo = r_lo;
    R.r_hi = r_hi;
    R.ipt = 4;
    std::vector<double> thr(n_bins + 1);
    for (int i = 0; i <= n_bins; ++i) {
        const double e = r_lo + i * ((r_hi - r_lo) / n_bins);
        thr[i] = e * e;
    }
    MDH_REQUIRE(rdf_filter_configure(R, thr.data(), sqrt_err), MDH_EINVAL,
                "triclinic_filter_window: the configuration is not eligible for the fp32 filter");
    const FilterPrep Q = rdf_filter_prep(R, sqrt_err);
    for (int f = 0; f < n_frames; ++f) {
        if (int rc = tri_check_matrix(cell + 9 * f, r_hi)) return rc;
        const float *m = cell + 9 * f;
        const TriBox h{(double)m[0], (double)m[3], (double)m[4], (double)m[6], (double)m[7],
                       (double)m[8]};
        unsigned k1[6], k2[6];
        for (int i = 0; i < 6; ++i) {
            const unsigned b1 = f32_bits(ext1[6 * f + i]), b2 = f32_bits(ext2[6 * f + i]);
            k1[i] = (b1 & 0x80000000u) ? ~b1 : (b1 | 0x80000000u);   // ext_key
            k2[i] = (b2 & 0x80000000u) ? ~b2 : (b2 | 0x80000000u);
        }
        double info[4];
        const TriFilter tf = tri_filter_prepare_frame(h, k1, k2, Q, info);
        double *o = frames + 8 * f;
        o[0] = tf.wlim != 0u ? 1.0 : 0.0;
        for (int i = 0; i < 4; ++i) o[1 + i] = info[i];
        o[5] = (double)tf.offm;
        o[6] = (double)tf.wlim;
        o[7] = (double)Q.k;
    }
    return MDH_OK;
}

// Device-free: the per-frame parameters of the cell-list filter
// (mdh_rdf_triclinic_cells_filter_window)
int rdf_triclinic_cells_filter_window_impl(int n_bins, double r_lo, double r_hi, double sqrt_err,
                                           int n_frames, const float *cell, double *frames)
{
    MDH_REQUIRE(n_bins >= 1 && n_bins <= 65536, MDH_EINVAL,
                "triclinic_cells_filter_window: n_bins must be in [1, 65536]");
    MDH_REQUIRE(r_hi > r_lo && r_lo >= 0, MDH_EINVAL,
                "triclinic_cells_filter_window: invalid range");
    MDH_REQUIRE(n_frames >= 1 && cell != nullptr && frames != nullptr, MDH_EINVAL,
                "triclinic_cells_filter_window: NULL argument");
    RdfState R;                    // host fields only: no device buffer is touched
    R.n_bins = n_bins;
    R.r_lo = r_lo;
    R.r_hi = r_hi;
    R.ipt = 4;
    std::vector<double> thr(n_bins + 1);
    for (int i = 0; i <= n_bins; ++i) {
        const double e = r_lo + i * ((r_hi - r_lo) / n_bins);
        thr[i] = e * e;
    }
    MDH_REQUIRE(rdf_filter_configure(R, thr.data(), sqrt_err), MDH_EINVAL,
                "triclinic_cells_filter_window: the configuration is not eligible for the fp32 "
                "filter");
    const FilterPrep Q = rdf_filter_prep(R, sqrt_err);
    for (int f = 0; f < n_frames; ++f) {
        if (int rc = tri_check_matrix(cell + 9 * f, r_hi)) return rc;
        double info[3];
        const TriCellFilter tf = tri_cells_filter_prepare(cell + 9 * f, Q, info);
        double *o = frames + 7 * f;
        o[0] = tf.wlim != 0u ? 1.0 : 0.0;
        for (int i = 0; i < 3; ++i) o[1 + i] = info[i];
        o[4] = (double)tf.offm;
        o[5] = (double)tf.wlim;
        o[6] = (double)Q.k;
    }
    return MDH_OK;
}

// pack kernel of rdf_device.cuh is instantiated in this translation unit as well
int rdf_accumulate_triclinic_impl(mdh_ctx *c, const float *pos1, int64_t s1, const float *pos2,
                                  int64_t s2, int location, const float *box9, int n_frames)
{
    RdfState &R = c->rdf;
    MDH_REQUIRE(R.configured, MDH_ESTATE, "rdf: accumulate before configure");
    MDH_REQUIRE(n_frames >= 1 && n_frames <= 65535, MDH_EINVAL,
                "rdf: n_frames per call must be in [1, 65535]");
    MDH_REQUIRE(box9 != nullptr, MDH_EINVAL, "rdf: box matrix is NULL");
    MDH_REQUIRE(location == MDH_HOST || location == MDH_DEVICE, MDH_EINVAL,
                "rdf: invalid location");
    MDH_REQUIRE(pos1 != nullptr && (R.same || pos2 != nullptr), MDH_EINVAL,
                "rdf: coordinate pointer is NULL");
    MDH_REQUIRE(s1 >= 3 * R.n1 && (R.same || s2 >= 3 * R.n2), MDH_EINVAL,
                "rdf: frame_stride < 3*n");
    const size_t smem = align16(sizeof(double) * (R.n_bins + 1)) + 256 * sizeof(float4) +
                        sizeof(unsigned) * kWarps * (size_t)R.n_bins;

    std::vector<TriBox> hb(n_frames);
    for (int f = 0; f < n_frames; ++f) {
        const float *m = box9 + 9 * f;
        MDH_REQUIRE(m[1] == 0.f && m[2] == 0.f && m[5] == 0.f, MDH_EINVAL,
                    "rdf: the cell matrix of frame %d is not lower triangular", f);
        MDH_REQUIRE(m[0] > 0.f && m[4] > 0.f && m[8] > 0.f && std::isfinite(m[0]) &&
                    std::isfinite(m[4]) && std::isfinite(m[8]), MDH_EINVAL,
                    "rdf: the cell matrix of frame %d is not a valid cell", f);
        hb[f] = TriBox{(double)m[0], (double)m[3], (double)m[4], (double)m[6], (double)m[7],
                       (double)m[8]};
    }

    // pair kernel: the cell list when asked for, or (auto) when every frame holds at least
    // 4 cells per axis and there are enough pairs -- the orthorhombic rule, applied to the
    // perpendicular widths
    // (with drop_axis = 2: the flat grid of tri_grid_plan_flat, 4 cells per kept width and
    // c_z >= r + M; drop_axis 0 or 1 has no cell list)
    int mode = R.mode;
    std::vector<TriGrid> grids;
    if (mode == MDH_RDF_CELLS)
        MDH_REQUIRE(R.drop_axis < 0 || R.drop_axis == 2, MDH_EINVAL,
                    "rdf: the triclinic cell list takes drop_axis 2 (z) only; use mode "
                    "\"allpairs\" or \"auto\" for drop_axis %d", R.drop_axis);
    if (mode == MDH_RDF_AUTO && R.drop_axis >= 0 && R.drop_axis != 2) mode = MDH_RDF_ALLPAIRS;
    if (mode != MDH_RDF_ALLPAIRS) {
        const double r_hi = sqrt(R.thr_hi);
        const bool flat = R.drop_axis == 2;
        bool fit4 = tri_cells_smem_bytes(R.n_bins) <= kMaxSmem && R.n1 <= (1ll << 25) &&
                    R.n2 <= (1ll << 25);
        grids.resize(n_frames);
        for (int f = 0; f < n_frames && (mode == MDH_RDF_CELLS || fit4); ++f) {
            TriPlan pl;
            if (int rc = flat ? tri_grid_plan_flat(box9 + 9 * f, r_hi, std::max(R.n1, R.n2), pl)
                              : tri_grid_plan(box9 + 9 * f, r_hi, std::max(R.n1, R.n2), pl)) {
                if (mode == MDH_RDF_CELLS) return rc;
                fit4 = false;                 // (auto) e.g. a non-finite tilt: all pairs
                break;
            }
            if (mode == MDH_RDF_CELLS) {
                MDH_REQUIRE(pl.nc[0] >= 3, MDH_EINVAL,
                            "rdf: cell-list mode needs every perpendicular width of the cell >= "
                            "3*(r_max + %g) (frame %d: %d, %d, %d cells fit)", pl.margin, f,
                            pl.fit[0], pl.fit[1], pl.fit[2]);
                MDH_REQUIRE(pl.c_ok, MDH_EINVAL,
                            "rdf: cell-list mode with drop_axis 2 needs c_z >= r_max + %g "
                            "(frame %d: c_z = %g)", pl.margin, f, (double)box9[9 * f + 8]);
            }
            fit4 = fit4 && pl.nc[0] >= 3 && pl.c_ok &&
                   std::min({pl.fit[0], pl.fit[1], flat ? 4 : pl.fit[2]}) >= 4;
            grids[f].h = hb[f];
            for (int k = 0; k < 3; ++k) grids[f].nc[k] = pl.nc[k];
            grids[f].ncell = pl.nc[0] * pl.nc[1] * pl.nc[2];
        }
        if (mode == MDH_RDF_AUTO)
            mode = fit4 && (double)R.n1 * (double)R.n2 >= 4e6 ? MDH_RDF_CELLS : MDH_RDF_ALLPAIRS;
    }
    if (mode == MDH_RDF_CELLS) {
        MDH_REQUIRE(tri_cells_smem_bytes(R.n_bins) <= kMaxSmem, MDH_EINVAL,
                    "rdf: too many bins for the triclinic cell-list kernel");
        MDH_REQUIRE(R.n1 <= (1ll << 25) && R.n2 <= (1ll << 25), MDH_EINVAL,
                    "rdf: cell-list mode takes at most 2^25 particles per group");
    } else {
        MDH_REQUIRE(smem <= kMaxSmem, MDH_EINVAL, "rdf: too many bins for the triclinic kernel");
    }

    DevBuf &d_box = R.cell[0];
    if (int rc = d_box.reserve(sizeof(TriBox) * n_frames)) return rc;
    MDH_CUDA(cudaMemcpyAsync(d_box.p, hb.data(), sizeof(TriBox) * n_frames,
                             cudaMemcpyHostToDevice, c->stream));
    MDH_CUDA(cudaStreamSynchronize(c->stream));        // hb is a local

    // fp32 filter (arith auto / on / audit) of the all-pairs path and of the cell list
    const bool use_filter = mode == MDH_RDF_ALLPAIRS && R.filter_ok &&
                            R.filter_mode != MDH_FILTER_OFF &&
                            tri_filter_smem_bytes(R.n_bins, R.fc.hslots, R.fc.cb) <= kMaxSmem;
    const bool cells_filter = mode == MDH_RDF_CELLS && R.filter_ok &&
                              R.filter_mode != MDH_FILTER_OFF;
    double sqrt_err = 0.0;         // measured once per process (rdf_filter.cu)
    if (use_filter || cells_filter)
        if (int rc = rdf_filter_sqrt_error(c, &sqrt_err)) return rc;
    // the cell list's per-frame window depends on the cell matrix only
    std::vector<TriCellFilter> cfilt;
    if (cells_filter) {
        const FilterPrep fq = rdf_filter_prep(R, sqrt_err);
        cfilt.resize(n_frames);
        for (int f = 0; f < n_frames; ++f) cfilt[f] = tri_cells_filter_prepare(box9 + 9 * f, fq);
    }
    const int64_t pq = use_filter ? kTriTile : 256;
    const int64_t pad1 = (R.n1 + pq - 1) / pq * pq, pad2 = (R.n2 + pq - 1) / pq * pq;
    const int n_groups = R.same ? 1 : 2;
    // the cell-list path times its whole pipeline (pack and wrap included)
    if (mode == MDH_RDF_CELLS)
        if (int rc = c->t_rdf.begin(c->stream)) return rc;
    for (int g = 0; g < n_groups; ++g) {
        const float *pos = g ? pos2 : pos1;
        const int64_t stride = g ? s2 : s1, n = g ? R.n2 : R.n1, npad = g ? pad2 : pad1;
        DevBuf &raw = g ? R.raw2[0] : R.raw1[0];
        DevBuf &pk = g ? R.pk2 : R.pk1;
        const float *dsrc = pos;
        int64_t dstride = stride;
        if (location == MDH_HOST) {
            if (int rc = raw.reserve(sizeof(float) * 3 * n * n_frames)) return rc;
            MDH_CUDA(mdh_copy_frames(raw.p, sizeof(float) * 3 * n, pos, sizeof(float) * stride,
                                       sizeof(float) * 3 * n, n_frames, cudaMemcpyHostToDevice,
                                       c->stream));
            dsrc = raw.as<float>();
            dstride = 3 * n;
        }
        if (int rc = pk.reserve(sizeof(float4) * npad * n_frames)) return rc;
        dim3 grid((unsigned)std::min<int64_t>((npad + 255) / 256, 2048), n_frames);
        // a dropped coordinate is zeroed here; the wrap below may move it again (drop_axis 0
        // or 1 on a tilted cell), as the reference's wrap does
        rdf_pack_kernel<<<grid, 256, 0, c->stream>>>(dsrc, dstride, pk.as<float4>(), n, npad,
                                                     g ? R.excl2 : R.excl1, R.drop_axis, nullptr,
                                                     nullptr);
        MDH_CUDA(cudaGetLastError());
        tri_wrap_kernel<<<grid, 256, 0, c->stream>>>(pk.as<float4>(), npad, (int)n,
                                                     d_box.as<TriBox>());
        MDH_CUDA(cudaGetLastError());
        c->launches += 2;
        if (use_filter) {
            // the filter's bound takes the extents of the wrapped coordinates
            DevBuf &ext = g ? R.ext2 : R.ext1;
            if (int rc = ext.reserve(sizeof(unsigned) * 6 * n_frames)) return rc;
            rdf_ext_init_kernel<<<(6 * n_frames + 255) / 256, 256, 0, c->stream>>>(
                ext.as<unsigned>(), 6 * n_frames);
            tri_extent_kernel<<<grid, 256, 0, c->stream>>>(pk.as<float4>(), npad, (int)n,
                                                           ext.as<unsigned>());
            MDH_CUDA(cudaGetLastError());
            c->launches += 2;
        }
    }
    if (mode == MDH_RDF_CELLS) {
        if (int rc = tri_cells_accumulate(c, grids, pad1, pad2, cfilt,
                                          R.filter_mode == MDH_FILTER_AUDIT))
            return rc;
        return c->t_rdf.end(c->stream);
    }

    TriParams P;
    P.p1 = R.pk1.as<float4>();
    P.p2 = R.same ? P.p1 : R.pk2.as<float4>();
    P.pad1 = pad1; P.pad2 = R.same ? pad1 : pad2;
    P.n1 = (int)R.n1; P.n2 = (int)R.n2;
    P.boxes = d_box.as<TriBox>();
    P.thr = R.thr.as<double>();
    P.n_bins = R.n_bins;
    P.counts = R.counts.as<unsigned long long>();
    // enough blocks to fill the device; a block's u32 words cannot overflow (256 x jchunk)
    const int64_t iblocks = (R.n1 + 255) / 256;
    int64_t jsplit = std::max<int64_t>(1, (4 * c->sm_count + iblocks * n_frames - 1) /
                                              (iblocks * n_frames));
    int64_t jchunk = ((R.n2 + jsplit - 1) / jsplit + 255) / 256 * 256;
    jchunk = std::min<int64_t>(jchunk, 1 << 22);
    P.jchunk = (int)jchunk;
    dim3 grid((unsigned)iblocks, (unsigned)((R.n2 + jchunk - 1) / jchunk), (unsigned)n_frames);
    MDH_REQUIRE(grid.y <= 65535, MDH_EINVAL, "rdf: group 2 is too large for the triclinic kernel");
    if (int rc = c->t_rdf.begin(c->stream)) return rc;
    if (use_filter) {
        // per-frame parameters on the host from the extents of the wrapped coordinates;
        // the declined frames then go to rdf_triclinic_kernel, run by run
        std::vector<unsigned> he(6 * (size_t)n_frames * n_groups);
        for (int g = 0; g < n_groups; ++g)
            MDH_CUDA(cudaMemcpyAsync(he.data() + 6 * (size_t)n_frames * g,
                                     (g ? R.ext2 : R.ext1).p, sizeof(unsigned) * 6 * n_frames,
                                     cudaMemcpyDeviceToHost, c->stream));
        MDH_CUDA(cudaStreamSynchronize(c->stream));
        const unsigned *he2 = he.data() + (R.same ? 0 : 6 * (size_t)n_frames);
        const FilterPrep fq = rdf_filter_prep(R, sqrt_err);
        std::vector<TriFilter> hf(n_frames);
        for (int f = 0; f < n_frames; ++f)
            hf[f] = tri_filter_prepare_frame(hb[f], he.data() + 6 * f, he2 + 6 * f, fq);
        if (int rc = R.filt.reserve(sizeof(TriFilter) * n_frames)) return rc;
        // pageable source: the runtime stages it before returning
        MDH_CUDA(cudaMemcpyAsync(R.filt.p, hf.data(), sizeof(TriFilter) * n_frames,
                                 cudaMemcpyHostToDevice, c->stream));
        TriFilterParams Q;
        Q.p1 = P.p1; Q.p2 = P.p2;
        Q.pad1 = P.pad1; Q.pad2 = P.pad2;
        Q.n1 = P.n1; Q.n2 = P.n2;
        Q.boxes = P.boxes;
        Q.filt = R.filt.as<TriFilter>();
        Q.thr = P.thr;
        Q.n_bins = P.n_bins;
        Q.guess = rdf_bin_guess(R);
        Q.fast_bins = R.fast_bins ? 1 : 0;
        Q.same = R.same;
        Q.fc = R.fc;
        Q.counts = P.counts;
        Q.fstats = R.fstats.as<unsigned long long>();
        Q.evals = R.cell[9].as<unsigned long long>();
        // tile pairs as the orthorhombic all-pairs launch (rdf.cu): about 12 blocks per SM,
        // and a block's u32 histogram below 2^31 weighted pairs
        const int n_itiles = (int)(pad1 / kTriTile);
        Q.n_jtiles = (int)(Q.pad2 / kTriTile);
        const int64_t target = (int64_t)c->sm_count * 2 * 6;
        int64_t n_jchunks = (target + (int64_t)n_itiles * n_frames - 1) /
                            ((int64_t)n_itiles * n_frames);
        n_jchunks = std::max<int64_t>(1, std::min<int64_t>(n_jchunks, Q.n_jtiles));
        n_jchunks = std::max<int64_t>(n_jchunks, (Q.n_jtiles + 1023) / 1024);
        Q.jtiles_per_chunk = (int)((Q.n_jtiles + n_jchunks - 1) / n_jchunks);
        Q.n_jchunks = (int)((Q.n_jtiles + Q.jtiles_per_chunk - 1) / Q.jtiles_per_chunk);
        const dim3 fgrid((unsigned)(n_itiles * Q.n_jchunks), (unsigned)n_frames);
        const bool audit = R.filter_mode == MDH_FILTER_AUDIT;
        if (int rc = R.excl1 > 0 ? launch_tri_filter_e<true>(c, Q, fgrid, audit)
                                 : launch_tri_filter_e<false>(c, Q, fgrid, audit))
            return rc;
        if (R.excl1 > 0)
            MDH_CUDA(cudaFuncSetAttribute(rdf_triclinic_kernel<true>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        else
            MDH_CUDA(cudaFuncSetAttribute(rdf_triclinic_kernel<false>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        for (int f0 = 0; f0 < n_frames;) {
            if (hf[f0].wlim != 0u) { ++f0; continue; }
            int f1 = f0 + 1;
            while (f1 < n_frames && hf[f1].wlim == 0u) ++f1;
            TriParams Pd = P;
            Pd.p1 = P.p1 + f0 * P.pad1;
            Pd.p2 = P.p2 + f0 * P.pad2;
            Pd.boxes = P.boxes + f0;
            const dim3 dgrid(grid.x, grid.y, (unsigned)(f1 - f0));
            if (R.excl1 > 0) rdf_triclinic_kernel<true><<<dgrid, 256, smem, c->stream>>>(Pd);
            else rdf_triclinic_kernel<false><<<dgrid, 256, smem, c->stream>>>(Pd);
            MDH_CUDA(cudaGetLastError());
            c->launches++;
            R.evals += R.n1 * R.n2 * (int64_t)(f1 - f0);
            f0 = f1;
        }
        return c->t_rdf.end(c->stream);
    }
    if (R.excl1 > 0) {
        MDH_CUDA(cudaFuncSetAttribute(rdf_triclinic_kernel<true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        rdf_triclinic_kernel<true><<<grid, 256, smem, c->stream>>>(P);
    } else {
        MDH_CUDA(cudaFuncSetAttribute(rdf_triclinic_kernel<false>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        rdf_triclinic_kernel<false><<<grid, 256, smem, c->stream>>>(P);
    }
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    R.evals += R.n1 * R.n2 * (int64_t)n_frames;
    return c->t_rdf.end(c->stream);
}
