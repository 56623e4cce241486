// rdf.cu -- minimum-image pair-distance histogram kernels (seam #1).
//
// Replaces, per frame, the reference's radial_histogram
// (/root/reference/src/mdhelper/analysis/structure.py:32-104), i.e. the
// third-party MDAnalysis capped_distance (arithmetic: SURVEY.md Appendix A)
// followed by the exclusion mask and numpy.histogram, without ever
// materialising the pair list.
//
// Per pair (i in group 1, j in group 2), bit for bit what the reference does:
//     dx_k = (double)(float)(pos2[j][k] - pos1[i][k])          fp32 subtract
//     s    = (double)inv_k * dx_k            inv_k = (float)(1.0 / box_k)
//     dx_k = (double)box_k * (s - round(s))
//     d2   = (dx0*dx0 + dx1*dx1) + dx2*dx2   every product rounded (no FMA)
// round() is evaluated with the 1.5*2^52 magic-number add (round-half-even);
// it differs from C round() only when s is exactly k+1/2, where s - round(s)
// is +-1/2 either way and the squared term is identical.  sqrt is never
// taken: IEEE sqrt is monotone, so numpy.histogram's "edges[k] <= d < edges[k+1]"
// is evaluated on d2 against thresholds T[k] = min{x : sqrt(x) >= edges[k]}
// prepared on the host (mdhelper_b200/analysis/_binning.py).
//
// All FP64 arithmetic on the path uses __dmul_rn/__dadd_rn/__dsub_rn so nvcc
// can never contract it; the file is additionally built with -fmad=false.
//
// Kernel shape (rdf_allpairs_kernel): 256 threads; every thread keeps IPT
// i-particles in registers; j-tiles of 256*IPT particles are staged in shared
// memory with cp.async (double buffered) and read as broadcast LDS.128; the
// inner loop is branch-free (certified bin guess + one fp64 compare) so that
// several pairs are in flight per thread; histograms are privatised per lane
// (packed 8-bit counters, no atomics) or per warp (u32 shared atomics) and
// merged into the global int64 histogram once per block.

#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "rdf_device.cuh"

using namespace rdfdev;

namespace {

template <int HIST, int IPT>
__host__ __device__ inline size_t pair_smem_bytes(int n_bins)
{
    return align16(sizeof(double) * (n_bins + 1)) + 2 * kThreads * IPT * sizeof(float4) +
           hist_smem_bytes<HIST>(n_bins);
}

// ---- x-sorted groups for the all-pairs filter kernel -------------------------------
// One block per frame: a counting sort of the frame's packed rows by an x-slab key
// (kXSlabs slabs over the frame's x extent), then the x extent of every tile of `tile`
// rows.  Rows keep their tags (.w), so exclusions and same-group runs see the same pairs;
// the order within a slab is whatever the shared-memory atomics give (the counts do not
// depend on the order of the rows).  Padding rows are copied as they are.
constexpr int kXSlabs = 1024;

__global__ void __launch_bounds__(1024)
    rdf_xsort_kernel(const float4 *__restrict__ in, float4 *__restrict__ out, int64_t n,
                     int64_t npad, const unsigned *__restrict__ ext, int tile,
                     float2 *__restrict__ tx)
{
    __shared__ unsigned cnt[kXSlabs];
    __shared__ unsigned wsum[32];
    const int frame = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float4 *src = in + (int64_t)frame * npad;
    float4 *dst = out + (int64_t)frame * npad;
    const float x0 = ext_unkey(ext[frame * 6]), x1 = ext_unkey(ext[frame * 6 + 3]);
    // slab of x: NaN and a frame of width 0 (or inf) fall into slab 0 or the last one
    const float inv = (float)kXSlabs / (x1 - x0);
    auto slab = [&](float x) {
        const float s = fminf(fmaxf((x - x0) * inv, 0.f), (float)(kXSlabs - 1));
        return (int)s;
    };
    static_assert(kXSlabs == 1024, "one slab per thread in the scan");
    cnt[tid] = 0;
    __syncthreads();
    for (int64_t i = tid; i < n; i += 1024) atomicAdd(&cnt[slab(src[i].x)], 1u);
    __syncthreads();
    // exclusive scan of the 1024 counts
    const unsigned c = cnt[tid];
    unsigned v = c;
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    if (lane == 31) wsum[warp] = v;
    __syncthreads();
    if (warp == 0) {
        unsigned w = wsum[lane];
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += t;
        }
        wsum[lane] = w;
    }
    __syncthreads();
    cnt[tid] = v - c + (warp ? wsum[warp - 1] : 0u);
    __syncthreads();
    for (int64_t i = tid; i < n; i += 1024) {
        const float4 p = src[i];
        dst[atomicAdd(&cnt[slab(p.x)], 1u)] = p;
    }
    for (int64_t i = n + tid; i < npad; i += 1024) dst[i] = src[i];
    __syncthreads();          // the block's global writes are visible to the block
    // x extent of every tile (rows below n), one warp per tile
    const int n_tiles = (int)(npad / tile);
    for (int t = warp; t < n_tiles; t += 32) {
        unsigned lo = 0xffffffffu, hi = 0u;
        const int64_t r1 = min((int64_t)(t + 1) * tile, n);
        for (int64_t r = (int64_t)t * tile + lane; r < r1; r += 32) {
            const unsigned k = ext_key(dst[r].x);
            lo = min(lo, k);
            hi = max(hi, k);
        }
        lo = __reduce_min_sync(0xffffffffu, lo);
        hi = __reduce_max_sync(0xffffffffu, hi);
        if (lane == 0) tx[(int64_t)frame * n_tiles + t] = make_float2(ext_unkey(lo), ext_unkey(hi));
    }
}

// filter_cleanx_form of every tile pair (i-tile, j-tile) of every frame from the tile
// extents tx1 [F][ni], tx2 [F][nj] of the sorted groups: out [F][ni][nj]
__global__ void rdf_cleanx_forms_kernel(const float2 *__restrict__ tx1,
                                               const float2 *__restrict__ tx2, int ni, int nj,
                                               const FrameBox *__restrict__ boxes,
                                               unsigned char *__restrict__ out)
{
    const int frame = blockIdx.y;
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= ni * nj) return;
    const int a = q / nj, b = q - a * nj;
    const float2 ti = tx1[(int64_t)frame * ni + a], tj = tx2[(int64_t)frame * nj + b];
    out[(int64_t)frame * ni * nj + q] =
        (unsigned char)filter_cleanx_form(ti.x, ti.y, tj.x, tj.y, (float)boxes[frame].box[0]);
}

template <int HIST, bool EXCL, bool FAST, int IPT>
__global__ void __launch_bounds__(kThreads, 2) rdf_allpairs_kernel(const PairParams P)
{
    constexpr int TILE = kThreads * IPT;
    extern __shared__ __align__(16) unsigned char smem[];
    double *sT = reinterpret_cast<double *>(smem);
    float4 *sJ = reinterpret_cast<float4 *>(smem + align16(sizeof(double) * (P.n_bins + 1)));
    unsigned *sH = reinterpret_cast<unsigned *>(sJ + 2 * TILE);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int frame = blockIdx.y;
    const int it = blockIdx.x / P.n_jchunks;
    const int jc = blockIdx.x - it * P.n_jchunks;
    int jt0 = jc * P.jtiles_per_chunk;
    const int jt1 = min(P.n_jtiles, jt0 + P.jtiles_per_chunk);
    if (P.same) jt0 = max(jt0, it);       // upper triangle of tile pairs
    if (jt0 >= jt1) return;
    // frames the fp32-filter kernel (rdf_filter.cu) has taken are not done again
    if (P.filt != nullptr && P.filt[frame].wlim != 0u) return;

    const int n_bins = P.n_bins;
    const int n_words = priv_words(n_bins);
    for (int k = tid; k <= n_bins; k += kThreads) sT[k] = P.thr[k];
    const int n_hist_words = (int)(hist_smem_bytes<HIST>(n_bins) / sizeof(unsigned));
    for (int k = tid; k < n_hist_words; k += kThreads) sH[k] = 0;

    const float4 *f1 = P.p1 + (int64_t)frame * P.pad1;
    const float4 *f2 = P.same ? f1 : P.p2 + (int64_t)frame * P.pad2;
    const FrameBox fb = P.boxes[frame];
    const BinGuess guess = P.guess;

    float xi[IPT], yi[IPT], zi[IPT];
    int gi[IPT];
    unsigned wv[IPT];
#pragma unroll
    for (int ii = 0; ii < IPT; ++ii) {
        const int i = it * TILE + ii * kThreads + tid;
        wv[ii] = i < P.n1 ? 1u : 0u;
        const float4 a = f1[min(i, P.n1 - 1)];
        // rows past the end of the group become NaN: every pair they form lands in
        // the "not counted" slot, so the inner loop needs no validity test
        xi[ii] = wv[ii] ? a.x : __int_as_float(0x7fc00000);
        yi[ii] = a.y; zi[ii] = a.z; gi[ii] = __float_as_int(a.w);
    }

    // warp-atomic layout per warp: [pad][n_bins bins][32 trash words]
    unsigned *myhist = (HIST == MDH_HIST_WARP_ATOMIC)
                           ? sH + warp * warp_hist_words(n_bins) + 1
                           : sH + (size_t)warp * n_words * 32;
    unsigned *bhist = sH + (size_t)kWarps * n_words * 32;         // LANE_PRIVATE only
    unsigned char *lane_base = reinterpret_cast<unsigned char *>(myhist) + 4 * lane;
    const unsigned hist32 = (unsigned)__cvta_generic_to_shared(myhist);
    const unsigned trash32 = hist32 + 4u * (unsigned)(n_bins + lane);

    // packed buffers are padded to whole tiles, so staging never reads out of bounds
    auto stage_tile = [&](int jt, int buf) {
        const float4 *src = f2 + (int64_t)jt * TILE;
        float4 *dst = sJ + buf * TILE;
#pragma unroll
        for (int q = 0; q < IPT; ++q)
            __pipeline_memcpy_async(dst + q * kThreads + tid, src + q * kThreads + tid,
                                    sizeof(float4));
        __pipeline_commit();
    };
    stage_tile(jt0, 0);

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
        const int jn = min(TILE, P.n2 - jt * TILE);
        const float4 *tile = sJ + buf * TILE;

        if (HIST == MDH_HIST_WARP_ATOMIC) {
#pragma unroll 2
            for (int jj = 0; jj < jn; ++jj) {
                const float4 pj = tile[jj];
#pragma unroll
                for (int ii = 0; ii < IPT; ++ii) {
                    const double d2 = pair_d2(xi[ii], yi[ii], zi[ii], pj, fb);
                    const bool keep = !(EXCL && gi[ii] == __float_as_int(pj.w));
                    if (FAST) {
                        bool below;
                        const int j = slot_fast_parts(d2, sT, n_bins, guess, below);
                        // bin j - 1 if below else bin j; j == n_bins && !below (above
                        // range, NaN rows, exclusions) goes to this lane's trash word
                        unsigned a = (below ? hist32 - 4u : hist32) + 4u * (unsigned)j;
                        if ((!below && j == n_bins) || !keep) a = trash32;
                        red_shared(a, weight);
                    } else {
                        const int slot = slot_search(d2, sT, n_bins);
                        if (keep && (unsigned)(slot - 1) < (unsigned)n_bins)
                            atomicAdd(&myhist[slot - 1], weight);
                    }
                }
            }
        } else {
            constexpr int kSeg = 254 / IPT;       // increments per lane per flush <= 254
            for (int j0 = 0; j0 < jn; j0 += kSeg) {
                const int j1 = min(jn, j0 + kSeg);
#pragma unroll 2
                for (int jj = j0; jj < j1; ++jj) {
                    const float4 pj = tile[jj];
                    int slot[IPT];
#pragma unroll
                    for (int ii = 0; ii < IPT; ++ii) {
                        const double d2 = pair_d2(xi[ii], yi[ii], zi[ii], pj, fb);
                        slot[ii] = slot_of<FAST>(d2, sT, n_bins, guess);
                        if (EXCL && gi[ii] == __float_as_int(pj.w)) slot[ii] = 0;
                    }
#pragma unroll
                    for (int ii = 0; ii < IPT; ++ii) priv_add(lane_base, slot[ii], wv[ii]);
                }
                priv_flush(myhist, bhist, n_words, n_bins, lane, weight);
            }
        }
        __syncthreads();
        buf ^= 1;
    }

    // merge into the global int64 histogram
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
}

template <int HIST, bool EXCL, bool FAST, int IPT>
int launch_allpairs(mdh_ctx *c, const PairParams &P, dim3 grid)
{
    const size_t smem = pair_smem_bytes<HIST, IPT>(P.n_bins);
    auto kern = rdf_allpairs_kernel<HIST, EXCL, FAST, IPT>;
    MDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)smem));
    kern<<<grid, kThreads, smem, c->stream>>>(P);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    return MDH_OK;
}

template <int HIST, bool EXCL, bool FAST>
int launch_allpairs_ipt(mdh_ctx *c, const PairParams &P, dim3 grid, int ipt)
{
    return ipt == 4 ? launch_allpairs<HIST, EXCL, FAST, 4>(c, P, grid)
                    : launch_allpairs<HIST, EXCL, FAST, 2>(c, P, grid);
}

template <int HIST>
int launch_allpairs_dyn(mdh_ctx *c, const PairParams &P, dim3 grid, bool excl, bool fast,
                        int ipt)
{
    if (excl)
        return fast ? launch_allpairs_ipt<HIST, true, true>(c, P, grid, ipt)
                    : launch_allpairs_ipt<HIST, true, false>(c, P, grid, ipt);
    return fast ? launch_allpairs_ipt<HIST, false, true>(c, P, grid, ipt)
                : launch_allpairs_ipt<HIST, false, false>(c, P, grid, ipt);
}

}  // namespace

// ---- host side ------------------------------------------------------------------

int rdf_cells_accumulate(mdh_ctx *c, const float *raw1, int64_t stride1, const float *raw2,
                         int64_t stride2, int f0, int n_frames, bool use_filter,
                         double sqrt_err);                        // rdf_cells.cu
static int rdf_accumulate_piece(mdh_ctx *c, const float *pos1, int64_t s1, const float *pos2,
                                int64_t s2, int location, int f0, int n_frames, int mode);
int rdf_filter_launch(mdh_ctx *c, const PairParams &P, dim3 grid, bool excl,
                      bool audit);                     // rdf_filter.cu

static double g_sqrt_err_cached = -1.0;

BinGuess rdf_bin_guess(const RdfState &R)
{
    BinGuess g;
    const double scale = R.n_bins / (R.r_hi - R.r_lo);
    const double margin = 1.0 / 64 + R.n_bins * (1.0 / 524288);
    g.scale = (float)scale;
    g.offset = (float)(-R.r_lo * scale + 0.5 - margin);
    return g;
}

int rdf_configure_impl(mdh_ctx *c, int64_t n1, int64_t n2, int same, int n_bins,
                       const double *thr, double r_lo, double r_hi, int64_t e1, int64_t e2,
                       int drop_axis, int mode, int hist)
{
    RdfState &R = c->rdf;
    MDH_REQUIRE(n1 > 0 && n2 > 0, MDH_EINVAL, "rdf: both groups must be non-empty");
    MDH_REQUIRE(n1 < (1ll << 30) && n2 < (1ll << 30), MDH_EINVAL,
                "rdf: at most 2^30 particles per group");
    MDH_REQUIRE(!same || n1 == n2, MDH_EINVAL, "rdf: same_group requires n1 == n2");
    MDH_REQUIRE(n_bins >= 1 && n_bins <= 65536, MDH_EINVAL,
                "rdf: n_bins must be in [1, 65536]");
    MDH_REQUIRE(thr != nullptr, MDH_EINVAL, "rdf: thresholds_sq is NULL");
    for (int k = 0; k < n_bins; ++k)
        MDH_REQUIRE(thr[k] < thr[k + 1], MDH_EINVAL,
                    "rdf: thresholds_sq must be strictly increasing (k=%d)", k);
    MDH_REQUIRE(thr[0] >= 0.0, MDH_EINVAL, "rdf: thresholds_sq[0] must be >= 0");
    MDH_REQUIRE((e1 > 0) == (e2 > 0) && e1 >= 0, MDH_EINVAL,
                "rdf: exclusion sizes must both be positive or both zero");
    MDH_REQUIRE(!same || e1 == e2, MDH_EINVAL,
                "rdf: same_group needs equal exclusion block sizes (i/excl1 == j/excl2 is not "
                "symmetric otherwise); pass the group twice with same_group = 0");
    MDH_REQUIRE(drop_axis >= -1 && drop_axis <= 2, MDH_EINVAL, "rdf: invalid drop_axis");
    MDH_REQUIRE(mode >= MDH_RDF_AUTO && mode <= MDH_RDF_CELLS, MDH_EINVAL,
                "rdf: invalid mode");
    MDH_REQUIRE(hist >= MDH_HIST_AUTO && hist <= MDH_HIST_LANE_PRIVATE, MDH_EINVAL,
                "rdf: invalid hist");
    MDH_REQUIRE(r_hi > r_lo && r_lo >= 0, MDH_EINVAL, "rdf: invalid range");

    // tuning knobs for experiments: MDH_TUNE="ipt=4,fast=0"
    int ipt = 4, allow_fast = 1, allow_filter = 1;
    if (const char *t = getenv("MDH_TUNE")) {
        if (const char *p = strstr(t, "ipt=")) ipt = atoi(p + 4) == 4 ? 4 : 2;
        if (const char *p = strstr(t, "fast=")) allow_fast = atoi(p + 5) != 0;
        if (const char *p = strstr(t, "filter=")) allow_filter = atoi(p + 7) != 0;
        if (const char *p = strstr(t, "occ=")) R.filter_occ = std::min(4, std::max(2, atoi(p + 4)));
        if (const char *p = strstr(t, "cws=")) R.cells_ws_mb = std::max(1.0, atof(p + 4));
        if (const char *p = strstr(t, "cchunk=")) R.cells_chunk = std::max(1, atoi(p + 7));
        if (const char *p = strstr(t, "cipt=")) R.cells_ipt = atoi(p + 5) == 2 ? 2 : 4;
        if (const char *p = strstr(t, "cdbg=")) R.cells_debug = atoi(p + 5) != 0;
    }
    // measured on B200 (profiles/): per-warp shared-memory atomics beat the
    // lane-private byte counters at every bin count tried, and need less memory
    if (hist == MDH_HIST_AUTO) hist = MDH_HIST_WARP_ATOMIC;
    const size_t need = hist == MDH_HIST_LANE_PRIVATE
                            ? pair_smem_bytes<MDH_HIST_LANE_PRIVATE, 4>(n_bins)
                            : pair_smem_bytes<MDH_HIST_WARP_ATOMIC, 4>(n_bins);
    MDH_REQUIRE(need <= kMaxSmem, MDH_EINVAL,
                "rdf: n_bins=%d needs %zu bytes of shared memory (> %zu)", n_bins, need,
                kMaxSmem);

    R.configured = false;
    R.n1 = n1; R.n2 = n2; R.same = same ? 1 : 0; R.n_bins = n_bins;
    R.excl1 = e1; R.excl2 = e2; R.drop_axis = drop_axis; R.mode = mode; R.hist = hist;
    R.r_lo = r_lo; R.r_hi = r_hi; R.thr_hi = thr[n_bins];
    R.evals = 0;
    R.ipt = ipt;

    if (int rc = R.thr.reserve(sizeof(double) * (n_bins + 2))) return rc;
    if (int rc = R.counts.reserve(sizeof(unsigned long long) * n_bins)) return rc;
    if (int rc = R.cell[9].reserve(sizeof(unsigned long long) + sizeof(int))) return rc;
    if (int rc = R.fstats.reserve(sizeof(unsigned long long) * 11)) return rc;
    MDH_CUDA(cudaMemsetAsync(R.fstats.p, 0, sizeof(unsigned long long) * 11, c->stream));
    std::vector<double> t(thr, thr + n_bins + 1);
    t.push_back(INFINITY);
    MDH_CUDA(cudaMemcpyAsync(R.thr.p, t.data(), sizeof(double) * t.size(),
                             cudaMemcpyHostToDevice, c->stream));
    MDH_CUDA(cudaMemsetAsync(R.counts.p, 0, sizeof(unsigned long long) * n_bins, c->stream));
    MDH_CUDA(cudaMemsetAsync(R.cell[9].p, 0, sizeof(unsigned long long) + sizeof(int),
                             c->stream));
    R.evals_dev_init = true;

    // certify the branch-free bin guess for this configuration (else: binary search)
    int *d_bad = reinterpret_cast<int *>(R.cell[9].as<unsigned long long>() + 1);
    int h_bad = 0;
    rdf_selfcheck_kernel<<<(n_bins + 1 + 127) / 128, 128, 0, c->stream>>>(
        R.thr.as<double>(), n_bins, rdf_bin_guess(R), d_bad);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    MDH_CUDA(cudaMemcpyAsync(&h_bad, d_bad, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
    MDH_CUDA(cudaStreamSynchronize(c->stream));   // also: t is a local
    R.selfcheck_bad = h_bad;
    R.fast_bins = allow_fast && h_bad == 0;

    // fp32 filter: needs the 4-particle tile, the shared-atomic histogram layout and
    // uniform edges; the approximation error of MUFU.SQRT is measured, not assumed
    R.filter_ok = false;
    if (allow_filter && hist == MDH_HIST_WARP_ATOMIC) {
        if (int rc = rdf_filter_sqrt_error(c, &g_sqrt_err_cached)) return rc;
        rdf_filter_configure(R, thr, g_sqrt_err_cached);
    }
    R.configured = true;
    return MDH_OK;
}

// Exhaustive check of the configured thresholds and bin guess (rdf_guess_audit_kernel):
// out = {classes checked, disagreements, bits of the smallest bad d2 (-1: none), its fast
// slot minus its exact slot}.
int rdf_bin_guess_audit_impl(mdh_ctx *c, int64_t *out)
{
    RdfState &R = c->rdf;
    MDH_REQUIRE(R.configured, MDH_ESTATE, "rdf: bin guess audit before configure");
    DevBuf buf;
    if (int rc = buf.reserve(2 * sizeof(unsigned long long) + sizeof(int))) return rc;
    unsigned long long *d_out = buf.as<unsigned long long>();
    const unsigned long long init[2] = {0ull, ~0ull};
    MDH_CUDA(cudaMemcpyAsync(d_out, init, sizeof(init), cudaMemcpyHostToDevice, c->stream));
    const BinGuess g = rdf_bin_guess(R);
    const size_t smem = sizeof(double) * (R.n_bins + 1);
    MDH_CUDA(cudaFuncSetAttribute(rdf_guess_audit_kernel,
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    rdf_guess_audit_kernel<<<c->sm_count * 8, 256, smem, c->stream>>>(R.thr.as<double>(),
                                                                       R.n_bins, g, d_out);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    unsigned long long h[2];
    MDH_CUDA(cudaMemcpyAsync(h, d_out, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    MDH_CUDA(cudaStreamSynchronize(c->stream));
    int diff = 0;
    if (h[0]) {
        int *d_diff = reinterpret_cast<int *>(d_out + 2);
        double d2;
        memcpy(&d2, &h[1], sizeof(d2));
        rdf_guess_probe_kernel<<<1, 1, 0, c->stream>>>(R.thr.as<double>(), R.n_bins, g, d2,
                                                       d_diff);
        MDH_CUDA(cudaGetLastError());
        c->launches++;
        MDH_CUDA(cudaMemcpyAsync(&diff, d_diff, sizeof(int), cudaMemcpyDeviceToHost,
                                 c->stream));
        MDH_CUDA(cudaStreamSynchronize(c->stream));
    }
    out[0] = kGuessClasses;
    out[1] = (int64_t)h[0];
    out[2] = h[0] ? (int64_t)h[1] : -1;
    out[3] = diff;
    return MDH_OK;
}

// host input: the copy into `raw` is queued on the stager's copy stream (the caller
// brackets the group copies of a piece with stager.acquire / publish).  tx (with ext): the
// packed rows are sorted by x and tx receives the x extents of their tiles of `tile` rows
// (rdf_xsort_kernel), for the x-clean tile pairs of the all-pairs filter kernel.
static int rdf_upload_group(mdh_ctx *c, const float *pos, int64_t stride, int location,
                            int64_t n, int64_t npad, int64_t excl, int n_frames,
                            DevBuf &raw, DevBuf &pk, DevBuf *ext, bool copy_only, int f0,
                            DevBuf *tx = nullptr, int tile = 0)
{
    RdfState &R = c->rdf;
    MDH_REQUIRE(pos != nullptr, MDH_EINVAL, "rdf: coordinate pointer is NULL");
    MDH_REQUIRE(stride >= 3 * n, MDH_EINVAL, "rdf: frame_stride (%lld) < 3*n (%lld)",
                (long long)stride, (long long)(3 * n));
    const float *dsrc = pos;
    int64_t dstride = stride;
    if (location == MDH_HOST) {
        if (copy_only) {
            if (int rc = raw.reserve(sizeof(float) * 3 * n * n_frames)) return rc;
            MDH_CUDA(mdh_copy_frames(raw.p, sizeof(float) * 3 * n, pos,
                                       sizeof(float) * stride, sizeof(float) * 3 * n, n_frames,
                                       cudaMemcpyHostToDevice, c->stager.copy));
            return MDH_OK;
        }
        dsrc = raw.as<float>();
        dstride = 3 * n;
    }
    if (int rc = pk.reserve(sizeof(float4) * npad * n_frames)) return rc;
    unsigned *d_ext = nullptr;
    if (ext) {
        // per frame {min x, y, z, max x, y, z} as order-preserving keys
        if (int rc = ext->reserve(sizeof(unsigned) * 6 * n_frames)) return rc;
        d_ext = ext->as<unsigned>();
        rdf_ext_init_kernel<<<(6 * n_frames + 255) / 256, 256, 0, c->stream>>>(d_ext,
                                                                              6 * n_frames);
        MDH_CUDA(cudaGetLastError());
        c->launches++;
    }
    const bool sort = tx != nullptr && d_ext != nullptr;
    if (sort) {
        if (int rc = R.xsort.reserve(sizeof(float4) * npad * n_frames)) return rc;
        if (int rc = tx->reserve(sizeof(float2) * (npad / tile) * n_frames)) return rc;
    }
    dim3 grid((unsigned)std::min<int64_t>((npad + 255) / 256, 2048), n_frames);
    rdf_pack_kernel<<<grid, 256, 0, c->stream>>>(dsrc, dstride,
                                                 (sort ? R.xsort : pk).as<float4>(), n, npad,
                                                 excl, R.drop_axis, d_ext,
                                                 R.boxes.as<FrameBox>() + f0);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    if (sort) {
        rdf_xsort_kernel<<<n_frames, 1024, 0, c->stream>>>(R.xsort.as<float4>(), pk.as<float4>(),
                                                           n, npad, d_ext, tile,
                                                           tx->as<float2>());
        MDH_CUDA(cudaGetLastError());
        c->launches++;
    }
    return MDH_OK;
}

int rdf_accumulate_impl(mdh_ctx *c, const float *pos1, int64_t s1, const float *pos2,
                        int64_t s2, int location, const float *box, int n_frames)
{
    RdfState &R = c->rdf;
    MDH_REQUIRE(R.configured, MDH_ESTATE, "rdf: accumulate before configure");
    MDH_REQUIRE(n_frames >= 1 && n_frames <= 65535, MDH_EINVAL,
                "rdf: n_frames per call must be in [1, 65535]");
    MDH_REQUIRE(box != nullptr, MDH_EINVAL, "rdf: box is NULL");
    MDH_REQUIRE(location == MDH_HOST || location == MDH_DEVICE, MDH_EINVAL,
                "rdf: invalid location");
    MDH_REQUIRE(pos1 != nullptr && (R.same || pos2 != nullptr), MDH_EINVAL,
                "rdf: coordinate pointer is NULL");
    MDH_REQUIRE(s1 >= 3 * R.n1, MDH_EINVAL, "rdf: frame_stride (%lld) < 3*n (%lld)",
                (long long)s1, (long long)(3 * R.n1));
    MDH_REQUIRE(R.same || s2 >= 3 * R.n2, MDH_EINVAL, "rdf: frame_stride (%lld) < 3*n (%lld)",
                (long long)s2, (long long)(3 * R.n2));

    // per-frame box: box_k and inv_k = (float)(1.0 / (double)box_k)  (Appendix A item 3)
    R.h_boxes.resize(n_frames);
    float min_edge = FLT_MAX;
    for (int f = 0; f < n_frames; ++f)
        for (int k = 0; k < 3; ++k) {
            const float b = box[3 * f + k];
            MDH_REQUIRE(b > FLT_EPSILON && std::isfinite(b), MDH_EINVAL,
                        "rdf: box edge %d of frame %d is not a positive length", k, f);
            R.h_boxes[f].box[k] = (double)b;
            R.h_boxes[f].inv[k] = (double)(float)(1.0 / (double)b);
            if (k != R.drop_axis) min_edge = std::min(min_edge, b);
        }
    // Which arithmetic the reference's capped_distance would use for each frame (SURVEY.md
    // Appendix A item 2, MDAnalysis' method choice): its grid search moves the coordinates
    // into the cell in float32 first, its brute force takes them as given.
    for (int f = 0; f < n_frames; ++f) {
        bool grid = R.n1 >= 10 && R.n2 >= 10;
        if (grid && (double)R.n1 * (double)R.n2 < 1e8)
            for (int k = 0; k < 3; ++k)
                if (R.r_hi > 0.3 * (double)box[3 * f + k]) grid = false;
        R.h_boxes[f].prewrap = R.prewrap_mode == MDH_WRAP_ALWAYS ||
                               (R.prewrap_mode == MDH_WRAP_AUTO && grid);
        R.h_boxes[f].pad = 0;
    }
    if (int rc = R.boxes.reserve(sizeof(FrameBox) * n_frames)) return rc;
    // upload through a pinned staging buffer so the call stays asynchronous; the
    // event guards the buffer against being rewritten before the copy has run
    if (R.h_boxes_cap < (size_t)n_frames) {
        if (R.h_boxes_pinned) {
            MDH_CUDA(cudaStreamSynchronize(c->stream));
            MDH_CUDA(cudaFreeHost(R.h_boxes_pinned));
            R.h_boxes_pinned = nullptr;
        }
        R.h_boxes_cap = std::max<size_t>(256, (size_t)n_frames);
        MDH_CUDA(cudaMallocHost(&R.h_boxes_pinned, sizeof(FrameBox) * R.h_boxes_cap));
    }
    MDH_TRACE("rdf_accumulate: %d frames, location %d; waiting for the previous box upload",
              n_frames, location);
    if (!R.ev_boxes) MDH_CUDA(cudaEventCreateWithFlags(&R.ev_boxes, cudaEventDisableTiming));
    else MDH_CUDA(cudaEventSynchronize(R.ev_boxes));
    MDH_TRACE("rdf_accumulate: boxes");
    memcpy(R.h_boxes_pinned, R.h_boxes.data(), sizeof(FrameBox) * n_frames);
    MDH_CUDA(cudaMemcpyAsync(R.boxes.p, R.h_boxes_pinned, sizeof(FrameBox) * n_frames,
                             cudaMemcpyHostToDevice, c->stream));
    MDH_CUDA(cudaEventRecord(R.ev_boxes, c->stream));

    int mode = R.mode;
    if (mode == MDH_RDF_AUTO) {
        // cells pay off when the cut-off sphere (circle, with a dropped axis) is a small part
        // of the box; min_edge leaves the dropped axis out
        const double r_cut = sqrt(R.thr_hi);
        const bool cells_ok = min_edge / (r_cut * 1.00001) >= 4.0 &&
                              (double)R.n1 * (double)R.n2 >= 4e6;
        mode = cells_ok ? MDH_RDF_CELLS : MDH_RDF_ALLPAIRS;
    }
    // Host input is cut into pieces so that the copy of one piece (copy stream) overlaps
    // the kernels of the previous one (compute stream).
    if (location == MDH_HOST) {
        int f0 = 0;
        for (int nf : mdh_plan_pieces(n_frames, 12.0 * (double)(R.n1 + (R.same ? 0 : R.n2)))) {
            if (int rc = rdf_accumulate_piece(c, pos1 + (int64_t)f0 * s1, s1,
                                              pos2 ? pos2 + (int64_t)f0 * s2 : nullptr, s2,
                                              location, f0, nf, mode)) return rc;
            f0 += nf;
        }
        return MDH_OK;
    }
    const int rc = rdf_accumulate_piece(c, pos1, s1, pos2, s2, location, 0, n_frames, mode);
    MDH_TRACE("rdf_accumulate: queued, rc %d", rc);
    return rc;
}

// One piece of an accumulate call: frames [f0, f0 + n_frames) of the batch whose boxes
// are already on the device (R.boxes / R.h_boxes).
static int rdf_accumulate_piece(mdh_ctx *c, const float *pos1, int64_t s1, const float *pos2,
                                int64_t s2, int location, int f0, int n_frames, int mode)
{
    RdfState &R = c->rdf;
    const int tile = kThreads * R.ipt;
    const int64_t pad1 = (R.n1 + tile - 1) / tile * tile;
    const int64_t pad2 = (R.n2 + tile - 1) / tile * tile;
    const bool use_filter = R.filter_ok && R.filter_mode != MDH_FILTER_OFF;

    int slot = 0;
    if (location == MDH_HOST) {
        if (int rc = c->stager.acquire(&slot)) return rc;
        if (int rc = rdf_upload_group(c, pos1, s1, location, R.n1, pad1, R.excl1, n_frames,
                                      R.raw1[slot], R.pk1, nullptr, true, f0)) return rc;
        if (!R.same)
            if (int rc = rdf_upload_group(c, pos2, s2, location, R.n2, pad2, R.excl2, n_frames,
                                          R.raw2[slot], R.pk2, nullptr, true, f0)) return rc;
        if (int rc = c->stager.publish(c->stream, slot)) return rc;
    }
    if (mode == MDH_RDF_CELLS) {
        // the cell-list pipeline sorts straight from the raw coordinates (rdf_cells.cu)
        const bool host = location == MDH_HOST;
        if (int rc = c->t_rdf.begin(c->stream)) return rc;
        if (int rc = rdf_cells_accumulate(
                c, host ? R.raw1[slot].as<float>() : pos1, host ? 3 * R.n1 : s1,
                R.same ? nullptr : (host ? R.raw2[slot].as<float>() : pos2),
                host ? 3 * R.n2 : s2, f0, n_frames, use_filter, g_sqrt_err_cached)) return rc;
        if (int rc = c->t_rdf.end(c->stream)) return rc;
        if (host)
            if (int rc = c->stager.retire(c->stream, slot)) return rc;
        return MDH_OK;
    }
    // the filter kernel's groups are sorted by x (x-clean tile pairs); the exact kernel
    // reads the same sorted rows
    if (int rc = rdf_upload_group(c, pos1, s1, location, R.n1, pad1, R.excl1, n_frames,
                                  R.raw1[slot], R.pk1, use_filter ? &R.ext1 : nullptr, false,
                                  f0, use_filter ? &R.tx1 : nullptr, tile))
        return rc;
    if (!R.same)
        if (int rc = rdf_upload_group(c, pos2, s2, location, R.n2, pad2, R.excl2, n_frames,
                                      R.raw2[slot], R.pk2, use_filter ? &R.ext2 : nullptr,
                                      false, f0, use_filter ? &R.tx2 : nullptr, tile)) return rc;
    // the raw staging slot has been consumed by the pack kernels
    if (location == MDH_HOST)
        if (int rc = c->stager.retire(c->stream, slot)) return rc;
    if (use_filter)
        if (int rc = rdf_filter_prepare(c, f0, n_frames, g_sqrt_err_cached)) return rc;

    if (int rc = c->t_rdf.begin(c->stream)) return rc;

    {
        PairParams P;
        P.p1 = R.pk1.as<float4>();
        P.p2 = R.same ? P.p1 : R.pk2.as<float4>();
        P.pad1 = pad1; P.pad2 = R.same ? pad1 : pad2;
        P.n1 = (int)R.n1; P.n2 = (int)R.n2;
        P.boxes = R.boxes.as<FrameBox>() + f0;
        P.thr = R.thr.as<double>();
        P.n_bins = R.n_bins;
        P.guess = rdf_bin_guess(R);
        P.same = R.same;
        P.counts = R.counts.as<unsigned long long>();
        const int n_itiles = (int)(pad1 / tile);
        P.n_jtiles = (int)(P.pad2 / tile);
        const int64_t target = (int64_t)c->sm_count * 2 * 6;
        int64_t n_jchunks = (target + (int64_t)n_itiles * n_frames - 1) /
                            ((int64_t)n_itiles * n_frames);
        n_jchunks = std::max<int64_t>(1, std::min<int64_t>(n_jchunks, P.n_jtiles));
        // a block's u32 partial histogram must not overflow: <= 2^31 weighted pairs
        n_jchunks = std::max<int64_t>(n_jchunks, (P.n_jtiles + 1023) / 1024);
        P.jtiles_per_chunk = (int)((P.n_jtiles + n_jchunks - 1) / n_jchunks);
        P.n_jchunks = (int)((P.n_jtiles + P.jtiles_per_chunk - 1) / P.jtiles_per_chunk);
        dim3 grid((unsigned)(n_itiles * P.n_jchunks), (unsigned)n_frames);
        const bool excl = R.excl1 > 0;
        P.filt = nullptr;
        P.fc = use_filter ? R.fca : R.fc;       // R.fca: set by rdf_filter_prepare
        P.fast_bins = R.fast_bins ? 1 : 0;
        P.fstats = R.fstats.as<unsigned long long>();
        P.xform = nullptr;
        if (use_filter) {
            const int64_t n_pairs = (int64_t)n_itiles * P.n_jtiles;
            if (int rc = R.xform.reserve(n_pairs * n_frames)) return rc;
            const float2 *tx1 = R.tx1.as<float2>(), *tx2 = R.same ? tx1 : R.tx2.as<float2>();
            rdf_cleanx_forms_kernel<<<dim3((unsigned)((n_pairs + 127) / 128), n_frames), 128, 0,
                                      c->stream>>>(tx1, tx2, n_itiles, P.n_jtiles, P.boxes,
                                                   R.xform.as<unsigned char>());
            MDH_CUDA(cudaGetLastError());
            c->launches++;
            P.xform = R.xform.as<unsigned char>();
        }
        if (use_filter) {
            // the filter kernel takes every frame whose error bound is small against a
            // bin; the exact kernel below then only runs the frames it declined
            P.filt = R.filt.as<FrameFilter>();
            if (int rc = rdf_filter_launch(c, P, grid, excl,
                                           R.filter_mode == MDH_FILTER_AUDIT)) return rc;
        }
        int rc = R.hist == MDH_HIST_LANE_PRIVATE
                     ? launch_allpairs_dyn<MDH_HIST_LANE_PRIVATE>(c, P, grid, excl, R.fast_bins,
                                                                  R.ipt)
                     : launch_allpairs_dyn<MDH_HIST_WARP_ATOMIC>(c, P, grid, excl, R.fast_bins,
                                                                 R.ipt);
        if (rc) return rc;
        // pair evaluations the kernel performs (upper-triangle tiles when same_group)
        int64_t ev;
        if (R.same) {
            ev = 0;
            for (int a = 0; a < n_itiles; ++a) {
                const int64_t ca = std::min<int64_t>(tile, R.n1 - (int64_t)a * tile);
                ev += ca * (R.n1 - (int64_t)a * tile);          // j >= a*tile
            }
        } else {
            ev = R.n1 * R.n2;
        }
        R.evals += ev * n_frames;
    }
    return c->t_rdf.end(c->stream);
}
