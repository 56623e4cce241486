// rdf_device.cuh -- device helpers shared by the pair kernels (rdf.cu, rdf_cells.cu).
// See rdf.cu for the statement of the reference arithmetic these implement.
#pragma once

#include <cuda_pipeline.h>
#include <float.h>
#include <math.h>
#include <string.h>

#include "common.cuh"

namespace rdfdev {

constexpr int kThreads = 256;          // 8 warps
constexpr int kWarps = kThreads / 32;
constexpr double kMagic = 6755399441055744.0;  // 1.5 * 2^52
constexpr float kMagicF = 12582912.0f;         // 1.5 * 2^23
constexpr size_t kMaxSmem = 227 * 1024;

// ---- pack: float[F][n][3] -> float4[F][npad] (x, y, z, exclusion block id) ------
// Also reduces the coordinate extents of every frame (per axis minimum and maximum,
// as order-preserving unsigned keys) for the error bound of the fp32 filter.

__device__ __forceinline__ unsigned ext_key(float f)
{
    // the move is opaque on purpose: seeing a float, nvcc sets the sign bit with
    // FADD -|x|, -0, which turns every NaN into the canonical 0x7fffffff (= key of -0)
    unsigned b;
    asm("mov.b32 %0, %1;" : "=r"(b) : "f"(f));
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ inline float ext_unkey(unsigned k)
{
    const unsigned b = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
    return __uint_as_float(b);
#else
    float f; memcpy(&f, &b, 4); return f;
#endif
}

// Restated MDAnalysis `_ortho_pbc` (lib/include/calc_distances.h, applied by the grid search
// FastNS to both coordinate sets; SURVEY.md Appendix A item 4; [recall], not pinned against
// MDAnalysis): one coordinate into the primary cell, IN FLOAT32 STORAGE.  A single box
// shift is computed in double and stored as float (so -1e-9 becomes exactly box); farther
// coordinates take floor(c / box) shifts in float arithmetic plus one corrective shift.
// oracle/mdh_oracle.c::mdho_ortho_pbc is the same code on the CPU.
__device__ __forceinline__ float ortho_pbc_f32(float c, double boxd)
{
    const float box = (float)boxd;                   // boxd is a float32 value
    double crd = (double)c;
    if (crd < 0.0) {
        crd += boxd;
        if (crd < 0.0) {
            const int s = (int)floor((double)c * (1.0 / boxd));
            c = __fsub_rn(c, __fmul_rn((float)s, box));
            if (c < 0.f) c = __fadd_rn(c, box);
        } else {
            c = (float)crd;
        }
    }
    if (crd >= boxd) {
        crd -= boxd;
        if (crd >= boxd) {
            const int s = (int)floor((double)c * (1.0 / boxd));
            c = __fsub_rn(c, __fmul_rn((float)s, box));
            if (c >= box) c = __fsub_rn(c, box);
        } else {
            c = (float)crd;
        }
    }
    return c;
}

static __global__ void rdf_ext_init_kernel(unsigned *ext, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) ext[i] = (i % 6) < 3 ? 0xffffffffu : 0u;
}

// ext: unsigned[F][6] = {min x, y, z, max x, y, z} keys, initialised by
// rdf_ext_init_kernel (or nullptr)
static __global__ void __launch_bounds__(256)
    rdf_pack_kernel(const float *__restrict__ raw, int64_t frame_stride,
                    float4 *__restrict__ out, int64_t n, int64_t npad, int64_t excl,
                    int drop_axis, unsigned *__restrict__ ext,
                    const FrameBox *__restrict__ boxes)
{
    __shared__ float stage[3 * 256];
    __shared__ unsigned red[8][6];
    const int frame = blockIdx.y;
    const int tid = threadIdx.x;
    const float *src = raw + (int64_t)frame * frame_stride;
    float4 *dst = out + (int64_t)frame * npad;
    const bool prewrap = boxes != nullptr && boxes[frame].prewrap != 0;
    unsigned lo[3] = {0xffffffffu, 0xffffffffu, 0xffffffffu}, hi[3] = {0u, 0u, 0u};
    // 256 particles per step: their 768 floats are read as one contiguous run
    // (coalesced, unlike three stride-3 loads per thread) and regrouped through
    // shared memory
    for (int64_t i0 = (int64_t)blockIdx.x * 256; i0 < npad; i0 += (int64_t)gridDim.x * 256) {
        const int64_t f0 = 3 * i0, fend = 3 * n;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int64_t f = f0 + k * 256 + tid;
            stage[k * 256 + tid] = f < fend ? src[f] : 0.f;
        }
        __syncthreads();
        const int64_t i = i0 + tid;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < n) {
            v.x = stage[3 * tid];
            v.y = stage[3 * tid + 1];
            v.z = stage[3 * tid + 2];
            if (drop_axis == 0) v.x = 0.f;
            if (drop_axis == 1) v.y = 0.f;
            if (drop_axis == 2) v.z = 0.f;
            if (prewrap) {
                v.x = ortho_pbc_f32(v.x, boxes[frame].box[0]);
                v.y = ortho_pbc_f32(v.y, boxes[frame].box[1]);
                v.z = ortho_pbc_f32(v.z, boxes[frame].box[2]);
            }
            v.w = __int_as_float((int)(excl > 0 ? i / excl : i));
            const unsigned kx = ext_key(v.x), ky = ext_key(v.y), kz = ext_key(v.z);
            lo[0] = min(lo[0], kx); hi[0] = max(hi[0], kx);
            lo[1] = min(lo[1], ky); hi[1] = max(hi[1], ky);
            lo[2] = min(lo[2], kz); hi[2] = max(hi[2], kz);
        }
        if (i < npad) dst[i] = v;
        __syncthreads();
    }
    if (ext) {
        // block-level extents first: six global atomics per block, not per warp
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
            if (tid < 3) { if (v != 0xffffffffu) atomicMin(&ext[frame * 6 + tid], v); }
            else if (v != 0u) atomicMax(&ext[frame * 6 + tid], v);
        }
    }
}

// ---- the reference arithmetic, one coordinate ---------------------------------

__device__ __forceinline__ double min_image_sq(float a, float b, double box, double inv)
{
    const float df = __fsub_rn(b, a);
    const double d = (double)df;
    const double s = __dmul_rn(inv, d);
    const double r = __dsub_rn(__dadd_rn(s, kMagic), kMagic);
    const double m = __dmul_rn(box, __dsub_rn(s, r));
    return __dmul_rn(m, m);
}

__device__ __forceinline__ double pair_d2(float xi, float yi, float zi, const float4 &pj,
                                          const FrameBox &fb)
{
    const double sx = min_image_sq(xi, pj.x, fb.box[0], fb.inv[0]);
    const double sy = min_image_sq(yi, pj.y, fb.box[1], fb.inv[1]);
    const double sz = min_image_sq(zi, pj.z, fb.box[2], fb.inv[2]);
    return __dadd_rn(__dadd_rn(sx, sy), sz);
}

// ---- bin lookup -----------------------------------------------------------------
// sT[0..n_bins] are the squared thresholds.  A "slot" is bin + 1: slot 0 = below
// T[0] (or NaN), slots 1..n_bins = bins 0..n_bins-1, slot n_bins+1 = at or above
// T[n_bins].  Slots 0 and n_bins+1 are never counted.

struct BinGuess {
    float scale;     // n_bins / (r_hi - r_lo)
    float offset;    // -r_lo * scale + 0.5 - margin
};

// exact: binary search (always correct; used when the guess cannot be certified)
static __device__ __noinline__ int slot_search(double d2, const double *sT, int n_bins)
{
    if (!(d2 < sT[n_bins])) return n_bins + 1;       // above range, inf, NaN
    if (d2 < sT[0]) return 0;
    int lo = 0, hi = n_bins;
    while (hi - lo > 1) {
        const int mid = (lo + hi) >> 1;
        if (d2 >= sT[mid]) lo = mid; else hi = mid;
    }
    return lo + 1;
}

// fast: branch-free.  A float estimate of (sqrt(d2) - r_lo) * scale, biased low by
// `margin`, gives j = floor(estimate + 1) with  j - 1 <= true bin <= j  (certified
// per configuration by rdf_selfcheck_kernel); one fp64 compare against T[j]
// settles it.  No XU conversions: d2 -> float by bit manipulation (truncation),
// float -> int by the 1.5*2^23 magic add.
// Returns j in [0, n_bins] with  j - 1 <= true bin <= j  and sets below = (d2 < T[j]):
// the pair belongs to bin j - 1 if below (not counted when j == 0), else to bin j
// (not counted when j == n_bins, which is also where inf / NaN end up).
__device__ __forceinline__ int slot_fast_parts(double d2, const double *sT, int n_bins,
                                               const BinGuess g, bool &below)
{
    unsigned hi = (unsigned)__double2hiint(d2);
    const unsigned lo = (unsigned)__double2loint(d2);
    // clamp the exponent into float range: below 2^-127 (and 0) -> ~0; huge, inf
    // and NaN -> ~2^127 (they end in the "above range" slot)
    hi = min(max(hi, 0x38000000u), 0x47e00000u);
    // fp64 -> fp32 bits by truncation: the shifted word carries exponent bit 8 in
    // the sign position (cleared) and needs its 8-bit exponent re-biased by -896,
    // i.e. bit 30 flipped
    const float f =
        __uint_as_float((__funnelshift_l(lo, hi, 3) & 0x7fffffffu) ^ 0x40000000u);
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(f));
    const float e = __fadd_rn(fmaf(r, g.scale, g.offset), kMagicF);
    int j = __float_as_int(e) - 0x4B400000;          // rint(estimate + 0.5 - margin)
    j = min(max(j, 0), n_bins);
    below = d2 < sT[j];                              // false for NaN
    return j;
}

__device__ __forceinline__ int slot_fast(double d2, const double *sT, int n_bins,
                                         const BinGuess g)
{
    bool below;
    const int j = slot_fast_parts(d2, sT, n_bins, g, below);
    return j + (below ? 0 : 1);
}

template <bool FAST>
__device__ __forceinline__ int slot_of(double d2, const double *sT, int n_bins,
                                       const BinGuess g)
{
    return FAST ? slot_fast(d2, sT, n_bins, g) : slot_search(d2, sT, n_bins);
}

// Certifies slot_fast for one configuration: at every threshold and its fp64
// neighbours (where a biased guess is most exposed) the fast slot must equal the
// exact one.  *bad counts disagreements.
static __global__ void rdf_selfcheck_kernel(const double *__restrict__ thr, int n_bins,
                                            BinGuess g, int *bad)
{
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k > n_bins) return;
    const double t = thr[k];
    // neighbours of a non-negative double through its bit pattern
    auto up = [](double x) { return __longlong_as_double(__double_as_longlong(x) + 1); };
    auto down = [](double x) {
        return x > 0.0 ? __longlong_as_double(__double_as_longlong(x) - 1) : -1.0;
    };
    const double probes[5] = {
        t, down(t), up(t),
        k < n_bins ? 0.5 * (t + thr[k + 1]) : t * 1.5 + 1.0,
        k < n_bins ? down(thr[k + 1]) : t * 4.0 + 1e30};
    int wrong = 0;
    for (int p = 0; p < 5; ++p) {
        const double d2 = probes[p];
        if (!(d2 >= 0.0)) continue;
        if (slot_fast(d2, thr, n_bins, g) != slot_search(d2, thr, n_bins)) ++wrong;
    }
    if (k == 0) {
        if (slot_fast(0.0, thr, n_bins, g) != slot_search(0.0, thr, n_bins)) ++wrong;
        if (slot_fast(1e-300, thr, n_bins, g) != slot_search(1e-300, thr, n_bins)) ++wrong;
        const double nan = __longlong_as_double(0x7ff8000000000000ll);
        if (slot_fast(nan, thr, n_bins, g) != n_bins + 1) ++wrong;
        if (slot_fast(INFINITY, thr, n_bins, g) != n_bins + 1) ++wrong;
        if (slot_fast(1e300, thr, n_bins, g) != n_bins + 1) ++wrong;
    }
    if (wrong) atomicAdd(bad, wrong);
}

// Checks slot_fast for one configuration over EVERY double d2 >= 0 (certified or not).
// slot_fast_parts builds its float from the clamped hi word and the top 3 bits of the lo
// word, so the guess j is constant on each of kGuessClasses classes (hi in [kGuessHiMin,
// kGuessHiMax], lo >> 29); slot_search is monotone in d2 and the compare against T[j] is
// exact, so slot_fast is right on a whole class iff it is right at the class's smallest
// and largest d2.  The clamped end classes absorb every d2 below 2^-127 (from 0 up) and
// every finite d2 above 2^127; +inf and NaN (both signs, every lo >> 29) are checked
// separately.  out[0] += disagreements, out[1] = min(out[1], bits of a bad d2).
constexpr unsigned kGuessHiMin = 0x38000000u, kGuessHiMax = 0x47e00000u;
constexpr long long kGuessClasses = ((long long)(kGuessHiMax - kGuessHiMin) + 1) * 8;

static __global__ void __launch_bounds__(256)
    rdf_guess_audit_kernel(const double *__restrict__ thr, int n_bins, BinGuess g,
                           unsigned long long *out)
{
    extern __shared__ double sTa[];
    for (int k = threadIdx.x; k <= n_bins; k += blockDim.x) sTa[k] = thr[k];
    __syncthreads();
    unsigned long long bad = 0, first = ~0ull;
    auto check = [&](unsigned long long bits) {
        const double d2 = __longlong_as_double((long long)bits);
        if (slot_fast(d2, sTa, n_bins, g) != slot_search(d2, sTa, n_bins)) {
            ++bad;
            first = min(first, bits);
        }
    };
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long c = (long long)blockIdx.x * blockDim.x + threadIdx.x; c < kGuessClasses;
         c += stride) {
        const unsigned long long hi = kGuessHiMin + (unsigned long long)(c >> 3);
        const unsigned long long t = (unsigned long long)(c & 7) << 29;
        const unsigned long long hi_min = hi == kGuessHiMin ? 0ull : hi;
        const unsigned long long hi_max = hi == kGuessHiMax ? 0x7fefffffull : hi;
        check((hi_min << 32) | t);
        check((hi_max << 32) | t | 0x1fffffffull);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        check(0x7ff0000000000000ull);                                  // +inf
        for (unsigned long long t = 0; t < 8; ++t) {
            check(0x7ff8000000000000ull | (t << 29));                  // NaN
            check(0xfff8000000000000ull | (t << 29));
        }
    }
    for (int o = 16; o; o >>= 1) {
        bad += __shfl_xor_sync(0xffffffffu, bad, o);
        first = min(first, __shfl_xor_sync(0xffffffffu, first, o));
    }
    if ((threadIdx.x & 31) == 0 && bad) {
        atomicAdd(&out[0], bad);
        atomicMin(&out[1], first);
    }
}

// fast slot minus exact slot of one d2 (the audit's first disagreement)
static __global__ void rdf_guess_probe_kernel(const double *__restrict__ thr, int n_bins,
                                              BinGuess g, double d2, int *diff)
{
    *diff = slot_fast(d2, thr, n_bins, g) - slot_search(d2, thr, n_bins);
}

// ---- shared-memory layout and histogram privatisation ------------------------------

// Per-warp u32 histogram for the shared-atomic scheme: one pad word (receives the
// rare "below range" pairs), n_bins bins, then 32 per-lane trash words so that the
// many "above range" pairs never contend for one address.  Every pair then issues
// exactly one unconditional RED.shared (no branch around the atomic).
__host__ __device__ inline int warp_hist_words(int n_bins) { return n_bins + 33; }

__device__ __forceinline__ void red_shared(unsigned smem_addr, unsigned v)
{
    asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(smem_addr), "r"(v) : "memory");
}

__host__ __device__ inline size_t align16(size_t x) { return (x + 15) & ~size_t(15); }
__host__ __device__ inline int priv_words(int n_bins) { return (n_bins + 2 + 3) / 4; }

// bytes of histogram storage behind the threshold table
template <int HIST>
__host__ __device__ inline size_t hist_smem_bytes(int n_bins)
{
    if (HIST == MDH_HIST_WARP_ATOMIC)
        return sizeof(unsigned) * kWarps * warp_hist_words(n_bins);
    return sizeof(unsigned) * ((size_t)kWarps * priv_words(n_bins) * 32 + n_bins);
}

// Lane-private packed histograms: lane l of warp w owns the 32-bit words
// priv[(w*n_words + word)*32 + l]; each word holds four 8-bit slot counters
// (slot = 4*word + byte), so the byte read-modify-write is bank-conflict free and
// needs no atomics.  A lane makes at most 254 increments between flushes, so no
// counter can overflow.
__device__ __forceinline__ void priv_add(unsigned char *lane_base, int slot, unsigned inc)
{
    unsigned char *p = lane_base + (((unsigned)slot & ~3u) << 5) + ((unsigned)slot & 3u);
    *p = (unsigned char)(*p + inc);
}

__device__ __forceinline__ void priv_flush(unsigned *priv_w, unsigned *bhist, int n_words,
                                           int n_bins, int lane, unsigned weight)
{
    __syncwarp();
    for (int w = 0; w < n_words; ++w) {
        const unsigned v = priv_w[w * 32 + lane];
        if (__any_sync(0xffffffffu, v != 0)) {
            priv_w[w * 32 + lane] = 0;
            const unsigned a = __reduce_add_sync(0xffffffffu, v & 0x00ff00ffu);
            const unsigned b = __reduce_add_sync(0xffffffffu, (v >> 8) & 0x00ff00ffu);
            if (lane < 4) {
                unsigned val = (lane & 1) ? b : a;
                val = (lane & 2) ? (val >> 16) : (val & 0xffffu);
                const int bin = 4 * w + lane - 1;          // slot - 1
                if (bin >= 0 && bin < n_bins && val) atomicAdd(&bhist[bin], val * weight);
            }
        }
    }
    __syncwarp();
}

// ---- packed fp32 arithmetic (sm_100: FADD2 / FMUL2 / FFMA2, two IEEE round-to-nearest
// operations per issue slot; a scalar operand is broadcast by the hardware) -----------
typedef unsigned long long f32x2;

__device__ __forceinline__ f32x2 pk2(float lo, float hi)
{
    f32x2 d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi));
    return d;
}
__device__ __forceinline__ void upk2(f32x2 v, float &lo, float &hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b)
{
    f32x2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b)
{
    f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c)
{
    f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}

__device__ __forceinline__ f32x2 abs2(f32x2 v)
{
    float lo, hi;
    upk2(v, lo, hi);
    return pk2(fabsf(lo), fabsf(hi));     // ptxas folds this into the |x| operand of FADD2
}

// The fp32 evaluation of TWO pairs at once: coordinate differences d = b + a per axis
// with a = the NEGATED coordinates of the group-1 particle(s) and b = the group-2
// particle(s) -- the all-pairs kernel packs two group-1 particles against one tile row
// (b broadcast), the cell-list kernel one group-1 particle (a broadcast) against two
// neighbours.  Returns the fixed-point bin coordinates u0, u1 (relative to slot 0 when
// LOWER, else with the bits of 1.5*2^(23-k) still added).  Main loops and exact
// re-evaluations go through this one function, so they see identical bits.
// first half: packed squared minimum-image distances of two pairs.  Two forms of the
// minimum image (FrameFilter::halfbox; the error bound of each: filter_prepare_frame):
//   HALF = false  m = fma(-box, rint(df * inv), df)        4 packed instructions per axis
//   HALF = true   m = ||df| - box/2| - box/2               2 packed instructions per axis,
//                 |m| is the minimum image for |df| <= 1.5 box (only |m| matters for m^2)
//   CX (HALF only, x axis): m_x = bx + ax, no fold -- the all-pairs kernel's x-clean tile
//                 pairs (filter_cleanx_form), whose operands already carry the shift S
template <bool HALF, bool CX = false>
__device__ __forceinline__ f32x2 filter_d2(f32x2 ax, f32x2 ay, f32x2 az, f32x2 bx, f32x2 by,
                                           f32x2 bz, const FrameFilter &ff)
{
    static_assert(HALF || !CX, "the x-clean form is a variant of the half-box form");
    const f32x2 dx = add2(bx, ax);
    const f32x2 dy = add2(by, ay);
    const f32x2 dz = add2(bz, az);
    f32x2 mx, my, mz;
    if (HALF) {
        const f32x2 hx = pk2(ff.nhalf[0], ff.nhalf[0]);
        const f32x2 hy = pk2(ff.nhalf[1], ff.nhalf[1]);
        const f32x2 hz = pk2(ff.nhalf[2], ff.nhalf[2]);
        mx = CX ? dx : add2(abs2(add2(abs2(dx), hx)), hx);
        my = add2(abs2(add2(abs2(dy), hy)), hy);
        mz = add2(abs2(add2(abs2(dz), hz)), hz);
    } else {
        const f32x2 magic = pk2(kMagicF, kMagicF), nmagic = pk2(-kMagicF, -kMagicF);
        const f32x2 rx = add2(fma2(dx, pk2(ff.inv[0], ff.inv[0]), magic), nmagic);
        const f32x2 ry = add2(fma2(dy, pk2(ff.inv[1], ff.inv[1]), magic), nmagic);
        const f32x2 rz = add2(fma2(dz, pk2(ff.inv[2], ff.inv[2]), magic), nmagic);
        mx = fma2(pk2(ff.nbox[0], ff.nbox[0]), rx, dx);
        my = fma2(pk2(ff.nbox[1], ff.nbox[1]), ry, dy);
        mz = fma2(pk2(ff.nbox[2], ff.nbox[2]), rz, dz);
    }
    return fma2(mz, mz, fma2(my, my, mul2(mx, mx)));
}

// second half: square roots and fixed-point bin coordinates
template <bool LOWER>
__device__ __forceinline__ void filter_bin2(f32x2 d2, float scale, float offm, unsigned cbits,
                                            unsigned &u0, unsigned &u1)
{
    float a, b, s0, s1;
    upk2(d2, a, b);
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s0) : "f"(a));
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(s1) : "f"(b));
    const f32x2 e = fma2(pk2(s0, s1), pk2(scale, scale), pk2(offm, offm));
    upk2(e, a, b);
    u0 = __float_as_uint(a) - (LOWER ? cbits : 0u);
    u1 = __float_as_uint(b) - (LOWER ? cbits : 0u);
}

template <bool LOWER, bool HALF = false, bool CX = false>
__device__ __forceinline__ void filter_eval2(f32x2 ax, f32x2 ay, f32x2 az, f32x2 bx, f32x2 by,
                                             f32x2 bz, const FrameFilter &ff, float scale,
                                             float offm, unsigned cbits, unsigned &u0,
                                             unsigned &u1)
{
    filter_bin2<LOWER>(filter_d2<HALF, CX>(ax, ay, az, bx, by, bz, ff), scale, offm, cbits, u0,
                       u1);
}

// The x form of one tile pair of the all-pairs filter kernel, from the x extents of its
// i-tile [lo_i, hi_i] and j-tile [lo_j, hi_j] (float32 values) and the box edge L (a
// float32 value); every x difference xj - xi of the pair lies in [lo_j - hi_i, hi_j - lo_i]
// (exact in fp64).  If that interval shifted by S in {0, +L, -L} lies inside (-h + delta,
// h - delta), h = L/2, every pair has the same x image and m_x = (xj - S) - xi is ONE
// rounded FADD (DESIGN.md section 4.1b):
//   0  dirty: the half-box fold, as for every other body
//   1  S = 0
//   2  S = +L, applied to the j-tile: xj - L is exact (Sterbenz) for xj in [L/2, 2L]
//   3  S = -L, applied to the negated i-coordinates: L - xi is exact for xi in [L/2, 2L],
//      and (L - xi) - L gives -xi back exactly
// delta = 2^-20 L > 2^-23 * 1.5 L: the float32 difference df = fl(xj - xi) of the
// reference then also has |df - S| < h, so |df - S| is df's minimum image.  NaN extents
// compare false: dirty.
__host__ __device__ inline int filter_cleanx_form(float lo_i, float hi_i, float lo_j, float hi_j,
                                                  float L)
{
    const double l = (double)L, h = 0.5 * l, dl = l * (1.0 / 1048576.0);
    const double lo = (double)lo_j - (double)hi_i, hi = (double)hi_j - (double)lo_i;
    const bool sterbenz_j = (double)lo_j >= h && (double)hi_j <= 2.0 * l;
    const bool sterbenz_i = (double)lo_i >= h && (double)hi_i <= 2.0 * l;
    if (lo > -h + dl && hi < h - dl) return 1;
    if (sterbenz_j && lo - l > -h + dl && hi - l < h - dl) return 2;
    if (sterbenz_i && lo + l > -h + dl && hi + l < h - dl) return 3;
    return 0;
}

// Per-frame parameters of the fp32 filter from the frame's box and coordinate extents
// (error bound: rdf_filter.cu header and DESIGN.md 4.1b).  e1 / e2: the six extent keys
// {min x, y, z, max x, y, z} of the two groups.
struct FilterPrep {            // per configuration (host)
    int k;
    int halfbox;               // frames may take the half-box minimum image (all-pairs
                               // kernel; the cell-list kernels evaluate the rint form only)
    double scale;              // n_bins / (r_hi - r_lo)
    double d_max;              // largest distance that can still be binned
    double sqrt_err;           // measured relative error of sqrt.approx.ftz.f32
    double offbase;            // FilterConst::offbase
    double fscale;             // FilterConst::scale (the float32 value)
    int hslots;                // FilterConst::hslots if half-box frames may run unclamped, else 0
};

// Upper bound of the fixed-point bin coordinate (in bins, relative to slot 0) that
// filter_d2 + filter_bin2 can produce when every computed |m_k| <= mb[k]; c0 = offm -
// 1.5*2^(23-k) is the frame's offset coordinate.  floor() of it is the largest slot the
// frame can reach (DESIGN.md section 4.1b):
//     d2  <= (mx^2 + my^2 + mz^2) (1 + 2^-24)^3      mul, fma, fma, each rounding up
//     s   <= sqrt(d2) (1 + sqrt_err)                   sqrt.approx, measured
//     u   <= s * scale + c0 + 2^-(k+1)                 fma in the binade of 1.5*2^(23-k)
// scale is the float32 value the kernel multiplies by, so its rounding is exact here.
__host__ __device__ inline double filter_reach(const double mb[3], double fscale, double c0,
                                               double sqrt_err, int k)
{
    const double e24 = 1.0 / 16777216.0;
    const double d2 = (mb[0] * mb[0] + mb[1] * mb[1] + mb[2] * mb[2]) * (1.0 + 4.0 * e24);
    const double s = sqrt(d2) * (1.0 + sqrt_err);
    // (1 + 1e-12): the fp64 roundings of this evaluation
    return (s * fscale + c0) * (1.0 + 1e-12) + 1.0 / (double)(2u << k);
}

// Bound on the computed |m_k| of the half-box form for a frame whose |df_k| <= D_k <= 1.5
// box_k (h = box_k / 2): both FADDs round towards a result in [-h, h], and for |df| < h
// the result is within 2^-24 h (one rounding) of |df|.
__host__ __device__ inline double filter_halfbox_mbound(double D, double h)
{
    return fmin(D + h / 8388608.0, h) * (1.0 + 1.0 / 8388608.0);
}

// bits of a float, on the host and on the device
__host__ __device__ inline unsigned f32_bits(float f)
{
#ifdef __CUDA_ARCH__
    return __float_as_uint(f);
#else
    unsigned b; memcpy(&b, &f, 4); return b;
#endif
}

// Host and device: the preparation kernels run it per frame, mdh_rdf_filter_window on the
// host (device-free tests of the window).  mu (optional): the bound in bins, before the
// 1.25 margin of the window.  CLEANX: the all-pairs filter kernel, whose x-clean tile pairs
// (filter_cleanx_form) widen the half-box term of the x axis.
template <bool CLEANX = false>
__host__ __device__ inline FrameFilter filter_prepare_frame(const FrameBox &fb, const unsigned *e1,
                                                            const unsigned *e2, const FilterPrep &Q,
                                                            double *mu_out = nullptr)
{
    const double e24 = 1.0 / 16777216.0;
    bool ok = true, half = Q.halfbox != 0;
    double a2 = 0.0, h2 = 0.0, mb[3];
    FrameFilter ff;
    for (int k = 0; k < 3; ++k) {
        const float e4[4] = {ext_unkey(e1[k]), ext_unkey(e1[3 + k]), ext_unkey(e2[k]),
                             ext_unkey(e2[3 + k])};
        // inf / NaN coordinates (all-ones exponent) make the bound meaningless
        for (int q = 0; q < 4; ++q)
            if ((f32_bits(e4[q]) & 0x7f800000u) == 0x7f800000u) ok = false;
        const double lo1 = (double)e4[0], hi1 = (double)e4[1];
        const double lo2 = (double)e4[2], hi2 = (double)e4[3];
        // D >= every |df| of the frame, the float32 rounding of df included
        const double D = fmax(fmax(hi2 - lo1, hi1 - lo2), 0.0) * (1.0 + 2.0 * e24);
        const double box = fb.box[k], inv = fb.inv[k];
        // the magic-number rounding needs |df * inv| well inside 2^22
        if (!(D * inv < 1048576.0)) ok = false;
        const double eps_b = fabs(box * inv - 1.0);       // exact: 24-bit x 24-bit
        // first term: the fp32 rounding of the minimum image; then the reference vs the
        // exact minimum image of df: eps_b * D from its float32 inverse box, D * 2^-51
        // from its fp64 roundings -- the product inv*df may also round across a
        // half-integer that the exact product does not cross (|m| changes by at most
        // box * 2^-52 * |inv*df| <= 2^-51 D)
        // rint form: one rounding of fma(-box, r, df), |m_f| <= box/2 + eps_b D + 2^-24 D
        const double a = e24 * (0.5 * box + eps_b * D + e24 * D) * (1.0 + 1e-6) + eps_b * D +
                         D / 2251799813685248.0 + 1e-30;
        a2 += a * a;
        // half-box form, |df| <= D <= 1.5 box: e = |df| - h, m = |e| - h with h = box/2.
        // By Sterbenz at most one of the two rounds, and the rounded result lies in
        // [h/2, h] (|df| < h/2: e; h/2 <= |df| <= box: m) or in [h, 2h] (|df| > box: e).
        if (!(D <= 1.5 * box)) half = false;
        double ah = e24 * (D <= box ? 0.5 * box : box) * (1.0 + 1e-6) + eps_b * D +
                    D / 2251799813685248.0 + 1e-30;
        // x axis of the all-pairs kernel, x-clean tile pairs (filter_cleanx_form): m_x =
        // fl(xj - xi - S) with |xj - xi - S| < h rounds once (2^-24 h) from the exact
        // difference, which is within 2^-24 D of the reference's df - S
        if (CLEANX && k == 0)
            ah = fmax(ah, e24 * (0.5 * box + D) * (1.0 + 1e-6) + eps_b * D +
                              D / 2251799813685248.0 + 1e-30);
        h2 += ah * ah;
        mb[k] = filter_halfbox_mbound(D, 0.5 * box);
        ff.nbox[k] = -(float)box;                          // box is a float32 value
        ff.inv[k] = (float)inv;
        ff.nhalf[k] = -0.5f * (float)box;                  // exact
    }
    if (half) a2 = h2;
    const double two_k = (double)(1u << Q.k);
    const double mu = Q.scale * (sqrt(a2) + Q.d_max * (1.5 * e24 * 1.001 + Q.sqrt_err)) +
                      e24 * Q.scale * Q.d_max * 1.001 + 1.0 / two_k + 1e-9;
    if (mu_out) *mu_out = mu;
    const double m = ceil(1.25 * mu * two_k) + 1.0;
    if (!(m >= 1.0) || !(2.0 * m + 1.0 < two_k / 8.0)) ok = false;
    if (ok) {
        // shifted coordinate: exactly representable (a multiple of 2^-k in the binade)
        ff.offm = (float)(Q.offbase + m / two_k);
        ff.wlim = 2u * (unsigned)m + 1u;
    } else {
        ff.offm = 0.f;
        ff.wlim = 0u;
    }
    ff.halfbox = ok && half ? 1 : 0;
    // the frame's own reachable slot must be a word of the launch's histogram
    const double magic = 1.5 * (double)(1u << (23 - Q.k));
    ff.unclamped = ff.halfbox && Q.hslots > 0 &&
                   filter_reach(mb, Q.fscale, (double)ff.offm - magic, Q.sqrt_err, Q.k) <
                       (double)Q.hslots;
    return ff;
}

// RED without the "memory" clobber: the compiler may move the tile loads of the next
// iteration across it (they never alias the histogram); __syncthreads() orders the
// histogram against its final read.
// (a & b) | c in one LOP3 (ALU pipe)
__device__ __forceinline__ unsigned lop3_and_or(unsigned a, unsigned b, unsigned c)
{
    unsigned d;
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

__device__ __forceinline__ void red_shared_hot(unsigned smem_addr, unsigned v)
{
    asm volatile("red.shared.add.u32 [%0], %1;" :: "r"(smem_addr), "r"(v));
}
// ---- parameters of the all-pairs kernels (rdf.cu, rdf_filter.cu) -------------------

struct PairParams {
    const float4 *p1, *p2;
    int64_t pad1, pad2;            // float4 per frame
    int n1, n2;
    const FrameBox *boxes;
    const double *thr;             // T[0..n_bins]
    int n_bins;
    BinGuess guess;
    int same;
    int n_jchunks, jtiles_per_chunk, n_jtiles;
    unsigned long long *counts;
    // fp32 filter (rdf_filter.cu); filt == nullptr: the exact kernel does every frame
    const FrameFilter *filt;
    FilterConst fc;
    int fast_bins;                 // slot_fast certified (used by the exact re-evaluation)
    unsigned long long *fstats;    // [0] deferred entries, [1] inline fixes, [2] audit
                                   // violations, [3] audited uncertain pairs, [4] frames
                                   // declined by the filter, [5] / [6] frames the all-pairs
                                   // filter evaluated in the half-box / rint form,
                                   // [7] half-box frames it evaluated unclamped
                                   // (counted by rdf_filter_prepare_kernel), [8] pairs it
                                   // evaluated in x-clean tile pairs
    // x form of every tile pair of the x-sorted groups (rdf_cleanx_forms_kernel),
    // [F][pad1 / tile][n_jtiles]; nullptr: the groups are not sorted, every pair is dirty
    const unsigned char *xform;
};

}  // namespace rdfdev

rdfdev::BinGuess rdf_bin_guess(const RdfState &R);   // rdf.cu
rdfdev::FilterPrep rdf_filter_prep(const RdfState &R, double sqrt_err);   // rdf_filter.cu
