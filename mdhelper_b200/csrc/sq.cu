// sq.cu -- direct-sum structure factor kernels (seam #2).
//
// Replaces, per frame, the reference's
//     rho[i] = sum_j exp(i q_i . r_j)
// (delta_fourier_transform_sum_2d_2d and its prange twin,
// /root/reference/src/mdhelper/algorithm/accelerated.py:81-165) and the
// accumulation that follows it in StructureFactor._single_frame
// (/root/reference/src/mdhelper/analysis/structure.py:1481-1508):
//     ssf[p] += |rho_j|^2              (j == k, or all particles when mode=None)
//     ssf[p] += 2 Re(rho_j conj(rho_k))  (j != k)
// Normalisation, unique-|q| grouping and sorting stay on the host (numpy).
//
// Kernels
//   sq_lattice_mma_kernel    wavevectors on the reciprocal lattice, q = n * b (the
//       reference's default grid, structure.py:1376-1416).  exp(i q.r) factorises into
//       per-axis phase factors E_a(n) = exp(i n b_a r_a), which turns the sum into the
//       complex rank-N update rho[(nx, ny)][nz] = sum_j (E_x E_y)[j] E_z[j]: warp-
//       specialised, producer warps build the E_a tables (fp64 sincospi + recurrence) into
//       an mbarrier-guarded shared-memory ring, consumer warps run the update on the FP64
//       matrix unit (mma.m8n8k4.f64, 3-multiplication complex product).  Default for all
//       but small wavevector sets (~1e-13 relative to the reference).
//   sq_lattice_kernel<T>     the same factorisation with scalar FMAs: each thread owns two
//       (nx, ny) columns x 8 consecutive nz in registers,
//           A = E_x(nx) E_y(ny);   acc[r] += A * E_z(nz0 + r)     (4 FMA per term)
//       T = double: small wavevector sets;  T = float: approximate mode on the FP32 pipe.
//   sq_general_kernel        arbitrary wavevectors: fp64 dot product + fp64 sincos.
//   sq_finalize_kernel       ssf += per-frame |rho|^2 / cross terms.

#include <cuda_pipeline.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <map>

#include "common.cuh"

namespace {

constexpr int kSqThreads = 256;
#ifndef MDH_SQ_KPS
#define MDH_SQ_KPS 32
#endif
constexpr int kPS = MDH_SQ_KPS;    // particles per shared-memory sub-chunk
constexpr int kSqProducers = 64;   // table-building threads at the end of every block

template <typename T> struct C2;
template <> struct C2<double> { using type = double2; };
template <> struct C2<float> { using type = float2; };

struct LatticeParams {
    const float *raw;              // [F][stride]
    int64_t stride;
    // optional: virtual frame z -> {frame index of r, frame index of r0 or -1, ., .}:
    // the sums run over the displacements r - r0 (intermediate scattering function,
    // structure.py:1991-1996); nullptr: frame z, no reference frame
    const int4 *vmap;
    const int4 *chunks;            // {start, end, rho_row, 0}
    const SqWorkItem *items;
    const int *qidx;               // [n_items][kSqTM][kSqTN]
    double *rho;                   // [F][n_rho][n_q][2]
    int n_rho, n_q;
    // single-chain mode (SingleChainStructureFactor): every chunk is one chain and
    // |rho_chain(q)|^2 is added to chain_out[q]; a block walks the chunks
    // blockIdx.y, blockIdx.y + gridDim.y, ...
    double *chain_out;             // nullptr: normal mode
    int n_chunks;
    double b[3];
    int nmax[3];                   // largest n per axis
    int offy, offz, nt;            // table layout per particle (in table elements)
};

// One sub-chunk of particles into the register accumulators.  The per-thread
// tile is kSqTM columns x R z-terms (R warp-uniform, 1..8), i.e. per particle
// 2*kSqTM complex loads of E_x / E_y and R of E_z feed 4*kSqTM*(R + 1) FP64 FMAs.
//
// Table row of one particle (elements of T): E_x real parts, E_x imaginary parts,
// E_y real, E_y imaginary -- split because every lane reads a different n: 8-byte
// loads of 17 distinct entries are bank-conflict free per half-warp, whereas 16-byte
// (re, im) entries put n and n + 8 in the same banks and cost ~3x the wavefronts --
// then E_z as interleaved (re, im) pairs, which are warp-uniform (one broadcast
// LDS.128 each).
template <typename T, int R>
__device__ __forceinline__ void sq_accumulate_subchunk(const T *tab, int nt,
                                                       const int (&ixr)[kSqTM],
                                                       const int (&ixi)[kSqTM],
                                                       const int (&iyr)[kSqTM],
                                                       const int (&iyi)[kSqTM], int iz,
                                                       T (&acc_re)[kSqTM][kSqTN],
                                                       T (&acc_im)[kSqTM][kSqTN])
{
    using T2 = typename C2<T>::type;
#pragma unroll 1
    for (int p = 0; p < kPS; ++p) {
        const T *row = tab + p * nt;
        T ar[kSqTM], ai[kSqTM];
#pragma unroll
        for (int m = 0; m < kSqTM; ++m) {
            const T exr = row[ixr[m]], exi = row[ixi[m]];
            const T eyr = row[iyr[m]], eyi = row[iyi[m]];
            ar[m] = exr * eyr - exi * eyi;
            ai[m] = exr * eyi + exi * eyr;
        }
        const T2 *zrow = reinterpret_cast<const T2 *>(row + iz);
#pragma unroll
        for (int r = 0; r < R; ++r) {
            const T2 ez = zrow[r];
#pragma unroll
            for (int m = 0; m < kSqTM; ++m) {
                acc_re[m][r] += ar[m] * ez.x;
                acc_re[m][r] -= ai[m] * ez.y;
                acc_im[m][r] += ar[m] * ez.y;
                acc_im[m][r] += ai[m] * ez.x;
            }
        }
    }
}

// Block = S.block consumer threads (one work item each) followed by kSqProducers
// producer threads.  The producers build the phase-factor tables of sub-chunk s + 1
// in the second table buffer while the consumers accumulate sub-chunk s: one barrier
// per sub-chunk, and nobody waits for the sincos / recurrence chains (the single-buffer
// version spent 2 of 3 stall cycles at its barriers).
template <typename T>
__global__ void __launch_bounds__(kSqThreads, 2) sq_lattice_kernel(const LatticeParams P)
{
    using T2 = typename C2<T>::type;
    extern __shared__ __align__(16) unsigned char smem[];
    const int nt = P.nt;                             // elements of T per particle
    T *sTab = reinterpret_cast<T *>(smem);           // [2][kPS][nt]

    const int tid = threadIdx.x;
    const int n_cons = (int)blockDim.x - kSqProducers;
    const bool producer = tid >= n_cons;
    const int frame = blockIdx.z;
    int4 chunk = P.chunks[blockIdx.y];
    const int4 vm = P.vmap ? P.vmap[frame] : make_int4(frame, -1, 0, 0);
    const float *pos = P.raw + (int64_t)vm.x * P.stride;
    const float *pos0 = vm.y >= 0 ? P.raw + (int64_t)vm.y * P.stride : nullptr;

    // tables of particles [p0, p0 + np): task <-> (particle, axis); one fp64 sincos,
    // then E(n+1) = E(n) E(1); rows past np are zero so that the consumers never test
    auto build = [&](T *tab, int p0) {
        const int np = min(kPS, chunk.y - p0);
        for (int task = tid - n_cons; task < kPS * 3; task += kSqProducers) {
            const int p = task / 3, a = task - 3 * p;
            const int nm = P.nmax[a];
            // real parts at re[n * st], imaginary parts at im[n * st]; npad entries
            T *re, *im;
            int st, npad;
            if (a == 2) {
                re = tab + p * nt + P.offz; im = re + 1; st = 2; npad = (nt - P.offz) / 2;
            } else {
                re = tab + p * nt + (a == 0 ? 0 : P.offy); im = re + nm + 1; st = 1;
                npad = nm + 1;
            }
            double s1 = 0.0, c1 = 0.0, er = 0.0, ei = 0.0;
            if (p < np) {
                double x = (double)pos[3 * (int64_t)(p0 + p) + a];
                // displacement in fp64 of the float32 coordinates: exact, as the
                // reference's float64 position buffer makes it
                if (pos0) x -= (double)pos0[3 * (int64_t)(p0 + p) + a];
                sincos(P.b[a] * x, &s1, &c1);
                er = 1.0;
            }
            for (int n = 0; n < npad; ++n) {
                const bool live = n <= nm;
                re[n * st] = live ? (T)er : T(0);
                im[n * st] = live ? (T)ei : T(0);
                const double nr = er * c1 - ei * s1;
                ei = er * s1 + ei * c1;
                er = nr;
            }
        }
    };

    const int item_index = blockIdx.x * n_cons + min(tid, n_cons - 1);
    const SqWorkItem item = P.items[item_index];
    // warp-uniform number of z-terms
    const int wlen = __reduce_max_sync(0xffffffffu, max(item.len[0], item.len[1]));

    T acc_re[kSqTM][kSqTN], acc_im[kSqTM][kSqTN];
#pragma unroll
    for (int m = 0; m < kSqTM; ++m)
#pragma unroll
        for (int r = 0; r < kSqTN; ++r) acc_re[m][r] = acc_im[m][r] = T(0);

    int ixr[kSqTM], ixi[kSqTM], iyr[kSqTM], iyi[kSqTM];
#pragma unroll
    for (int m = 0; m < kSqTM; ++m) {
        ixr[m] = item.nx[m];
        ixi[m] = P.nmax[0] + 1 + item.nx[m];
        iyr[m] = P.offy + item.ny[m];
        iyi[m] = P.offy + P.nmax[1] + 1 + item.ny[m];
    }
    const int iz = P.offz + 2 * item.nz0;

    const int *qi = P.qidx + (int64_t)item_index * (kSqTM * kSqTN);
    // normal mode: one chunk per block (gridDim.y == n_chunks); chain mode: a stride
    // loop over the chains with the accumulators squared and cleared in between
    for (int ci = blockIdx.y; ci < P.n_chunks; ci += gridDim.y) {
    chunk = P.chunks[ci];
    if (producer) build(sTab, chunk.x);
    __syncthreads();
    int buf = 0;
    for (int p0 = chunk.x; p0 < chunk.y; p0 += kPS) {
        const T *tab = sTab + (size_t)buf * kPS * nt;
        if (producer) {
            if (p0 + kPS < chunk.y) build(sTab + (size_t)(buf ^ 1) * kPS * nt, p0 + kPS);
        } else {
#define MDH_SQ_CASE(R) \
    case R: sq_accumulate_subchunk<T, R>(tab, nt, ixr, ixi, iyr, iyi, iz, acc_re, acc_im); break;
            switch (wlen) {
                MDH_SQ_CASE(1) MDH_SQ_CASE(2) MDH_SQ_CASE(3) MDH_SQ_CASE(4)
                MDH_SQ_CASE(5) MDH_SQ_CASE(6) MDH_SQ_CASE(7) MDH_SQ_CASE(8)
                default: break;
            }
#undef MDH_SQ_CASE
        }
        __syncthreads();
        buf ^= 1;
    }
    if (producer) continue;

    double *out = P.rho + ((int64_t)frame * P.n_rho + chunk.z) * P.n_q * 2;
#pragma unroll
    for (int m = 0; m < kSqTM; ++m)
#pragma unroll
        for (int r = 0; r < kSqTN; ++r) {
            if (r < item.len[m]) {
                const int q = qi[m * kSqTN + r];
                if (q >= 0) {
                    if (P.chain_out) {
                        const double re = (double)acc_re[m][r], im = (double)acc_im[m][r];
                        atomicAdd(P.chain_out + q, re * re + im * im);
                    } else {
                        atomicAdd(out + 2 * q, (double)acc_re[m][r]);
                        atomicAdd(out + 2 * q + 1, (double)acc_im[m][r]);
                    }
                }
            }
            acc_re[m][r] = acc_im[m][r] = T(0);
        }
    }
}

// ---- lattice sum on the FP64 matrix unit (DMMA m8n8k4) ---------------------------------
//
// With A[c][j] = E_x(nx_c)[j] E_y(ny_c)[j] (c = (nx, ny) column, j = particle) and
// B[j][nz] = E_z(nz)[j] the lattice sum is the complex rank-N update
//     rho[c][nz] = sum_j A[c][j] B[j][nz]
// i.e. four real matrix products (re re, im im, re im, im re).  mma.sync.m8n8k4.f64
// (SASS DMMA.8x8x4) sustains the full 64 FMA/clk/SM with two 64-bit register operands
// per 8 FMAs of a thread, where the scalar DFMA of sq_lattice_kernel is limited by
// register-operand bandwidth to 42.6 (tools/microbench3.cu, profiles/microbench3_r01.json).
//
// A warp owns up to kMmaG groups of 8 columns x up to kMmaTZ tiles of 8 consecutive nz.
// Fragment layout of m8n8k4 (lane = 4 g + k): A[g][k], B[k][g], C[g][2k], C[g][2k + 1].
// Per step of 4 particles lane (g, k) loads E_x(nx_g), E_y(ny_g) of particle k (two
// LDS.128), multiplies them (the A element), loads E_z(8 t + g) of particle k per tile
// (one LDS.128 = the B elements re / im) and issues 4 DMMAs per (group, tile).
//
// Issue slots are the scarce resource: on sm_100 a DMMA.8x8x4 occupies its scheduler for
// the 16 cycles it occupies the pipe, and every other instruction of any warp on that
// scheduler adds its own issue cycles on top (tools/microbench3.cu: 2 IMADs per DMMA cost
// 11 %, one LDS.128 + DADD per DMMA 27 %).  The consumer loop therefore carries nothing but
// loads with immediate offsets, the complex product and the DMMAs: the 8 steps of a
// sub-chunk are unrolled, the tile counts are template parameters, and the table layout
// makes every address a per-lane base plus a compile-time constant.
//
// Table of one sub-chunk (32 particles): rows of kRowSlots = 36 double2 (re, im) entries --
// 32 particles + 4 pad --, one row per table entry: E_x(0..nmax_x) | E_y(0..nmax_y) |
// E_z(0..8 * tiles - 1, zero past nmax_z).  A step reads 4 consecutive particles of a row
// (64 bytes); the row stride of 576 bytes puts neighbouring rows 16 banks apart, so the
// 16-byte loads of a quarter-warp (two columns x four particles) are conflict-free whenever
// the two columns' nx (ny) are equal or differ by an odd number -- the host pairs the
// columns that way (E_z rows of a quarter-warp are always neighbours).
#ifndef MDH_SQ_MMA_G
#define MDH_SQ_MMA_G 2
#endif
constexpr int kMmaG = MDH_SQ_MMA_G;     // column groups per warp item (1 or 2)
constexpr int kMmaTZ = 4;
constexpr int kRowSlots = kPS + 4;   // entries per table row
// 3-multiplication complex product (Gauss / "3M"): with P1 = sum A_r B_r, P2 = sum A_i B_i,
// P3 = sum (A_r + A_i)(B_r + B_i):  Re = P1 - P2, Im = P3 - P1 - P2 -- three DMMAs per
// (group, tile) and step instead of four, for one DADD per group and step and a third
// table value B_r + B_i (written by the producers).  Every accumulator is touched once per
// step, so no DMMA depends on a recent one.
#ifndef MDH_SQ_MMA_3M
#define MDH_SQ_MMA_3M 1
#endif
constexpr bool kMma3M = MDH_SQ_MMA_3M != 0;
constexpr int kMmaAcc = kMma3M ? 3 : 2;   // accumulator pairs per (group, tile)
// double2 entries of one table stage: R rows of kRowSlots (re, im) entries, then (3M) nzpad
// rows of kRowSlots doubles B_r + B_i -- 288-byte rows, 8 banks apart, so that the 8-byte
// loads of a half-warp (four neighbouring rows x four particles) are conflict-free
__host__ __device__ inline int mma_stage_entries(int R, int nzpad)
{
    return R * kRowSlots + (kMma3M ? nzpad * kRowSlots / 2 : 0);
}
#ifndef MDH_SQ_MMA_WARPS
#define MDH_SQ_MMA_WARPS 14
#endif
#ifndef MDH_SQ_MMA_PRODUCERS
#define MDH_SQ_MMA_PRODUCERS 64
#endif
constexpr int kMmaMaxWarps = MDH_SQ_MMA_WARPS;   // consumer warps per block

struct SqMmaItem {                 // one warp's work
    int16_t nx[kMmaG][8], ny[kMmaG][8];
    int nt[kMmaG];                 // nz tiles of each group, nt[0] >= nt[1]; 0: unused
    int t0, pad;                   // first tile
};

struct MmaParams {
    const float *raw;
    int64_t stride;
    const int4 *vmap;              // as in LatticeParams
    const int4 *chunks;
    const SqMmaItem *items;
    const int *qidx;               // [n_items][kMmaG][kMmaTZ][8][8]
    double *rho;
    int n_rho, n_q;
    double *chain_out;
    int n_chunks, n_units;         // work units = (frame, chunk), frame-major
    double b[3];
    int nmax[3];
    int offy, offz, nzpad, R;      // table rows: first E_y / E_z row, E_z rows, all rows
};

__device__ __forceinline__ void dmma884(double (&c)[2], double a, double b)
{
    // volatile: keeps the issue order chosen in the loops below
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c[0]), "+d"(c[1]) : "d"(a), "d"(b));
}

// One sub-chunk (kPS particles, 4 per step) into the accumulators.  nt0 / nt1: nz tiles
// of the item's first / second column group (nt0 >= nt1; nt1 = 0: no second group) --
// compile-time.  bx / by / bz: this lane's E_x / E_y / E_z entries of the sub-chunk's first
// step (row * kRowSlots + k); step ks is 4 * ks entries further, tile t 8 rows further.
template <int nt0, int nt1>
__device__ __forceinline__ void sq_mma_subchunk(const double2 *tab, const int (&bx)[kMmaG],
                                                const int (&by)[kMmaG], int bz,
                                                const double *sums, int bs,
                                                double (&acc)[kMmaAcc][kMmaG][nt0][2])
{
    constexpr int NG = nt1 > 0 ? 2 : 1;
#pragma unroll
    for (int ks = 0; ks < kPS / 4; ++ks) {
        double ar[NG], ai[NG], ax[NG];   // ax: A_r + A_i (3M) or -A_i
#pragma unroll
        for (int i = 0; i < NG; ++i) {
            const double2 ex = tab[bx[i] + 4 * ks], ey = tab[by[i] + 4 * ks];
            ar[i] = ex.x * ey.x - ex.y * ey.y;
            ai[i] = ex.x * ey.y + ex.y * ey.x;
            ax[i] = kMma3M ? ar[i] + ai[i]
                           : __hiloint2double(__double2hiint(ai[i]) ^ (int)0x80000000,
                                              __double2loint(ai[i]));
        }
        if (kMma3M) {
#pragma unroll
            for (int t = 0; t < nt0; ++t) {
                const double2 ez = tab[bz + 4 * ks + 8 * kRowSlots * t];
                const double es = sums[bs + 4 * ks + 8 * kRowSlots * t];
#pragma unroll
                for (int i = 0; i < NG; ++i)
                    if (i == 0 || t < nt1) {
                        dmma884(acc[0][i][t], ar[i], ez.x);
                        dmma884(acc[1][i][t], ai[i], ez.y);
                        dmma884(acc[kMmaAcc - 1][i][t], ax[i], es);
                    }
            }
        } else {
            // all E_z tiles first, then two passes over the (group, tile) pairs so that the
            // two DMMAs into the same accumulator are far apart
            double2 ez[nt0];
#pragma unroll
            for (int t = 0; t < nt0; ++t) ez[t] = tab[bz + 4 * ks + 8 * kRowSlots * t];
#pragma unroll
            for (int t = 0; t < nt0; ++t)
#pragma unroll
                for (int i = 0; i < NG; ++i)
                    if (i == 0 || t < nt1) {
                        dmma884(acc[0][i][t], ar[i], ez[t].x);
                        dmma884(acc[1][i][t], ar[i], ez[t].y);
                    }
#pragma unroll
            for (int t = 0; t < nt0; ++t)
#pragma unroll
                for (int i = 0; i < NG; ++i)
                    if (i == 0 || t < nt1) {
                        dmma884(acc[0][i][t], ax[i], ez[t].y);
                        dmma884(acc[1][i][t], ai[i], ez[t].x);
                    }
        }
    }
}

// mbarrier helpers (CTA scope): producers -> consumers "stage full", consumers ->
// producers "stage empty"; arrive has release, try_wait acquire semantics
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;"
                 :: "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}"
                 :: "r"((unsigned)__cvta_generic_to_shared(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity)
{
    asm volatile(
        "{\n\t.reg .pred p;\n"
        "W_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@!p bra W_%=;\n\t}"
        :: "r"((unsigned)__cvta_generic_to_shared(bar)), "r"(parity) : "memory");
}

#ifndef MDH_SQ_MMA_STAGES
#define MDH_SQ_MMA_STAGES 2
#endif
constexpr int kMmaStages = MDH_SQ_MMA_STAGES;      // table buffers in flight
// producer threads; the 4 * kPS tasks of a sub-chunk are (particle, table part) with the
// parts E_x, E_y and the two halves of E_z
constexpr int kMmaProducers = MDH_SQ_MMA_PRODUCERS;
constexpr int kMmaRounds = 4 * kPS / kMmaProducers;
static_assert(kMmaRounds * kMmaProducers == 4 * kPS, "producer threads must divide the tasks");

// Position of producer warp j in a block of W consumer warps: with at least 6 consumers the
// (two) producers sit at warps 3 and 7, i.e. on the same scheduler (warp w runs on
// scheduler w mod 4), which then carries few consumer warps -- the producers' scalar FP64
// chains lose the arbitration against DMMAs, so they should meet as few as possible;
// smaller blocks keep the producers behind the consumers.
__host__ __device__ inline int mma_producer_warp(int W, int j)
{
    return (kMmaProducers == 64 && W >= 6) ? 3 + 4 * j : W + j;
}
// warp index of consumer slot c
__host__ __device__ inline int mma_consumer_warp(int W, int c)
{
    int w = c;
    for (int j = 0; j < kMmaProducers / 32; ++j)
        if (w >= mma_producer_warp(W, j)) ++w;
    return w;
}


// A consumer warp without work (items are padded to whole blocks): waits for every table
// stage and releases it at once.
__device__ __forceinline__ void sq_mma_idle(const MmaParams &P, uint64_t *bar_full,
                                            uint64_t *bar_empty, int lane)
{
    int it = 0;
    for (int u = blockIdx.y; u < P.n_units; u += gridDim.y) {
        const int frame = u / P.n_chunks;
        const int4 chunk = P.chunks[u - frame * P.n_chunks];
        for (int p0 = chunk.x; p0 < chunk.y; p0 += kPS, ++it) {
            const int stage = it % kMmaStages, use = it / kMmaStages;
            mbar_wait(bar_full + stage, use & 1);
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_empty + stage);
        }
    }
}

// The consumer loop of one warp item with NT0 / NT1 nz tiles in its two column groups:
// walks the block's work units, waits for each table stage, runs the sub-chunk update and
// adds the finished unit to rho (or |rho_chain|^2 to the chain accumulator).
template <int NT0, int NT1>
__device__ __forceinline__ void sq_mma_consume(const MmaParams &P, const double2 *sTab, int R,
                                               uint64_t *bar_full, uint64_t *bar_empty,
                                               const int (&bx)[kMmaG], const int (&by)[kMmaG],
                                               int bz, int bs, const int *qi, int g, int k,
                                               int lane)
{
    double acc[kMmaAcc][kMmaG][NT0][2];
#pragma unroll
    for (int c = 0; c < kMmaAcc; ++c)
#pragma unroll
        for (int i = 0; i < kMmaG; ++i)
#pragma unroll
            for (int t = 0; t < NT0; ++t) acc[c][i][t][0] = acc[c][i][t][1] = 0.0;

    int it = 0;
    for (int u = blockIdx.y; u < P.n_units; u += gridDim.y) {
        const int frame = u / P.n_chunks;
        const int4 chunk = P.chunks[u - frame * P.n_chunks];
        for (int p0 = chunk.x; p0 < chunk.y; p0 += kPS, ++it) {
            const int stage = it % kMmaStages, use = it / kMmaStages;
            mbar_wait(bar_full + stage, use & 1);
            const double2 *tab = sTab + (size_t)stage * mma_stage_entries(R, P.nzpad);
            const double *sums = reinterpret_cast<const double *>(tab + R * kRowSlots);
            sq_mma_subchunk<NT0, NT1>(tab, bx, by, bz, sums, bs, acc);
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_empty + stage);
        }

        double *out = P.rho + ((int64_t)frame * P.n_rho + chunk.z) * P.n_q * 2;
#pragma unroll
        for (int i = 0; i < kMmaG; ++i)
#pragma unroll
            for (int t = 0; t < NT0; ++t) {
                if (t < (i == 0 ? NT0 : NT1)) {
                    // this lane holds C[g][2k], C[g][2k + 1]
                    const int2 q2 = *reinterpret_cast<const int2 *>(
                        qi + ((i * kMmaTZ + t) * 8 + g) * 8 + 2 * k);
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        const int q = j ? q2.y : q2.x;
                        if (q < 0) continue;
                        const double p1 = acc[0][i][t][j], p2 = acc[1][i][t][j];
                        const double re = kMma3M ? p1 - p2 : p1;
                        const double im = kMma3M ? acc[kMmaAcc - 1][i][t][j] - p1 - p2 : p2;
                        if (P.chain_out) {
                            atomicAdd(P.chain_out + q, re * re + im * im);
                        } else {
                            atomicAdd(out + 2 * q, re);
                            atomicAdd(out + 2 * q + 1, im);
                        }
                    }
#pragma unroll
                    for (int c = 0; c < kMmaAcc; ++c) acc[c][i][t][0] = acc[c][i][t][1] = 0.0;
                }
            }
    }
}

// Persistent block = n_cons consumer warps (one SqMmaItem each) and kMmaProducers producer
// threads (warp roles: mma_producer_warp).  The block walks the work units (frame, particle chunk) blockIdx.y,
// blockIdx.y + gridDim.y, ...; the producers build the phase-factor tables of the
// sub-chunks (32 particles) into a ring of kMmaStages buffers, running ahead of the
// consumers across unit boundaries; "full" / "empty" mbarriers per stage -- a consumer
// warp waits only for the producers, never for the other consumer warps.
__global__ void __launch_bounds__(kMmaMaxWarps * 32 + kMmaProducers, 1)
    sq_lattice_mma_kernel(const MmaParams P)
{
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ uint64_t bar_full[kMmaStages], bar_empty[kMmaStages];
    double2 *sTab = reinterpret_cast<double2 *>(smem);      // [kMmaStages][R][kRowSlots]
    const int R = P.R;
    const int tid = threadIdx.x, lane = tid & 31;
    const int n_cons = (int)blockDim.x - kMmaProducers;
    // warp roles: the producer warps sit at the positions mma_producer_warp() says (on ONE
    // scheduler when the block is large enough), the consumers fill the rest in order
    const int warp = tid >> 5;
    int prod_index = -1, cons_index = warp;
#pragma unroll
    for (int j = 0; j < kMmaProducers / 32; ++j) {
        const int pw = mma_producer_warp(n_cons >> 5, j);
        if (warp == pw) prod_index = j;
        if (warp > pw) --cons_index;
    }
    const bool producer = prod_index >= 0;
    const int ptid = prod_index * 32 + lane;       // thread index among the producers
    if (tid == 0)
        for (int s = 0; s < kMmaStages; ++s) {
            mbar_init(bar_full + s, kMmaProducers);
            mbar_init(bar_empty + s, n_cons >> 5);
        }
    __syncthreads();

    if (producer) {
        // task r of this thread: particle p of the sub-chunk, part 0 = E_x, 1 = E_y, 2 / 3 =
        // first / second half of E_z (entries n0 .. n0 + cnt - 1 of the axis, zero past nmax);
        // the lanes of a warp write the same entry of 32 consecutive particles (one row).
        // Four interleaved recurrences E(n) = E(n - 4) E(4) keep the dependent chains short:
        // every scalar FP64 instruction queues behind the consumers' DMMAs.  A partial last
        // sub-chunk gets zero columns, so the consumers never test.
        const int zhalf = (P.nzpad / 2 + 3) / 4 * 4;
        // coordinate for task r of the sub-chunk at p0 of unit u; fetched one sub-chunk
        // ahead so that the global-memory latency is off the critical path
        // (raw floats: converted only when used, or the conversion would wait for the load
        // right here; second value: the reference frame of a displacement, else 0; NaN: a
        // particle past the end of the chunk)
        auto fetch = [&](int r, int u, int p0) -> float2 {
            const int task = ptid + r * kMmaProducers;
            const int part = task / kPS, p = task - part * kPS, a = min(part, 2);
            if (u >= P.n_units) return make_float2(0.f, 0.f);
            const int frame = u / P.n_chunks;
            const int4 ch = P.chunks[u - frame * P.n_chunks];
            if (p0 + p >= ch.y) return make_float2(nanf(""), 0.f);
            const int4 vm = P.vmap ? P.vmap[frame] : make_int4(frame, -1, 0, 0);
            const int64_t idx = 3 * (int64_t)(p0 + p) + a;
            float2 v = make_float2(P.raw[(int64_t)vm.x * P.stride + idx], 0.f);
            if (vm.y >= 0) v.y = P.raw[(int64_t)vm.y * P.stride + idx];
            return v;
        };
        int it = 0;
        int u = blockIdx.y;
        int4 chunk = u < P.n_units ? P.chunks[u % P.n_chunks] : make_int4(0, 0, 0, 0);
        int p0 = chunk.x;
        float2 x[kMmaRounds], xn[kMmaRounds];
#pragma unroll
        for (int r = 0; r < kMmaRounds; ++r) x[r] = fetch(r, u, p0);
        while (u < P.n_units) {
            // next (unit, sub-chunk)
            int un = u, pn = p0 + kPS;
            int4 chn = chunk;
            if (pn >= chunk.y) {
                un = u + gridDim.y;
                if (un < P.n_units) chn = P.chunks[un % P.n_chunks];
                pn = chn.x;
            }
#pragma unroll
            for (int r = 0; r < kMmaRounds; ++r) xn[r] = fetch(r, un, pn);

            const int stage = it % kMmaStages, use = it / kMmaStages;
            if (use > 0) mbar_wait(bar_empty + stage, (use - 1) & 1);
#pragma unroll
            for (int r = 0; r < kMmaRounds; ++r) {
                const int task = ptid + r * kMmaProducers;
                const int part = task / kPS, p = task - part * kPS, a = min(part, 2);
                const int nm = P.nmax[a];
                const int n0 = part == 3 ? zhalf : 0;
                const int cnt = part < 2 ? nm + 1 : part == 2 ? zhalf : P.nzpad - zhalf;
                double er[4], ei[4], c4 = 0.0, s4 = 0.0;
#pragma unroll
                for (int j = 0; j < 4; ++j) er[j] = ei[j] = 0.0;
                if (x[r].x == x[r].x) {           // NaN: past the end of the chunk -> zero row
                    // displacement in fp64 of the float32 coordinates: exact, as the
                    // reference's float64 position buffer makes it
                    // phase = pi * (b / pi) * x: sincospi needs no Cody-Waite reduction
                    const double th = (P.b[a] * 0.31830988618379067154) *
                                      ((double)x[r].x - (double)x[r].y);
                    double s1, c1;
                    sincospi(th, &s1, &c1);
                    const double c2 = c1 * c1 - s1 * s1, s2 = 2.0 * (c1 * s1);
                    c4 = c2 * c2 - s2 * s2; s4 = 2.0 * (c2 * s2);
                    er[0] = 1.0;
                    // second half of E_z: start at E(n0) = E(4)^(n0 / 4) (n0 is a multiple of 4)
                    for (int m = 0; m < n0; m += 4) {
                        const double nr = er[0] * c4 - ei[0] * s4;
                        ei[0] = er[0] * s4 + ei[0] * c4;
                        er[0] = nr;
                    }
                    er[1] = er[0] * c1 - ei[0] * s1; ei[1] = er[0] * s1 + ei[0] * c1;
                    er[2] = er[0] * c2 - ei[0] * s2; ei[2] = er[0] * s2 + ei[0] * c2;
                    er[3] = er[1] * c2 - ei[1] * s2; ei[3] = er[1] * s2 + ei[1] * c2;
                }
                // entry n of this part: row (offset + n0 + n), slot p
                double2 *stab = sTab + (size_t)stage * mma_stage_entries(R, P.nzpad);
                double2 *e = stab + ((a == 0 ? 0 : a == 1 ? P.offy : P.offz) + n0) * kRowSlots + p;
                // B_r + B_i of E_z entry n0 + n: row n0 + n of the doubles behind the table
                double *es = reinterpret_cast<double *>(stab + R * kRowSlots) + n0 * kRowSlots + p;
                for (int n = 0; n < cnt; n += 4) {
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        if (n + j < cnt) {
                            const bool live = n0 + n + j <= nm;
                            e[(n + j) * kRowSlots] = live ? make_double2(er[j], ei[j])
                                                          : make_double2(0.0, 0.0);
                            if (kMma3M && a == 2)
                                es[(n + j) * kRowSlots] = live ? er[j] + ei[j] : 0.0;
                        }
                        const double nr = er[j] * c4 - ei[j] * s4;
                        ei[j] = er[j] * s4 + ei[j] * c4;
                        er[j] = nr;
                    }
                }
            }
            mbar_arrive(bar_full + stage);
            ++it;
            u = un; p0 = pn; chunk = chn;
#pragma unroll
            for (int r = 0; r < kMmaRounds; ++r) x[r] = xn[r];
        }
        return;
    }

    const int item_index = blockIdx.x * (n_cons >> 5) + cons_index;
    const SqMmaItem *item = P.items + item_index;
    const int nt0 = item->nt[0], nt1 = kMmaG > 1 ? item->nt[kMmaG - 1] : 0;
    const int g = lane >> 2, k = lane & 3;
    int bx[kMmaG], by[kMmaG];
#pragma unroll
    for (int i = 0; i < kMmaG; ++i) {
        bx[i] = item->nx[i][g] * kRowSlots + k;
        by[i] = (P.offy + item->ny[i][g]) * kRowSlots + k;
    }
    const int bz = (P.offz + 8 * item->t0 + g) * kRowSlots + k;
    // this lane's B_r + B_i entry (doubles, behind the R double2 rows of the stage)
    const int bs = (8 * item->t0 + g) * kRowSlots + k;

    const int *qi = P.qidx + (int64_t)item_index * (kMmaG * kMmaTZ * 64);
    // the whole consumer loop is instantiated per (tiles of group 0, tiles of group 1): the
    // accumulators of an item then are exactly the registers it needs (a runtime tile count
    // kept all 3 x 2 x 4 pairs -- 96 registers -- alive and spilled in the hot loop)
#define MDH_MMA_CASE(A, B)                                                                   \
    case A * 8 + B:                                                                          \
        sq_mma_consume<A, B>(P, sTab, R, bar_full, bar_empty, bx, by, bz, bs, qi, g, k, lane); \
        break;
    switch (nt0 * 8 + nt1) {
        MDH_MMA_CASE(1, 0) MDH_MMA_CASE(2, 0) MDH_MMA_CASE(3, 0) MDH_MMA_CASE(4, 0)
#if MDH_SQ_MMA_G > 1
        MDH_MMA_CASE(1, 1) MDH_MMA_CASE(2, 1) MDH_MMA_CASE(2, 2) MDH_MMA_CASE(3, 1)
        MDH_MMA_CASE(3, 2) MDH_MMA_CASE(3, 3) MDH_MMA_CASE(4, 1) MDH_MMA_CASE(4, 2)
        MDH_MMA_CASE(4, 3) MDH_MMA_CASE(4, 4)
#endif
        default:
            // a padding item (no tiles): the warp still takes part in the stage hand-over,
            // or the producers would wait for its "empty" arrival forever
            sq_mma_idle(P, bar_full, bar_empty, lane);
            break;
    }
#undef MDH_MMA_CASE
}

struct GeneralParams {
    const float *raw;
    int64_t stride;
    const int4 *vmap;              // as in LatticeParams
    const int4 *chunks;
    const double *qv;              // [n_q][3]
    double *rho;
    int n_rho, n_q;
};

__global__ void __launch_bounds__(128) sq_general_kernel(const GeneralParams P)
{
    __shared__ double sx[256], sy[256], sz[256];
    const int tid = threadIdx.x;
    const int frame = blockIdx.z;
    const int4 chunk = P.chunks[blockIdx.y];
    const int q = blockIdx.x * 128 + tid;
    const bool qvalid = q < P.n_q;
    const double qx = qvalid ? P.qv[3 * q] : 0.0;
    const double qy = qvalid ? P.qv[3 * q + 1] : 0.0;
    const double qz = qvalid ? P.qv[3 * q + 2] : 0.0;
    const int4 vm = P.vmap ? P.vmap[frame] : make_int4(frame, -1, 0, 0);
    const float *pos = P.raw + (int64_t)vm.x * P.stride;
    const float *pos0 = vm.y >= 0 ? P.raw + (int64_t)vm.y * P.stride : nullptr;
    double re = 0.0, im = 0.0;
    for (int p0 = chunk.x; p0 < chunk.y; p0 += 256) {
        const int np = min(256, chunk.y - p0);
        for (int p = tid; p < np; p += 128) {
            sx[p] = (double)pos[3 * (int64_t)(p0 + p)];
            sy[p] = (double)pos[3 * (int64_t)(p0 + p) + 1];
            sz[p] = (double)pos[3 * (int64_t)(p0 + p) + 2];
            if (pos0) {
                sx[p] -= (double)pos0[3 * (int64_t)(p0 + p)];
                sy[p] -= (double)pos0[3 * (int64_t)(p0 + p) + 1];
                sz[p] -= (double)pos0[3 * (int64_t)(p0 + p) + 2];
            }
        }
        __syncthreads();
        if (qvalid) {
            for (int p = 0; p < np; ++p) {
                double s, c;
                sincos(qx * sx[p] + qy * sy[p] + qz * sz[p], &s, &c);
                re += c;
                im += s;
            }
        }
        __syncthreads();
    }
    if (qvalid) {
        double *out = P.rho + ((int64_t)frame * P.n_rho + chunk.z) * P.n_q * 2;
        atomicAdd(out + 2 * q, re);
        atomicAdd(out + 2 * q + 1, im);
    }
}

__global__ void sq_finalize_kernel(const double2 *__restrict__ rho, int n_frames, int n_rho,
                                   int n_q, const int *__restrict__ pairs, int n_pairs,
                                   double *__restrict__ ssf)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    const int p = blockIdx.y;
    if (q >= n_q) return;
    int j = pairs[2 * p], k = pairs[2 * p + 1];
    if (j < 0) j = k = 0;
    double acc = 0.0;
    for (int f = 0; f < n_frames; ++f) {
        const double2 rj = rho[((int64_t)f * n_rho + j) * n_q + q];
        if (j == k) {
            acc += rj.x * rj.x + rj.y * rj.y;
        } else {
            const double2 rk = rho[((int64_t)f * n_rho + k) * n_q + q];
            acc += 2.0 * (rj.x * rk.x + rj.y * rk.y);
        }
    }
    ssf[(int64_t)p * n_q + q] += acc;
}

// Row layout of the scalar lattice kernel's tables, in elements per particle:
// E_x re | E_x im | E_y re | E_y im | E_z (re, im) pairs padded to whole kSqTN tiles.
static int lattice_row_elems(const int (&nmax)[3], int *offy, int *offz)
{
    const int oy = 2 * (nmax[0] + 1);
    const int oz = (oy + 2 * (nmax[1] + 1) + 3) / 4 * 4;     // 16-byte aligned
    if (offy) *offy = oy;
    if (offz) *offz = oz;
    return oz + 2 * ((nmax[2] + kSqTN) / kSqTN * kSqTN);
}
constexpr size_t kSqMaxSmem = 227 * 1024;

template <typename T>
int launch_lattice(mdh_ctx *c, const LatticeParams &P, dim3 grid, int block)
{
    using T2 = typename C2<T>::type;
    const size_t smem = 2 * sizeof(T) * kPS * P.nt;           // double-buffered tables
    auto kern = sq_lattice_kernel<T>;
    MDH_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)smem));
    kern<<<grid, block + kSqProducers, smem, c->stream>>>(P);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    return MDH_OK;
}


// ---- host side: work items of the DMMA kernel ---------------------------------------

struct Column { int nx, ny; std::vector<int> q; };   // q[nz] = wavevector index or -1

static int column_top(const Column &c)                // 1 + largest nz present
{
    int t = 0;
    for (int z = 0; z < (int)c.q.size(); ++z) if (c.q[z] >= 0) t = z + 1;
    return t;
}

// table layout of sq_lattice_mma_kernel (double2 entries per particle)
static void mma_layout(const int (&nmax)[3], int *offy, int *offz, int *nzpad, int *R)
{
    *offy = nmax[0] + 1;
    *offz = *offy + nmax[1] + 1;
    *nzpad = (nmax[2] + 8) / 8 * 8;
    *R = *offz + *nzpad;                  // double2 rows of a sub-chunk table
}
static size_t mma_smem_bytes(const int (&nmax)[3])
{
    int offy, offz, nzpad, R;
    mma_layout(nmax, &offy, &offz, &nzpad, &R);
    return (size_t)kMmaStages * mma_stage_entries(R, nzpad) * sizeof(double2);
}
constexpr size_t kMmaSmemLimit = 200 * 1024;
constexpr int kMmaAutoTiles = 16;

// wavevector list -> columns (nx, ny) with their nz entries; false if the indices are not
// usable by the lattice kernels (negative, > 1023 or duplicated)
static bool build_columns(int n_q, const int32_t *lat_n, int (&nm)[3], std::vector<Column> &cols)
{
    nm[0] = nm[1] = nm[2] = 0;
    for (int i = 0; i < n_q; ++i)
        for (int k = 0; k < 3; ++k) {
            const int n = lat_n[3 * i + k];
            if (n < 0 || n > 1023) return false;
            nm[k] = std::max(nm[k], n);
        }
    std::map<std::pair<int, int>, int> where;
    for (int i = 0; i < n_q; ++i) {
        const std::pair<int, int> key{lat_n[3 * i], lat_n[3 * i + 1]};
        auto it = where.find(key);
        if (it == where.end()) {
            it = where.emplace(key, (int)cols.size()).first;
            cols.push_back(Column{key.first, key.second, std::vector<int>(nm[2] + 1, -1)});
        }
        int &slot = cols[it->second].q[lat_n[3 * i + 2]];
        if (slot >= 0) return false;                          // duplicate wavevector
        slot = i;
    }
    return true;
}

// Columns are paired so that the two columns a
// quarter-warp loads together have nx (and ny) equal or an odd distance apart (see the
// bank analysis at the kernel), four pairs make a group of 8, kMmaG consecutive groups x
// <= kMmaTZ nz tiles make a warp item; items are dealt to blocks and, inside a block, to
// the four warp schedulers (warp w runs on scheduler w % 4) by decreasing cost so that
// every scheduler's FP64 unit gets the same number of DMMAs between two barriers.
static void mma_build_items(std::vector<Column> cols, const int (&nm)[3],
                            std::vector<SqMmaItem> &out_items, std::vector<int> &out_qidx,
                            int &warps_per_block, int (&stats)[4])
{
    // by decreasing number of nz tiles, then row by row: neighbours (nx, ny), (nx + 1, ny)
    // are compatible, and a group of 8 never mixes tile counts except at one boundary
    std::sort(cols.begin(), cols.end(), [](const Column &a, const Column &b) {
        const int ta = (column_top(a) + 7) / 8, tb = (column_top(b) + 7) / 8;
        if (ta != tb) return ta > tb;
        if (a.ny != b.ny) return a.ny < b.ny;
        return a.nx < b.nx;
    });
    const int n = (int)cols.size();
    auto compatible = [&](int a, int b) {
        const int dx = std::abs(cols[a].nx - cols[b].nx), dy = std::abs(cols[a].ny - cols[b].ny);
        return (dx == 0 || (dx & 1)) && (dy == 0 || (dy & 1));
    };
    std::vector<int> slot;                            // column index or -1 (dummy), pairs
    std::vector<char> used(n, 0);
    for (int a = 0; a < n; ++a) {
        if (used[a]) continue;
        used[a] = 1;
        int partner = -1;
        for (int b = a + 1; b < n && b < a + 96; ++b)
            if (!used[b] && compatible(a, b)) { partner = b; break; }
        if (partner >= 0) used[partner] = 1;
        slot.push_back(a);
        slot.push_back(partner);
    }
    while (slot.size() % 8) slot.push_back(-1);
    const int n_groups = (int)slot.size() / 8;
    auto group_tiles = [&](int gi) {
        int t = 0;
        for (int m = 0; m < 8; ++m)
            if (slot[gi * 8 + m] >= 0) t = std::max(t, (column_top(cols[slot[gi * 8 + m]]) + 7) / 8);
        return t;
    };
    // groups are sorted by decreasing tile count; kMmaG consecutive groups x one segment
    // of <= kMmaTZ tiles make an item (the second group may need fewer tiles)
    // pieces = (group, segment of <= kMmaTZ tiles); an item pairs two pieces of the same
    // segment, the largest with the smallest, so that all warps carry about the same number
    // of tiles: the block advances at the pace of its slowest warp (a warp releases a table
    // stage only when it is done with it), and one warp alone cannot keep the DMMA pipe busy
    // cost() in 1/8 of the scheduler time of one (group, tile) pair per sub-chunk (8 steps x
    // 3 or 4 DMMAs x 16 cycles): the complex products of a group cost about 5/8 (3/8 with 4
    // DMMAs per pair) of that -- scalar FP64 instructions share the DMMA pipe at ~5 cycles
    // each -- and a producer warp is charged 80/8 (60/8): measured optimum (cfg4: 21.7k
    // frames/s at 40/8, 22.6k at 60/8, 23.0k at 80/8, 22.9k at 100/8); its FP64 chains lose
    // the arbitration against the DMMAs of its scheduler, so the consumers there must be few
    struct Proto {
        int ga, gb, t0, nt[2];
        int tiles() const { return nt[0] + nt[1]; }
        int cost() const { return 8 * tiles() + (kMma3M ? 5 : 3) * ((nt[0] > 0) + (nt[1] > 0)); }
    };
#ifndef MDH_SQ_MMA_PCOST
#define MDH_SQ_MMA_PCOST (kMma3M ? 160 : 120)
#endif
    constexpr int kProducerCost = MDH_SQ_MMA_PCOST * 32 / kMmaProducers;   // per producer warp
    static_assert(kMmaG == 1 || kMmaG == 2, "items are built for one or two groups");
    std::vector<Proto> protos;
    int max_tiles = 0;
    for (int gi = 0; gi < n_groups; ++gi) max_tiles = std::max(max_tiles, group_tiles(gi));
    for (int t0 = 0; t0 < max_tiles; t0 += kMmaTZ) {
        std::vector<std::pair<int, int>> pieces;         // (tiles, group)
        for (int gi = 0; gi < n_groups; ++gi) {
            const int nt = std::min(kMmaTZ, group_tiles(gi) - t0);
            if (nt > 0) pieces.push_back({nt, gi});
        }
        std::sort(pieces.begin(), pieces.end(), [](const std::pair<int, int> &x,
                                                   const std::pair<int, int> &y) {
            return x.first != y.first ? x.first > y.first : x.second < y.second;
        });
        size_t lo = 0, hi = pieces.size();
        if (kMmaG == 1 || (hi - lo) % 2) {               // odd: the largest piece stays alone
            const size_t solo = kMmaG == 1 ? hi : 1;
            for (; lo < solo; ++lo)
                protos.push_back(Proto{pieces[lo].second, -1, t0, {pieces[lo].first, 0}});
        }
        for (; lo + 1 < hi; ++lo, --hi)
            protos.push_back(Proto{pieces[lo].second, pieces[hi - 1].second, t0,
                                   {pieces[lo].first, pieces[hi - 1].first}});
    }
    std::stable_sort(protos.begin(), protos.end(),
                     [](const Proto &a, const Proto &b) { return a.cost() > b.cost(); });
    const int n_items = (int)protos.size();
    const int n_blocks = (n_items + kMmaMaxWarps - 1) / kMmaMaxWarps;
    const int W = (n_items + n_blocks - 1) / n_blocks;
    warps_per_block = W;
    // bins = (block, scheduler); capacity = warps of the block on that scheduler
    std::vector<int> load(n_blocks * 4, 0), fill(n_blocks * 4, 0);
    std::vector<int> place(n_blocks * W, -1);         // slot -> proto
    for (int b = 0; b < n_blocks; ++b)                // the producer warps follow the consumers
        for (int j = 0; j < kMmaProducers / 32; ++j)
            load[b * 4 + (mma_producer_warp(W, j) & 3)] += kProducerCost;
    // consumer slots of a block by scheduler
    std::vector<int> slots_of[4];
    for (int c = 0; c < W; ++c) slots_of[mma_consumer_warp(W, c) & 3].push_back(c);
    auto sched_of = [&](int c) { return mma_consumer_warp(W, c) & 3; };
    for (int p = 0; p < n_items; ++p) {
        int best = -1;
        for (int bin = 0; bin < n_blocks * 4; ++bin) {
            if (fill[bin] >= (int)slots_of[bin & 3].size()) continue;
            if (best < 0 || load[bin] < load[best]) best = bin;
        }
        place[(best >> 2) * W + slots_of[best & 3][fill[best]]] = p;
        fill[best]++;
        load[best] += protos[p].cost();
    }
    // local search: swap items between schedulers of a block while that lowers the larger
    // of the two loads (LPT with unequal capacities leaves easy gains)
    for (bool improved = true; improved;) {
        improved = false;
        for (int b = 0; b < n_blocks && !improved; ++b)
            for (int s1 = 0; s1 < W && !improved; ++s1)
                for (int s2 = 0; s2 < W && !improved; ++s2) {
                    const int b1 = b * 4 + sched_of(s1), b2 = b * 4 + sched_of(s2);
                    if (b1 == b2 || load[b1] <= load[b2]) continue;
                    const int p1 = place[b * W + s1], p2 = place[b * W + s2];
                    const int c1 = p1 < 0 ? 0 : protos[p1].cost(), c2 = p2 < 0 ? 0 : protos[p2].cost();
                    if (c1 > c2 && std::max(load[b1] - c1 + c2, load[b2] - c2 + c1) < load[b1]) {
                        std::swap(place[b * W + s1], place[b * W + s2]);
                        load[b1] += c2 - c1; load[b2] += c1 - c2;
                        improved = true;
                    }
                }
    }
    // {items, (group, tile) pairs = 64 accumulator slots each, largest scheduler load,
    //  schedulers}
    stats[0] = n_items; stats[1] = 0; stats[2] = 0; stats[3] = n_blocks * 4;
    for (const Proto &pr : protos) stats[1] += pr.tiles();
    for (int l : load) stats[2] = std::max(stats[2], (l + 7) / 8);
    if (getenv("MDH_SQ_DEBUG")) {
        fprintf(stderr, "mdh sq dmma: %d columns, %d groups, %d items in %d block(s) of %d warps, "
                "%d tiles; scheduler loads (1/8 tile, producers included):", n, n_groups, n_items,
                n_blocks, W, stats[1]);
        for (int l : load) fprintf(stderr, " %d", l);
        fprintf(stderr, "\n");
    }
    out_items.assign((size_t)n_blocks * W, SqMmaItem{});
    out_qidx.assign((size_t)n_blocks * W * kMmaG * kMmaTZ * 64, -1);
    for (int s = 0; s < n_blocks * W; ++s) {
        if (place[s] < 0) continue;
        const Proto &pr = protos[place[s]];
        SqMmaItem &it = out_items[s];
        it.t0 = pr.t0;
        for (int i = 0; i < kMmaG; ++i) {
            it.nt[i] = pr.nt[i];
            const int gi = i == 0 ? pr.ga : pr.gb;
            for (int m = 0; m < 8; ++m) {
                if (pr.nt[i] == 0) { it.nx[i][m] = it.ny[i][m] = 0; continue; }
                int ci = slot[gi * 8 + m];
                const bool dummy = ci < 0;
                if (dummy) ci = slot[gi * 8 + (m ^ 1)];             // partner's entries
                if (ci < 0) ci = 0;                                  // an all-dummy pair
                it.nx[i][m] = (int16_t)cols[ci].nx;
                it.ny[i][m] = (int16_t)cols[ci].ny;
                if (dummy) continue;
                for (int t = 0; t < pr.nt[i]; ++t)
                    for (int z = 0; z < 8; ++z) {
                        const int nz = 8 * (pr.t0 + t) + z;
                        if (nz < (int)cols[ci].q.size())
                            out_qidx[(((size_t)s * kMmaG + i) * kMmaTZ + t) * 64 + m * 8 + z] =
                                cols[ci].q[nz];
                    }
            }
        }
    }
    (void)nm;
}

// Work items of sq_lattice_kernel: columns sorted by their number of wavevectors (cols is
// reordered); thread tiles take two neighbouring columns (similar lengths) and one segment
// of kSqTN nz values.  Items are padded to whole blocks of `block` consumer threads.
static void lattice_build_items(std::vector<Column> &cols, const int (&nm)[3],
                                std::vector<SqWorkItem> &items, std::vector<int> &qidx,
                                int &block)
{
    std::stable_sort(cols.begin(), cols.end(), [](const Column &a, const Column &b) {
        return column_top(a) > column_top(b);
    });
    const int n_seg = (nm[2] + kSqTN) / kSqTN;
    for (int s = 0; s < n_seg; ++s)
        for (size_t c0 = 0; c0 < cols.size(); c0 += kSqTM) {
            SqWorkItem it{};
            it.nz0 = s * kSqTN;
            std::vector<int> qi(kSqTM * kSqTN, -1);
            bool any = false;
            for (int m = 0; m < kSqTM; ++m) {
                if (c0 + m >= cols.size()) continue;
                const Column &c = cols[c0 + m];
                it.nx[m] = c.nx; it.ny[m] = c.ny;
                for (int r = 0; r < kSqTN; ++r) {
                    const int z = it.nz0 + r;
                    if (z < (int)c.q.size() && c.q[z] >= 0) {
                        qi[m * kSqTN + r] = c.q[z];
                        it.len[m] = r + 1;
                        any = true;
                    }
                }
            }
            if (!any) continue;
            items.push_back(it);
            qidx.insert(qidx.end(), qi.begin(), qi.end());
        }
    // consumer threads per block: whole warps, at most kSqThreads minus the
    // producer warps; items padded to whole blocks
    const int max_cons = kSqThreads - kSqProducers;
    const int n_warps = (int)((items.size() + 31) / 32);
    const int n_blocks = (n_warps * 32 + max_cons - 1) / max_cons;
    block = ((n_warps + n_blocks - 1) / n_blocks) * 32;
    block = std::max(block, 32);
    while (items.size() % block) {
        items.push_back(SqWorkItem{});
        qidx.insert(qidx.end(), kSqTM * kSqTN, -1);
    }
}

}  // namespace

// Device-free planning of the DMMA kernel's work items (what mdh_sq_configure builds for
// MDH_SQ_LATTICE_DMMA); see mdh_sq_plan in the header.
int sq_plan_impl(int n_q, const int32_t *lat_n, int64_t *stats, int32_t *coverage,
                 int32_t *pair_rule_violations)
{
    MDH_REQUIRE(n_q >= 1 && lat_n && stats, MDH_EINVAL, "sq plan: missing argument");
    int nm[3];
    std::vector<Column> cols;
    MDH_REQUIRE(build_columns(n_q, lat_n, nm, cols), MDH_EINVAL,
                "sq plan: wavevector indices are not usable by the lattice kernels");
    std::vector<SqMmaItem> items;
    std::vector<int> qidx;
    int warps = 0, st[4] = {0, 0, 0, 0};
    mma_build_items(cols, nm, items, qidx, warps, st);
    for (int i = 0; i < 4; ++i) stats[i] = st[i];
    stats[4] = warps;
    stats[5] = (int64_t)mma_smem_bytes(nm);
    if (coverage) {
        for (int i = 0; i < n_q; ++i) coverage[i] = 0;
        for (int q : qidx) if (q >= 0 && q < n_q) coverage[q]++;
    }
    if (pair_rule_violations) {
        // the two columns a quarter-warp loads together (m = 2j, 2j + 1) must have equal or
        // odd-distance nx and ny, or their shared-memory loads conflict
        int bad = 0;
        for (const SqMmaItem &it : items)
            for (int i = 0; i < kMmaG; ++i) {
                if (it.nt[i] == 0) continue;
                for (int m = 0; m < 8; m += 2) {
                    const int dx = std::abs(it.nx[i][m] - it.nx[i][m + 1]);
                    const int dy = std::abs(it.ny[i][m] - it.ny[i][m + 1]);
                    if ((dx != 0 && !(dx & 1)) || (dy != 0 && !(dy & 1))) ++bad;
                }
            }
        *pair_rule_violations = bad;
    }
    return MDH_OK;
}

// Per-warp report of both lattice plans (what mdh_sq_configure builds); see
// mdh_sq_plan_items in the header.
int sq_plan_items_impl(int n_q, const int32_t *lat_n, int32_t *mma, int32_t *lattice_r,
                       int64_t cap, int64_t *counts)
{
    MDH_REQUIRE(n_q >= 1 && lat_n && counts && cap >= 0, MDH_EINVAL,
                "sq plan items: missing argument");
    int nm[3];
    std::vector<Column> cols;
    MDH_REQUIRE(build_columns(n_q, lat_n, nm, cols), MDH_EINVAL,
                "sq plan items: wavevector indices are not usable by the lattice kernels");
    std::vector<SqMmaItem> mitems;
    std::vector<int> mqidx;
    int warps = 0, st[4] = {0, 0, 0, 0};
    mma_build_items(cols, nm, mitems, mqidx, warps, st);
    std::vector<SqWorkItem> items;
    std::vector<int> qidx;
    int block = 0;
    lattice_build_items(cols, nm, items, qidx, block);
    counts[0] = (int64_t)mitems.size();
    counts[1] = (int64_t)(items.size() / 32);
    if (mma)
        for (int64_t s = 0; s < std::min<int64_t>(cap, counts[0]); ++s) {
            const SqMmaItem &it = mitems[s];
            // the kernel dispatches on (nt[0], nt[kMmaG - 1]); no tiles: an idle warp
            mma[4 * s + 0] = it.nt[0];
            mma[4 * s + 1] = kMmaG > 1 ? it.nt[kMmaG - 1] : 0;
            mma[4 * s + 2] = it.t0;
            mma[4 * s + 3] = it.nt[0] == 0;
        }
    if (lattice_r)
        for (int64_t w = 0; w < std::min<int64_t>(cap, counts[1]); ++w) {
            // sq_lattice_kernel's warp-uniform R: the longest column segment of the warp
            int r = 0;
            for (int l = 0; l < 32; ++l)
                for (int m = 0; m < kSqTM; ++m) r = std::max(r, items[32 * w + l].len[m]);
            lattice_r[w] = r;
        }
    return MDH_OK;
}

// ---- host side ------------------------------------------------------------------

int sq_configure_impl(mdh_ctx *c, int64_t n_total, int n_groups, const int64_t *goff,
                      int n_q, const double *wv, const int32_t *lat_n, const double *lat_b,
                      int n_pairs, const int32_t *pairs, int mode)
{
    SqState &S = c->sq;
    MDH_REQUIRE(n_total > 0 && n_total < (1ll << 31) / 3, MDH_EINVAL,
                "sq: n_total must be in [1, 2^31/3)");
    MDH_REQUIRE(n_groups >= 1 && goff != nullptr, MDH_EINVAL, "sq: groups missing");
    MDH_REQUIRE(goff[0] == 0 && goff[n_groups] == n_total, MDH_EINVAL,
                "sq: group_offsets must run from 0 to n_total");
    for (int g = 0; g < n_groups; ++g)
        MDH_REQUIRE(goff[g] < goff[g + 1], MDH_EINVAL, "sq: group %d is empty", g);
    MDH_REQUIRE(n_q >= 1 && wv != nullptr, MDH_EINVAL, "sq: wavevectors missing");
    MDH_REQUIRE(n_pairs >= 1 && pairs != nullptr, MDH_EINVAL, "sq: pairs missing");
    MDH_REQUIRE(mode >= MDH_SQ_AUTO && mode <= MDH_SQ_LATTICE_DMMA, MDH_EINVAL,
                "sq: invalid mode");
    bool all = false;
    for (int p = 0; p < n_pairs; ++p) {
        const int j = pairs[2 * p], k = pairs[2 * p + 1];
        if (j < 0 || k < 0) {
            MDH_REQUIRE(j == -1 && k == -1 && n_pairs == 1, MDH_EINVAL,
                        "sq: the pair (-1, -1) must be the only pair");
            all = true;
        } else {
            MDH_REQUIRE(j < n_groups && k < n_groups, MDH_EINVAL,
                        "sq: pair %d refers to a missing group", p);
        }
    }
    MDH_REQUIRE(mode != 2, MDH_EINVAL, "sq: invalid mode");   // retired selector value
    const bool want_lattice = mode == MDH_SQ_LATTICE_FP64 || mode == MDH_SQ_LATTICE_FP32 ||
                              mode == MDH_SQ_LATTICE_DMMA;
    MDH_REQUIRE(!want_lattice || (lat_n && lat_b), MDH_EINVAL,
                "sq: a lattice kernel was requested without lattice_n / lattice_b");

    S.configured = false;
    S.probe.pending = false;              // rates of another configuration do not carry over
    S.probe.copy_over_kernel = 0.0;
    S.n_total = n_total; S.n_groups = n_groups; S.n_q = n_q; S.n_pairs = n_pairs;
    S.n_rho = all ? 1 : n_groups;
    S.group_offsets.assign(goff, goff + n_groups + 1);
    S.pairs.assign(pairs, pairs + 2 * n_pairs);
    S.rho_frames = 0;
    S.n_chains = S.n_monomers = 0;
    S.cell = false;

    // ---- lattice work items (lattice_build_items) ----
    bool lattice = lat_n && lat_b && mode != MDH_SQ_GENERAL_FP64;
    std::vector<SqWorkItem> items;
    std::vector<int> qidx;
    std::vector<SqMmaItem> mitems;
    std::vector<int> mqidx;
    int mma_warps = 0;
    if (lattice) {
        int nm[3] = {0, 0, 0};
        std::vector<Column> cols;
        lattice = build_columns(n_q, lat_n, nm, cols);
        if (lattice) {
            lattice_build_items(cols, nm, items, qidx, S.block);
            for (int k = 0; k < 3; ++k) { S.nmax[k] = nm[k]; S.b[k] = lat_b[k]; }

            // ---- DMMA work items (sq_lattice_mma_kernel) ----
            if (mode == MDH_SQ_AUTO || mode == MDH_SQ_LATTICE_DMMA)
                mma_build_items(cols, nm, mitems, mqidx, mma_warps, S.mma_stats);
        }
    }
    MDH_REQUIRE(lattice || !want_lattice, MDH_EINVAL,
                "sq: wavevectors are not usable by the lattice kernels "
                "(need 0 <= n <= 1023 and no duplicates)");
    // The scalar lattice kernel keeps two phase-factor tables of (nx + ny + nz + 3) entries
    // x kPS particles in shared memory (launch_lattice): grids beyond ~75 points per axis
    // (fp64) do not fit, and the general kernel -- no tables -- takes them.
    if (lattice) {
        const size_t nt = (size_t)lattice_row_elems(S.nmax, nullptr, nullptr);
        const size_t elem = mode == MDH_SQ_LATTICE_FP32 ? sizeof(float) : sizeof(double);
        if (2 * elem * kPS * nt > kSqMaxSmem) {
            MDH_REQUIRE(mode == MDH_SQ_AUTO, MDH_EINVAL,
                        "sq: the phase-factor tables of this wavevector grid (%d x %d x %d) "
                        "do not fit in shared memory; use MDH_SQ_AUTO or MDH_SQ_GENERAL_FP64",
                        S.nmax[0] + 1, S.nmax[1] + 1, S.nmax[2] + 1);
            lattice = false;
            mitems.clear();
        }
    }
    S.lattice = lattice;
    // AUTO: the DMMA kernel needs enough (group, tile) pairs to load all four schedulers
    // of an SM (measured: 9 pairs lose to the scalar kernel by 27 %, 17 win by 4 %, 26 by 11 %, 49 by 1.8x)
    S.mma = lattice && !mitems.empty() && mma_smem_bytes(S.nmax) <= kMmaSmemLimit &&
            (mode == MDH_SQ_LATTICE_DMMA || S.mma_stats[1] >= kMmaAutoTiles);
    S.mode = !lattice ? MDH_SQ_GENERAL_FP64
             : mode == MDH_SQ_LATTICE_FP32 ? MDH_SQ_LATTICE_FP32
             : S.mma ? MDH_SQ_LATTICE_DMMA : MDH_SQ_LATTICE_FP64;
    S.n_items = (int)items.size();
    S.mma_items = S.mma ? (int)mitems.size() : 0;
    S.mma_warps = mma_warps;

    if (int rc = S.qv.reserve(sizeof(double) * 3 * n_q)) return rc;
    if (int rc = S.d_pairs.reserve(sizeof(int) * 2 * n_pairs)) return rc;
    if (int rc = S.ssf.reserve(sizeof(double) * (size_t)n_pairs * n_q)) return rc;
    MDH_CUDA(cudaMemcpyAsync(S.qv.p, wv, sizeof(double) * 3 * n_q, cudaMemcpyHostToDevice,
                             c->stream));
    MDH_CUDA(cudaMemcpyAsync(S.d_pairs.p, pairs, sizeof(int) * 2 * n_pairs,
                             cudaMemcpyHostToDevice, c->stream));
    MDH_CUDA(cudaMemsetAsync(S.ssf.p, 0, sizeof(double) * (size_t)n_pairs * n_q, c->stream));
    if (lattice) {
        if (int rc = S.items.reserve(sizeof(SqWorkItem) * items.size())) return rc;
        if (int rc = S.qidx.reserve(sizeof(int) * qidx.size())) return rc;
        MDH_CUDA(cudaMemcpyAsync(S.items.p, items.data(), sizeof(SqWorkItem) * items.size(),
                                 cudaMemcpyHostToDevice, c->stream));
        MDH_CUDA(cudaMemcpyAsync(S.qidx.p, qidx.data(), sizeof(int) * qidx.size(),
                                 cudaMemcpyHostToDevice, c->stream));
    }
    if (S.mma) {
        if (int rc = S.mitems.reserve(sizeof(SqMmaItem) * mitems.size())) return rc;
        if (int rc = S.mqidx.reserve(sizeof(int) * mqidx.size())) return rc;
        MDH_CUDA(cudaMemcpyAsync(S.mitems.p, mitems.data(), sizeof(SqMmaItem) * mitems.size(),
                                 cudaMemcpyHostToDevice, c->stream));
        MDH_CUDA(cudaMemcpyAsync(S.mqidx.p, mqidx.data(), sizeof(int) * mqidx.size(),
                                 cudaMemcpyHostToDevice, c->stream));
    }
    MDH_CUDA(cudaStreamSynchronize(c->stream));   // host sources are caller/local memory
    S.n_chunks = 0;
    S.configured = true;
    return MDH_OK;
}

// particle chunks: one rho row per group (or one row for everything)
static int sq_build_chunks(mdh_ctx *c, int n_frames)
{
    SqState &S = c->sq;
    const int item_blocks = S.mode == MDH_SQ_LATTICE_DMMA ? S.mma_items / S.mma_warps
                            : S.lattice ? S.n_items / S.block : (S.n_q + 127) / 128;
    // enough blocks for ~6 waves (two blocks per SM), chunks a multiple of the sub-chunk
    // length; the persistent DMMA kernel strides over ~40 small units per block instead
    // (its table pipeline runs across unit boundaries, so small units cost nothing and
    // the last, partial round is 1/40 of the launch)
    const int64_t rounds = S.mode == MDH_SQ_LATTICE_DMMA ? 40 : 12;
    int64_t want = ((int64_t)c->sm_count * rounds + (int64_t)item_blocks * n_frames - 1) /
                   ((int64_t)item_blocks * n_frames);
    int64_t len = (S.n_total + want - 1) / std::max<int64_t>(want, 1);
    len = std::max<int64_t>(256, std::min<int64_t>(len, 4096));
    // equal chunks (a short last chunk is a short last block of every frame)
    const int64_t span = S.n_rho == 1 ? S.n_total : S.n_total / S.n_groups;
    len = (span + (span + len - 1) / len - 1) / ((span + len - 1) / len);
    len = (len + kPS - 1) / kPS * kPS;
    if (S.n_chains > 0) len = -S.n_monomers;   // single-chain layout: its own cache key
    if (S.n_chunks > 0 && S.chunk_len == (int)len) return MDH_OK;
    std::vector<int4> ch;
    if (S.n_chains > 0) {
        for (int64_t k = 0; k < S.n_chains; ++k)
            ch.push_back(make_int4((int)(k * S.n_monomers), (int)((k + 1) * S.n_monomers), 0, 0));
    } else if (S.n_rho == 1) {
        for (int64_t s = 0; s < S.n_total; s += len)
            ch.push_back(make_int4((int)s, (int)std::min<int64_t>(S.n_total, s + len), 0, 0));
    } else {
        for (int g = 0; g < S.n_groups; ++g)
            for (int64_t s = S.group_offsets[g]; s < S.group_offsets[g + 1]; s += len)
                ch.push_back(make_int4((int)s,
                                       (int)std::min<int64_t>(S.group_offsets[g + 1], s + len),
                                       g, 0));
    }
    MDH_REQUIRE(S.n_chains > 0 || ch.size() <= 65535, MDH_EINVAL,
                "sq: too many particle chunks");
    if (int rc = S.chunks.reserve(sizeof(int4) * ch.size())) return rc;
    MDH_CUDA(cudaMemcpyAsync(S.chunks.p, ch.data(), sizeof(int4) * ch.size(),
                             cudaMemcpyHostToDevice, c->stream));
    MDH_CUDA(cudaStreamSynchronize(c->stream));
    S.n_chunks = (int)ch.size();
    S.chunk_len = (int)len;
    return MDH_OK;
}

// rho[v][row][q] = sum over the particles of row's group of exp(i q . r) for the
// n_vframes (virtual) frames of `raw`; vmap as in LatticeParams.  Zeroes rho first.
static int sq_compute_rho(mdh_ctx *c, const float *raw, int64_t stride, const int4 *vmap,
                          int n_vframes, double *rho, int nominal_frames)
{
    SqState &S = c->sq;
    if (int rc = sq_build_chunks(c, nominal_frames)) return rc;
    const size_t rho_bytes = sizeof(double) * 2 * (size_t)n_vframes * S.n_rho * S.n_q;
    if (S.n_chains == 0) MDH_CUDA(cudaMemsetAsync(rho, 0, rho_bytes, c->stream));
    MDH_REQUIRE(S.n_chains == 0 || S.lattice, MDH_ESTATE,
                "sq: single-chain mode needs lattice wavevectors");
    if (S.mode == MDH_SQ_LATTICE_DMMA) {
        MmaParams P;
        mma_layout(S.nmax, &P.offy, &P.offz, &P.nzpad, &P.R);
        P.raw = raw; P.stride = stride; P.vmap = vmap;
        P.chunks = S.chunks.as<int4>();
        P.items = S.mitems.as<SqMmaItem>();
        P.qidx = S.mqidx.as<int>();
        P.rho = rho;
        P.n_rho = S.n_rho; P.n_q = S.n_q;
        P.chain_out = S.n_chains > 0 ? S.ssf.as<double>() : nullptr;
        P.n_chunks = S.n_chunks;
        MDH_REQUIRE((int64_t)S.n_chunks * n_vframes < (1ll << 31), MDH_EINVAL,
                    "sq: too many (frame, chunk) work units in one call");
        P.n_units = S.n_chunks * n_vframes;
        for (int k = 0; k < 3; ++k) { P.b[k] = S.b[k]; P.nmax[k] = S.nmax[k]; }
        const size_t smem = mma_smem_bytes(S.nmax);
        MDH_CUDA(cudaFuncSetAttribute(sq_lattice_mma_kernel,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        // persistent: one block per SM (and item block), striding over the work units
        const int item_blocks = S.mma_items / S.mma_warps;
        dim3 grid(item_blocks, std::min(P.n_units, std::max(1, c->sm_count / item_blocks)));
        sq_lattice_mma_kernel<<<grid, S.mma_warps * 32 + kMmaProducers, smem, c->stream>>>(P);
        MDH_CUDA(cudaGetLastError());
        c->launches++;
        return MDH_OK;
    }
    if (S.lattice) {
        LatticeParams P;
        // row layout in table elements: E_x re | E_x im | E_y re | E_y im | E_z (re, im)
        P.nt = lattice_row_elems(S.nmax, &P.offy, &P.offz);
        P.raw = raw; P.stride = stride; P.vmap = vmap;
        P.chunks = S.chunks.as<int4>();
        P.items = S.items.as<SqWorkItem>();
        P.qidx = S.qidx.as<int>();
        P.rho = rho;
        P.n_rho = S.n_rho; P.n_q = S.n_q;
        P.chain_out = S.n_chains > 0 ? S.ssf.as<double>() : nullptr;
        P.n_chunks = S.n_chunks;
        for (int k = 0; k < 3; ++k) { P.b[k] = S.b[k]; P.nmax[k] = S.nmax[k]; }
        dim3 grid(S.n_items / S.block, std::min(S.n_chunks, 65535), n_vframes);
        return S.mode == MDH_SQ_LATTICE_FP32 ? launch_lattice<float>(c, P, grid, S.block)
                                             : launch_lattice<double>(c, P, grid, S.block);
    }
    GeneralParams P;
    P.raw = raw; P.stride = stride; P.vmap = vmap;
    P.chunks = S.chunks.as<int4>();
    P.qv = S.qv.as<double>();
    P.rho = rho;
    P.n_rho = S.n_rho; P.n_q = S.n_q;
    dim3 grid((S.n_q + 127) / 128, S.n_chunks, n_vframes);
    sq_general_kernel<<<grid, 128, 0, c->stream>>>(P);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    return MDH_OK;
}

// float64 coordinates -> the S(q) kernels' float32 frames without losing a bit that
// matters: frame f of dst = the coordinate rounded to float32 ("hi"), frame n_frames + f
// = hi - x rounded to float32 (the NEGATED remainder), vmap[f] = {f, n_frames + f}: the
// kernels' displacement path then forms (double)hi - (double)(hi - x) = x up to
// 2^-48 |x| in fp64 -- the reference's float64 position buffer
// (/root/reference/src/mdhelper/analysis/structure.py:1468-1486) to 14 digits.
__global__ void sq_split_kernel(const double *__restrict__ src, int64_t src_stride,
                                float *__restrict__ dst, int64_t n3, int n_frames,
                                int4 *__restrict__ vmap)
{
    const int f = blockIdx.y;
    const double *s = src + (int64_t)f * src_stride;
    float *hi = dst + (int64_t)f * n3;
    float *nlo = dst + (int64_t)(n_frames + f) * n3;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n3;
         k += (int64_t)gridDim.x * blockDim.x) {
        const double x = s[k];
        const float h = (float)x;
        hi[k] = h;
        nlo[k] = (float)((double)h - x);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) vmap[f] = make_int4(f, n_frames + f, 0, 0);
}

// A cell is set (mdh_sq_set_cell): every coordinate r enters as its fractional coordinates
// s = r H^-1, formed in fp64 by tri_frac.  With q = n B*, B* = 2 pi H^-T, q . r = 2 pi n . s,
// so the lattice kernels evaluate the reciprocal-lattice grid of the cell with
// lattice_b = (2 pi, 2 pi, 2 pi), and the general kernel any q given as k = q H^T.
// split != NULL: s is written as sq_split_kernel writes float64 coordinates (frame f of
// split: float32 hi, frame n_frames + f: negated float32 remainder; vmap[f]).  Else s itself
// goes to win ([n_frames][n][3] doubles: the ISF's float64 window).
template <typename T>
__global__ void sq_frac_kernel(const T *__restrict__ src, int64_t src_stride, int64_t n,
                               const TriBox h, int n_frames, float *__restrict__ split,
                               int4 *__restrict__ vmap, double *__restrict__ win)
{
    const int f = blockIdx.y;
    const T *r = src + (int64_t)f * src_stride;
    const int64_t n3 = 3 * n;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x) {
        double s[3];
        tri_frac(r[3 * i], r[3 * i + 1], r[3 * i + 2], h, s[0], s[1], s[2]);
        if (split) {
            float *hi = split + (int64_t)f * n3 + 3 * i;
            float *nlo = split + (int64_t)(n_frames + f) * n3 + 3 * i;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                const float v = (float)s[k];
                hi[k] = v;
                nlo[k] = (float)((double)v - s[k]);
            }
        } else {
            double *w = win + (int64_t)f * n3 + 3 * i;
#pragma unroll
            for (int k = 0; k < 3; ++k) w[k] = s[k];
        }
    }
    if (split && blockIdx.x == 0 && threadIdx.x == 0) vmap[f] = make_int4(f, n_frames + f, 0, 0);
}

template <typename T>
static int launch_frac(mdh_ctx *c, const T *src, int64_t src_stride, int n_frames,
                       float *split, int4 *vmap, double *win)
{
    const SqState &S = c->sq;
    dim3 grid((unsigned)std::min<int64_t>((S.n_total + 255) / 256, 1024), n_frames);
    sq_frac_kernel<T><<<grid, 256, 0, c->stream>>>(src, src_stride, S.n_total, S.h, n_frames,
                                                   split, vmap, win);
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    return MDH_OK;
}

int sq_set_cell_impl(mdh_ctx *c, const double *cell)
{
    SqState &S = c->sq;
    MDH_REQUIRE(S.configured, MDH_ESTATE, "sq: set the cell after mdh_sq_configure");
    if (cell) {
        for (int k = 0; k < 9; ++k)
            MDH_REQUIRE(std::isfinite(cell[k]), MDH_EINVAL, "sq: the cell matrix is not finite");
        MDH_REQUIRE(cell[1] == 0.0 && cell[2] == 0.0 && cell[5] == 0.0, MDH_EINVAL,
                    "sq: the cell matrix is not lower triangular");
        MDH_REQUIRE(cell[0] > 0.0 && cell[4] > 0.0 && cell[8] > 0.0, MDH_EINVAL,
                    "sq: the cell matrix is not a valid cell");
        S.h = TriBox{cell[0], cell[3], cell[4], cell[6], cell[7], cell[8]};
    }
    S.cell = cell != nullptr;
    // sums over other coordinates do not carry over; the ISF window's layout follows the
    // cell, so an ISF run is configured after this call
    S.rho_frames = 0;
    c->isf.on = false;
    MDH_CUDA(cudaMemsetAsync(S.ssf.p, 0, sizeof(double) * (size_t)S.n_pairs * S.n_q, c->stream));
    return MDH_OK;
}

template <typename T>
static int sq_accumulate_piece(mdh_ctx *c, const T *pos, int64_t stride, int location,
                               int n_frames, int nominal_frames, bool probe);

template <typename T>
static int sq_accumulate_any(mdh_ctx *c, const T *pos, int64_t stride, int location,
                             int n_frames)
{
    SqState &S = c->sq;
    MDH_REQUIRE(S.configured, MDH_ESTATE, "sq: accumulate before configure");
    MDH_REQUIRE(n_frames >= 1 && n_frames <= 65535, MDH_EINVAL,
                "sq: n_frames per call must be in [1, 65535]");
    MDH_REQUIRE(pos != nullptr, MDH_EINVAL, "sq: coordinate pointer is NULL");
    MDH_REQUIRE(stride >= 3 * S.n_total, MDH_EINVAL, "sq: frame_stride < 3*n_total");
    MDH_REQUIRE(location == MDH_HOST || location == MDH_DEVICE, MDH_EINVAL,
                "sq: invalid location");
    MDH_TRACE("sq_accumulate: %d frames of %d-byte coordinates, location %d", n_frames,
              (int)sizeof(T), location);
    // host input in pieces: the copy of one piece (copy stream) overlaps the kernels of
    // the previous one (compute stream); the particle chunks are laid out once, for the
    // whole call
    if (location == MDH_HOST) {
        S.probe.learn();
        const std::vector<int> pieces = mdh_plan_pieces(
            n_frames, 3.0 * sizeof(T) * (double)S.n_total, S.probe.copy_over_kernel);
        // staging of the largest piece up front: a buffer that grows between pieces would
        // be freed (a device synchronisation) while the previous piece is still running
        const int longest = *std::max_element(pieces.begin(), pieces.end());
        for (int slot = 0; slot < 2 && pieces.size() > 1; ++slot)
            if (int rc = S.raw[slot].reserve(sizeof(T) * 3 * S.n_total * (size_t)longest))
                return rc;
        if (sizeof(T) == 8 || S.cell) {
            if (int rc = S.split.reserve(sizeof(float) * 6 * S.n_total * (size_t)longest))
                return rc;
            if (int rc = S.split_vmap.reserve(sizeof(int4) * (size_t)longest)) return rc;
        }
        int f0 = 0;
        for (size_t k = 0; k < pieces.size(); ++k) {
            // the last piece of a call with several pieces is the rate probe of the next call
            const bool probe = pieces.size() > 1 && k + 1 == pieces.size() && !S.probe.pending;
            if (int rc = sq_accumulate_piece(c, pos + (int64_t)f0 * stride, stride, location,
                                             pieces[k], n_frames, probe)) return rc;
            f0 += pieces[k];
        }
        return MDH_OK;
    }
    return sq_accumulate_piece(c, pos, stride, location, n_frames, n_frames, false);
}

int sq_accumulate_impl(mdh_ctx *c, const float *pos, int64_t stride, int location,
                       int n_frames)
{
    return sq_accumulate_any(c, pos, stride, location, n_frames);
}

int sq_accumulate_f64_impl(mdh_ctx *c, const double *pos, int64_t stride, int location,
                           int n_frames)
{
    return sq_accumulate_any(c, pos, stride, location, n_frames);
}

// nominal_frames: the frame count the particle chunks are laid out for (the whole call;
// its pieces reuse the layout instead of rebuilding it)
template <typename T>
static int sq_accumulate_piece(mdh_ctx *c, const T *pos, int64_t stride, int location,
                               int n_frames, int nominal_frames, bool probe)
{
    constexpr bool kF64 = sizeof(T) == 8;
    SqState &S = c->sq;
    const T *dsrc = pos;
    int64_t dstride = stride;
    int slot = 0;
    probe = probe && location == MDH_HOST;
    if (probe)
        if (int rc = S.probe.ensure()) return rc;
    if (location == MDH_HOST) {
        if (int rc = c->stager.acquire(&slot)) return rc;
        DevBuf &raw = S.raw[slot];
        if (int rc = raw.reserve(sizeof(T) * 3 * S.n_total * n_frames)) return rc;
        if (probe) MDH_CUDA(cudaEventRecord(S.probe.ev[0], c->stager.copy));
        MDH_CUDA(mdh_copy_frames(raw.p, sizeof(T) * 3 * S.n_total, pos,
                                   sizeof(T) * stride, sizeof(T) * 3 * S.n_total,
                                   n_frames, cudaMemcpyHostToDevice, c->stager.copy));
        if (probe) MDH_CUDA(cudaEventRecord(S.probe.ev[1], c->stager.copy));
        if (int rc = c->stager.publish(c->stream, slot)) return rc;
        dsrc = raw.as<T>();
        dstride = 3 * S.n_total;
    }
    const size_t rho_bytes = sizeof(double) * 2 * (size_t)n_frames * S.n_rho * S.n_q;
    if (S.n_chains == 0)
        if (int rc = S.rho.reserve(rho_bytes)) return rc;
    const float *fsrc = nullptr;
    const int4 *vmap = nullptr;
    if (kF64 || S.cell) {
        const int64_t n3 = 3 * S.n_total;
        if (int rc = S.split.reserve(sizeof(float) * 2 * n3 * n_frames)) return rc;
        if (int rc = S.split_vmap.reserve(sizeof(int4) * (size_t)n_frames)) return rc;
        fsrc = S.split.as<float>();
        vmap = S.split_vmap.as<int4>();
    } else if constexpr (!kF64) {
        fsrc = dsrc;
    }

    if (int rc = c->t_sq.begin(c->stream)) return rc;
    if (probe) MDH_CUDA(cudaEventRecord(S.probe.ev[2], c->stream));
    if (S.cell) {
        if (int rc = launch_frac(c, dsrc, dstride, n_frames, S.split.as<float>(),
                                 S.split_vmap.as<int4>(), (double *)nullptr)) return rc;
        dstride = 3 * S.n_total;
    } else if constexpr (kF64) {
        const int64_t n3 = 3 * S.n_total;
        dim3 grid((unsigned)std::min<int64_t>((n3 + 255) / 256, 1024), n_frames);
        sq_split_kernel<<<grid, 256, 0, c->stream>>>(dsrc, dstride, S.split.as<float>(), n3,
                                                     n_frames, S.split_vmap.as<int4>());
        MDH_CUDA(cudaGetLastError());
        c->launches++;
        dstride = n3;
    }
    if (int rc = sq_compute_rho(c, fsrc, dstride, vmap, n_frames, S.rho.as<double>(),
                                nominal_frames)) return rc;
    if (S.n_chains > 0) {
        // the kernel has added |rho_chain|^2 to the accumulator itself
        S.rho_frames = 0;
        if (probe) {
            MDH_CUDA(cudaEventRecord(S.probe.ev[3], c->stream));
            S.probe.pending = true;
        }
        if (location == MDH_HOST)
            if (int rc = c->stager.retire(c->stream, slot)) return rc;
        return c->t_sq.end(c->stream);
    }
    dim3 fgrid((S.n_q + 127) / 128, S.n_pairs);
    sq_finalize_kernel<<<fgrid, 128, 0, c->stream>>>(S.rho.as<double2>(), n_frames, S.n_rho,
                                                     S.n_q, S.d_pairs.as<int>(), S.n_pairs,
                                                     S.ssf.as<double>());
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    S.rho_frames = n_frames;
    if (probe) {
        MDH_CUDA(cudaEventRecord(S.probe.ev[3], c->stream));
        S.probe.pending = true;
    }
    if (location == MDH_HOST)
        if (int rc = c->stager.retire(c->stream, slot)) return rc;
    return c->t_sq.end(c->stream);
}

// ---- intermediate scattering function (SURVEY.md section 8(f) rank 1) ---------------
// Replaces the per-frame work of IntermediateScatteringFunction._single_frame
// (/root/reference/src/mdhelper/analysis/structure.py:1959-2085):
//   coherent:    rho(q, t) of every frame is kept on the device; at fetch time
//                cisf[lag][pair] = sum_t Re(rho_j(t - lag) conj(rho_k(t))) (+ j <-> k)
//   incoherent:  iisf[lag][group] += Re sum_particles exp(i q . (r(t) - r(t - lag)))
//                -- the S(q) kernels on displacement vectors of a coordinate window
//                that holds the last n_lags - 1 frames.
// Normalisation, unique-|q| grouping and sorting stay on the host.

namespace {

__global__ void isf_coherent_kernel(const double2 *__restrict__ rho, int n_frames, int n_rho,
                                    int n_q, const int *__restrict__ pairs, int n_pairs,
                                    double *__restrict__ cisf)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    const int p = blockIdx.y, lag = blockIdx.z;
    if (q >= n_q) return;
    int j = pairs[2 * p], k = pairs[2 * p + 1];
    if (j < 0) j = k = 0;
    double acc = 0.0;
    for (int t = lag; t < n_frames; ++t) {
        const double2 aj = rho[((int64_t)(t - lag) * n_rho + j) * n_q + q];
        const double2 bk = rho[((int64_t)t * n_rho + k) * n_q + q];
        acc += aj.x * bk.x + aj.y * bk.y;              // Re(rho_j(t0) conj(rho_k(t)))
        if (j != k) {
            const double2 ak = rho[((int64_t)(t - lag) * n_rho + k) * n_q + q];
            const double2 bj = rho[((int64_t)t * n_rho + j) * n_q + q];
            acc += ak.x * bj.x + ak.y * bj.y;
        }
    }
    cisf[((int64_t)lag * n_pairs + p) * n_q + q] = acc;
}

// iisf[lag(v)][row][q] += Re rho_tmp[v][row][q]; one thread per (row, q) walks the
// virtual frames of the batch in order (deterministic, no atomics)
__global__ void isf_incoherent_kernel(const double2 *__restrict__ rho_tmp,
                                      const int4 *__restrict__ vmap, int n_v, int n_rho,
                                      int n_q, double *__restrict__ iisf)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    const int row = blockIdx.y;
    if (q >= n_q) return;
    for (int v = 0; v < n_v; ++v) {
        const int lag = vmap[v].z;
        iisf[((int64_t)lag * n_rho + row) * n_q + q] +=
            rho_tmp[((int64_t)v * n_rho + row) * n_q + q].x;
    }
}

// float64 window: displacement of virtual frame v = (t, t0, lag) in fp64, written as
// float32 + negated float32 remainder (frames v and n_v + v of dst; see sq_split_kernel)
__global__ void isf_displacement_split_kernel(const double *__restrict__ win, int64_t n3,
                                              const int4 *__restrict__ vin, int n_v,
                                              float *__restrict__ dst,
                                              int4 *__restrict__ vout)
{
    const int v = blockIdx.y;
    const int4 vm = vin[v];
    const double *a = win + (int64_t)vm.x * n3;
    const double *b = win + (int64_t)vm.y * n3;
    float *hi = dst + (int64_t)v * n3;
    float *nlo = dst + (int64_t)(n_v + v) * n3;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n3;
         k += (int64_t)gridDim.x * blockDim.x) {
        const double d = a[k] - b[k];
        const float h = (float)d;
        hi[k] = h;
        nlo[k] = (float)((double)h - d);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) vout[v] = make_int4(v, n_v + v, vm.z, 0);
}

}  // namespace

// Single-chain structure factor (SURVEY.md section 8(f) rank 3;
// /root/reference/src/mdhelper/analysis/polymer.py:1096-1099): the particles are
// n_chains consecutive runs of n_monomers; every accumulate call adds
// sum over frames and chains of |sum over the chain's monomers of exp(i q . r)|^2.
int sq_configure_chains_impl(mdh_ctx *c, int64_t n_chains, int64_t n_monomers)
{
    SqState &S = c->sq;
    MDH_REQUIRE(S.configured, MDH_ESTATE, "sq: configure the wavevectors first");
    MDH_REQUIRE(S.lattice, MDH_EINVAL,
                "sq: single-chain mode needs lattice wavevectors (lattice_n / lattice_b)");
    MDH_REQUIRE(S.n_pairs == 1 && S.n_rho == 1, MDH_EINVAL,
                "sq: single-chain mode needs the single pair (-1, -1)");
    MDH_REQUIRE(n_chains >= 1 && n_monomers >= 1 && n_chains * n_monomers == S.n_total,
                MDH_EINVAL, "sq: n_chains * n_monomers must equal n_total");
    S.n_chains = n_chains;
    S.n_monomers = n_monomers;
    S.n_chunks = 0;                    // rebuild the chunk list
    return MDH_OK;
}

int isf_configure_impl(mdh_ctx *c, int n_lags, int incoherent, int64_t max_frames)
{
    SqState &S = c->sq;
    IsfState &I = c->isf;
    MDH_REQUIRE(S.configured, MDH_ESTATE, "isf: the wavevectors are not configured");
    MDH_REQUIRE(S.n_chains == 0, MDH_ESTATE, "isf: not available in single-chain mode");
    MDH_REQUIRE(n_lags >= 1 && n_lags <= 65535, MDH_EINVAL, "isf: n_lags must be in [1, 65535]");
    MDH_REQUIRE(max_frames >= n_lags, MDH_EINVAL, "isf: fewer frames than time lags");
    I.on = false;
    I.n_lags = n_lags; I.incoherent = incoherent != 0; I.max_frames = max_frames;
    I.n_done = 0; I.window_frames = 0; I.which = 0;
    const size_t row = sizeof(double) * 2 * (size_t)S.n_rho * S.n_q;
    if (int rc = I.rho_all.reserve(row * (size_t)max_frames)) return rc;
    if (int rc = I.cisf.reserve(sizeof(double) * (size_t)n_lags * S.n_pairs * S.n_q)) return rc;
    if (I.incoherent) {
        const size_t bytes = sizeof(double) * (size_t)n_lags * S.n_rho * S.n_q;
        if (int rc = I.iisf.reserve(bytes)) return rc;
        MDH_CUDA(cudaMemsetAsync(I.iisf.p, 0, bytes, c->stream));
    }
    I.on = true;
    return MDH_OK;
}

// T = float: the window holds the float32 frames the kernels read directly; T = double
// (centres of mass: the reference's float64 position buffer, structure.py:1927-1957): the
// window holds doubles and the kernels get float32 + remainder copies.  A cell set: the
// window holds the fractional coordinates (sq_frac_kernel) as doubles, whatever T, and the
// float64 path follows (displacements s(t) - s(t - lag) in fp64).
template <typename T>
static int isf_accumulate_any(mdh_ctx *c, const T *pos, int64_t stride, int location,
                              int n_frames)
{
    SqState &S = c->sq;
    IsfState &I = c->isf;
    MDH_REQUIRE(S.configured && I.on, MDH_ESTATE, "isf: accumulate before configure");
    MDH_REQUIRE(n_frames >= 1 && n_frames <= 65535, MDH_EINVAL,
                "isf: n_frames per call must be in [1, 65535]");
    MDH_REQUIRE(pos != nullptr, MDH_EINVAL, "isf: coordinate pointer is NULL");
    MDH_REQUIRE(stride >= 3 * S.n_total, MDH_EINVAL, "isf: frame_stride < 3*n_total");
    MDH_REQUIRE(location == MDH_HOST || location == MDH_DEVICE, MDH_EINVAL,
                "isf: invalid location");
    MDH_REQUIRE(I.n_done + n_frames <= I.max_frames, MDH_EINVAL,
                "isf: more frames than announced at configure (%lld)", (long long)I.max_frames);

    // coordinate window: [frames kept from earlier calls][the frames of this call]
    const int64_t fsz = 3 * S.n_total;                     // coordinates per frame
    const bool wide = sizeof(T) == 8 || S.cell;           // the window holds doubles
    const size_t esz = wide ? sizeof(double) : sizeof(float);
    const int keep = I.window_frames;
    DevBuf &win = I.window[I.which];
    const size_t need = esz * fsz * (size_t)(keep + n_frames);
    if (win.cap < need) {
        // grow WITHOUT losing the frames kept from earlier calls (DevBuf::reserve frees)
        DevBuf bigger;
        if (int rc = bigger.reserve(need)) return rc;
        if (keep > 0)
            MDH_CUDA(cudaMemcpyAsync(bigger.p, win.p, esz * fsz * (size_t)keep,
                                     cudaMemcpyDeviceToDevice, c->stream));
        MDH_CUDA(cudaStreamSynchronize(c->stream));
        win.adopt(bigger);
    }
    const T *src = pos;                 // where sq_frac_kernel reads the frames
    int64_t src_stride = stride;
    if (!S.cell) {
        MDH_CUDA(mdh_copy_frames(win.as<T>() + fsz * keep, sizeof(T) * fsz, pos,
                                 sizeof(T) * stride, sizeof(T) * fsz, n_frames,
                                 location == MDH_HOST ? cudaMemcpyHostToDevice
                                                      : cudaMemcpyDeviceToDevice, c->stream));
    } else if (location == MDH_HOST) {
        if (int rc = I.stage.reserve(sizeof(T) * fsz * (size_t)n_frames)) return rc;
        MDH_CUDA(mdh_copy_frames(I.stage.p, sizeof(T) * fsz, pos, sizeof(T) * stride,
                                 sizeof(T) * fsz, n_frames, cudaMemcpyHostToDevice, c->stream));
        src = I.stage.as<T>();
        src_stride = fsz;
    }
    if (int rc = c->t_sq.begin(c->stream)) return rc;
    if (S.cell)
        if (int rc = launch_frac(c, src, src_stride, n_frames, nullptr, nullptr,
                                 win.as<double>() + fsz * keep)) return rc;

    // rho(q, t) of the new frames, straight into the per-frame store
    const size_t row = (size_t)2 * S.n_rho * S.n_q;        // doubles per frame
    const float *fwin = nullptr;
    if (wide) {
        if (int rc = S.split.reserve(sizeof(float) * 2 * fsz * n_frames)) return rc;
        if (int rc = S.split_vmap.reserve(sizeof(int4) * (size_t)n_frames)) return rc;
        dim3 grid((unsigned)std::min<int64_t>((fsz + 255) / 256, 1024), n_frames);
        sq_split_kernel<<<grid, 256, 0, c->stream>>>(win.as<double>() + fsz * keep, fsz,
                                                     S.split.as<float>(), fsz, n_frames,
                                                     S.split_vmap.as<int4>());
        MDH_CUDA(cudaGetLastError());
        c->launches++;
        if (int rc = sq_compute_rho(c, S.split.as<float>(), fsz, S.split_vmap.as<int4>(),
                                    n_frames, I.rho_all.as<double>() + row * I.n_done,
                                    n_frames)) return rc;
    } else {
        fwin = win.as<float>();
        if (int rc = sq_compute_rho(c, fwin + fsz * keep, fsz, nullptr, n_frames,
                                    I.rho_all.as<double>() + row * I.n_done, n_frames))
            return rc;
    }

    if (I.incoherent) {
        // virtual frames (t, lag): displacement r(t) - r(t - lag), lag = 0 included
        // (the reference evaluates it too: sum of exp(0) = N)
        MDH_REQUIRE((int64_t)n_frames * I.n_lags <= (1ll << 26), MDH_EINVAL,
                    "isf: n_frames * n_lags per call must not exceed 2^26 (pass fewer frames "
                    "per call)");
        std::vector<int4> vm;
        for (int t = 0; t < n_frames; ++t) {
            const int64_t tg = I.n_done + t;                // global frame index
            const int lags = (int)std::min<int64_t>(I.n_lags, tg + 1);
            for (int lag = 0; lag < lags; ++lag)
                vm.push_back(make_int4(keep + t, keep + t - lag, lag, 0));
        }
        // batches sized to ~256 MB of temporary rho
        int vmax = (int)std::max<size_t>(1, std::min<size_t>(
            8192, ((size_t)256 << 20) / (sizeof(double) * row)));
        if (wide) {
            // ... and to ~256 MB of materialised displacements
            vmax = (int)std::max<size_t>(1, std::min<size_t>(
                vmax, ((size_t)256 << 20) / (sizeof(float) * 2 * (size_t)fsz)));
            if (int rc = S.split.reserve(sizeof(float) * 2 * fsz * (size_t)vmax)) return rc;
            if (int rc = S.split_vmap.reserve(sizeof(int4) * (size_t)vmax)) return rc;
        }
        if (int rc = I.vmap.reserve(sizeof(int4) * (size_t)vmax)) return rc;
        if (int rc = S.rho.reserve(sizeof(double) * row * (size_t)vmax)) return rc;
        for (size_t v0 = 0; v0 < vm.size(); v0 += vmax) {
            const int nv = (int)std::min<size_t>(vmax, vm.size() - v0);
            // pageable source: staged by the runtime before the call returns
            MDH_CUDA(cudaMemcpyAsync(I.vmap.p, vm.data() + v0, sizeof(int4) * nv,
                                     cudaMemcpyHostToDevice, c->stream));
            const int4 *vdev = I.vmap.as<int4>();
            if (wide) {
                dim3 sgrid((unsigned)std::min<int64_t>((fsz + 255) / 256, 1024), nv);
                isf_displacement_split_kernel<<<sgrid, 256, 0, c->stream>>>(
                    win.as<double>(), fsz, I.vmap.as<int4>(), nv, S.split.as<float>(),
                    S.split_vmap.as<int4>());
                MDH_CUDA(cudaGetLastError());
                c->launches++;
                vdev = S.split_vmap.as<int4>();
                if (int rc = sq_compute_rho(c, S.split.as<float>(), fsz, vdev, nv,
                                            S.rho.as<double>(), std::max(nv, 64))) return rc;
            } else {
                if (int rc = sq_compute_rho(c, fwin, fsz, vdev, nv, S.rho.as<double>(),
                                            std::max(nv, 64))) return rc;
            }
            dim3 grid((S.n_q + 127) / 128, S.n_rho);
            isf_incoherent_kernel<<<grid, 128, 0, c->stream>>>(
                S.rho.as<double2>(), vdev, nv, S.n_rho, S.n_q, I.iisf.as<double>());
            MDH_CUDA(cudaGetLastError());
            c->launches++;
        }
        // keep the last n_lags - 1 frames for the next call (other window buffer)
        const int total = keep + n_frames;
        const int next_keep = std::min(total, I.n_lags - 1);
        DevBuf &nxt = I.window[I.which ^ 1];
        if (next_keep > 0) {
            if (int rc = nxt.reserve(esz * fsz * (size_t)next_keep)) return rc;
            MDH_CUDA(cudaMemcpyAsync(nxt.p, win.as<char>() + esz * fsz * (total - next_keep),
                                     esz * fsz * next_keep,
                                     cudaMemcpyDeviceToDevice, c->stream));
        }
        I.window_frames = next_keep;
        I.which ^= 1;
    }
    I.n_done += n_frames;
    S.rho_frames = 0;
    return c->t_sq.end(c->stream);
}

int isf_accumulate_impl(mdh_ctx *c, const float *pos, int64_t stride, int location,
                        int n_frames)
{
    MDH_REQUIRE(c->isf.n_done == 0 || !c->isf.f64, MDH_ESTATE,
                "isf: float32 frames after float64 frames in one run");
    c->isf.f64 = false;
    return isf_accumulate_any(c, pos, stride, location, n_frames);
}

int isf_accumulate_f64_impl(mdh_ctx *c, const double *pos, int64_t stride, int location,
                            int n_frames)
{
    MDH_REQUIRE(c->isf.n_done == 0 || c->isf.f64, MDH_ESTATE,
                "isf: float64 frames after float32 frames in one run");
    c->isf.f64 = true;
    return isf_accumulate_any(c, pos, stride, location, n_frames);
}

int isf_fetch_impl(mdh_ctx *c, double *cisf, double *iisf)
{
    SqState &S = c->sq;
    IsfState &I = c->isf;
    MDH_REQUIRE(S.configured && I.on, MDH_ESTATE, "isf: fetch before configure");
    MDH_REQUIRE(cisf != nullptr, MDH_EINVAL, "isf: cisf is NULL");
    MDH_REQUIRE(!iisf || I.incoherent, MDH_EINVAL,
                "isf: the incoherent part was not requested at configure");
    MDH_REQUIRE(I.n_done >= 1, MDH_ESTATE, "isf: no frame has been processed");
    dim3 grid((S.n_q + 127) / 128, S.n_pairs, I.n_lags);
    isf_coherent_kernel<<<grid, 128, 0, c->stream>>>(I.rho_all.as<double2>(), (int)I.n_done,
                                                     S.n_rho, S.n_q, S.d_pairs.as<int>(),
                                                     S.n_pairs, I.cisf.as<double>());
    MDH_CUDA(cudaGetLastError());
    c->launches++;
    MDH_CUDA(cudaMemcpyAsync(cisf, I.cisf.p, sizeof(double) * (size_t)I.n_lags * S.n_pairs * S.n_q,
                             cudaMemcpyDeviceToHost, c->stream));
    if (iisf)
        MDH_CUDA(cudaMemcpyAsync(iisf, I.iisf.p,
                                 sizeof(double) * (size_t)I.n_lags * S.n_rho * S.n_q,
                                 cudaMemcpyDeviceToHost, c->stream));
    MDH_CUDA(cudaStreamSynchronize(c->stream));
    return MDH_OK;
}
