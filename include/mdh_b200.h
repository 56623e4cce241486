/*
 * mdh_b200.h -- C ABI of libmdh_b200.so, the B200 (sm_100a) implementation of
 * mdhelper's per-frame structural-analysis hot path.
 *
 * The reference (bbye98/mdhelper) is pure Python and has no FFI boundary of its
 * own; the seams this ABI sits under are (paths relative to the reference root):
 *
 *   seam #1  radial_histogram(pos1, pos2, n_bins, range, dims, *, exclusion)
 *            src/mdhelper/analysis/structure.py:32-104, called per frame from
 *            RadialDistributionFunction._single_frame (:750-791) and
 *            _single_frame_parallel (:793-835)             -> mdh_rdf_*
 *   seam #2  self._delta_fourier_transform_sum(qs, rs) -> c16[N_q]
 *            src/mdhelper/algorithm/accelerated.py:81-165, called per frame from
 *            StructureFactor._single_frame (structure.py:1481-1527), followed by
 *            ssf += |rho|^2 or 2 Re(rho_j rho_k*)           -> mdh_sq_*
 *   frame loop  MDAnalysis AnalysisBase.run / ParallelAnalysisBase.run
 *            src/mdhelper/analysis/base.py:137-172, 312-507 -> the *_accumulate
 *            entry points take a BATCH of frames; the host keeps the loop.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross the boundary.
 *   - every function returns MDH_OK (0) or a negative MDH_E* code; the message is
 *     in a thread-local string returned by mdh_last_error().  Nothing throws or
 *     aborts across the ABI.
 *   - the caller owns every buffer it passes and must keep host buffers alive
 *     until mdh_sync() (accumulate calls are asynchronous w.r.t. the host when
 *     the host buffers are pinned).  The context owns all device memory.
 *   - a context is bound to one CUDA device and one stream; calls on one context
 *     are not re-entrant; different contexts may be driven from different host
 *     threads.
 *   - coordinates are float32, row-major [frame][particle][3]; frame_stride is
 *     the distance between consecutive frames in FLOATS (>= 3*n), so a slice of
 *     a larger [F][N][3] trajectory array can be passed without repacking.
 *   - boxes are float32 [frame][3] (orthorhombic edge lengths; this is
 *     ts.dimensions[:3] of the reference).  Triclinic cells go through
 *     mdh_rdf_accumulate_triclinic.
 */
#ifndef MDH_B200_H
#define MDH_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MDH_ABI_VERSION 1

enum {
    MDH_OK = 0,
    MDH_EINVAL = -1,   /* bad argument (Python layer raises ValueError)      */
    MDH_ECUDA = -2,    /* CUDA runtime failure (RuntimeError)                */
    MDH_ESTATE = -3,   /* call sequence error, e.g. accumulate before configure */
    MDH_ENOMEM = -4    /* host or device allocation failed                   */
};

/* where a coordinate pointer lives */
enum { MDH_HOST = 0, MDH_DEVICE = 1 };

/* pair-kernel strategy */
enum {
    MDH_RDF_AUTO = 0,      /* choose from n, box and cut-off per batch       */
    MDH_RDF_ALLPAIRS = 1,  /* tiled all-pairs (r_max up to half the box)     */
    MDH_RDF_CELLS = 2      /* cell list, 27-cell stencil (cut-off runs)      */
};

/* histogram privatisation inside the pair kernels (same counts either way) */
enum {
    MDH_HIST_AUTO = 0,
    MDH_HIST_WARP_ATOMIC = 1,  /* one u32 histogram per warp, shared-memory atomics */
    MDH_HIST_LANE_PRIVATE = 2  /* one packed 8-bit histogram per lane, no atomics   */
};

/* arithmetic of the all-pairs kernel (same counts either way, bit for bit) */
enum {
    MDH_FILTER_AUTO = 0,   /* fp32 filter whenever the configuration is eligible      */
    MDH_FILTER_OFF = 1,    /* every pair through the reference's fp64 arithmetic      */
    MDH_FILTER_ON = 2,     /* as AUTO (kept for symmetry with the other selectors)    */
    MDH_FILTER_AUDIT = 3   /* filter + every pair ALSO evaluated exactly and compared;
                              violations are reported by mdh_rdf_filter_stats (slow,
                              test aid)                                               */
};

/* coordinates outside the cell (same counts for coordinates inside [0, L)) */
enum {
    MDH_WRAP_AUTO = 0,     /* as the reference: MDAnalysis' capped_distance moves both
                              coordinate sets into the cell IN FLOAT32 before taking
                              differences whenever it picks its grid search (both groups
                              >= 10 particles and n1 * n2 >= 1e8 or r_max <= 0.3 * shortest
                              edge), and takes the differences of the coordinates as given
                              when it picks brute force                               */
    MDH_WRAP_NEVER = 1,    /* brute-force semantics for every frame                    */
    MDH_WRAP_ALWAYS = 2    /* grid-search semantics for every frame                    */
};

/* S(q) kernel strategy */
enum {
    MDH_SQ_AUTO = 0,
    MDH_SQ_LATTICE_FP64 = 1,  /* q = n*b: per-axis phase factors, fp64 complex FMA */
    /* 2 is retired (a MUFU sin/cos variant that was never built) and is rejected */
    MDH_SQ_GENERAL_FP64 = 3,  /* arbitrary q: fp64 dot product + fp64 sincos     */
    MDH_SQ_LATTICE_FP32 = 4,  /* q = n*b: the FP64 scheme on the FP32 pipe
                                 (approximate: ~1e-7 relative per term)          */
    MDH_SQ_LATTICE_DMMA = 5   /* q = n*b: per-axis phase factors, the complex rank-N
                                 update on the FP64 matrix unit (mma.m8n8k4.f64);
                                 what MDH_SQ_AUTO picks for lattice wavevectors; falls
                                 back to MDH_SQ_LATTICE_FP64 when the phase-factor
                                 tables do not fit in shared memory                */
};

typedef struct mdh_ctx mdh_ctx;

/* ---- context ----------------------------------------------------------------- */

int mdh_abi_version(void);
const char *mdh_last_error(void);

/* cuda_stream: a cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream), or NULL to
 * let the context create its own non-blocking stream.  NOTE: the default stream of a
 * framework has the handle 0 == NULL; pass cudaStreamLegacy ((cudaStream_t)0x1) or
 * cudaStreamPerThread ((cudaStream_t)0x2) to name it, as the Python layer does -- work on
 * a private stream is not ordered against the framework's events and collectives. */
int mdh_ctx_create(int device, void *cuda_stream, mdh_ctx **out);
int mdh_ctx_destroy(mdh_ctx *ctx);
int mdh_sync(mdh_ctx *ctx);

/* Device-side time (ms, CUDA events on the context's stream) spent in the pair
 * kernels / S(q) kernels by the LAST accumulate call, and launches issued by the
 * context since creation.  Both calls synchronise the stream. */
int mdh_last_kernel_ms(mdh_ctx *ctx, float *rdf_ms, float *sq_ms);
/* Sum of those per-call device times, and the number of accumulate calls they cover,
 * since the previous call with reset != 0 (synchronises the stream). */
int mdh_kernel_time(mdh_ctx *ctx, int reset, double *rdf_ms, int64_t *rdf_calls,
                    double *sq_ms, int64_t *sq_calls);
int mdh_launch_count(mdh_ctx *ctx, int64_t *launches);

/* ---- seam #1: radial histogram ------------------------------------------------- */

/*
 * n1, n2        particles in the two groups; same_group != 0 means pos2 is pos1
 *               (the reference's ag1 is ag2 case: ordered pairs, self pairs
 *               included, exactly as structure.py:93-104 counts them).
 * n_bins        number of histogram bins.
 * thresholds_sq n_bins+1 doubles, strictly increasing: bin k receives a pair iff
 *               thresholds_sq[k] <= d^2 < thresholds_sq[k+1], d^2 being the fp64
 *               squared minimum-image distance.  The host layer derives them from
 *               np.linspace(range) so that this is exactly numpy.histogram of
 *               sqrt(d^2) plus capped_distance's cut-offs (see
 *               mdhelper_b200/analysis/_binning.py).
 * r_lo, r_hi    the histogram range (only seeds the bin-index guess).
 * excl1, excl2  exclusion block sizes: pairs with i/excl1 == j/excl2 are dropped
 *               (structure.py:100-102); 0, 0 disables.
 * drop_axis     -1, or 0/1/2: that coordinate is zeroed before the distance
 *               (structure.py:766-767; the caller passes the widened box edge, or for
 *               mdh_rdf_accumulate_triclinic the cell matrix of the widened dimensions).
 *               Orthorhombic cells: every mode; the cell list then has one cell along the
 *               dropped axis.  Triclinic cells: all pairs for every axis, the cell list
 *               for drop_axis 2 only (see mdh_rdf_accumulate_triclinic).
 * mode, hist    MDH_RDF_* / MDH_HIST_* selectors.
 * Resets the accumulated counts.
 */
int mdh_rdf_configure(mdh_ctx *ctx, int64_t n1, int64_t n2, int same_group, int n_bins,
                      const double *thresholds_sq, double r_lo, double r_hi,
                      int64_t excl1, int64_t excl2, int drop_axis, int mode, int hist);

/* Adds the histograms of n_frames frames to the context's int64 counts.
 * pos2 is ignored when same_group.  box is a HOST pointer, [n_frames][3]. */
int mdh_rdf_accumulate(mdh_ctx *ctx, const float *pos1, int64_t frame_stride1,
                       const float *pos2, int64_t frame_stride2, int location,
                       const float *box, int n_frames);

/*
 * The same for TRICLINIC cells: cell is a HOST pointer, [n_frames][9], the row-major
 * lower-triangular cell matrix (a_x 0 0 / b_x b_y 0 / c_x c_y c_z) as float32 -- what
 * MDAnalysis' triclinic_vectors(ts.dimensions) gives; the reference passes ts.dimensions
 * with its angles to capped_distance (structure.py:93-96).  Coordinates are wrapped into
 * the cell, then every pair takes the shortest of its 27 images (fp64).  The configured
 * mode selects the pair kernel: MDH_RDF_ALLPAIRS evaluates all 27 images of every pair;
 * MDH_RDF_CELLS uses a cell list in fractional coordinates and evaluates, per candidate,
 * the one image that can be in range (same counts; MDH_EINVAL if some frame fits fewer
 * than 3 cells on an axis, see mdh_rdf_triclinic_grid); MDH_RDF_AUTO takes the cell list
 * when every frame fits at least 4 cells per axis and n1*n2 >= 4e6.  drop_axis: the
 * coordinate is zeroed before the wrap (which may move it again on a tilted cell, as in
 * the reference); every axis runs through all pairs.  With drop_axis 2 the cell list is
 * a flat grid of the (a, b) plane (one cell along c, mdh_rdf_cells_grid); it needs
 * c_z >= r_hi + M besides 3 cells per in-plane width (else MDH_EINVAL in MDH_RDF_CELLS,
 * all pairs in MDH_RDF_AUTO, whose rule is otherwise the one above for the two kept
 * widths).  drop_axis 0 or 1: MDH_RDF_CELLS is MDH_EINVAL, MDH_RDF_AUTO takes all pairs.
 * Restated from MDAnalysis' published algorithm and NOT pinned against MDAnalysis (see
 * DESIGN.md).
 */
int mdh_rdf_accumulate_triclinic(mdh_ctx *ctx, const float *pos1, int64_t frame_stride1,
                                 const float *pos2, int64_t frame_stride2, int location,
                                 const float *cell, int n_frames);

/*
 * Cell-list grid of one triclinic frame, as mdh_rdf_accumulate_triclinic would use it;
 * device-free.  cell: the [9] matrix as above; r_hi: sqrt of the last squared threshold;
 * n_max: the larger group size (about 2 particles per cell are kept).  Writes the cells
 * per axis (a, b, c; all 0 when fewer than 3 fit on some axis) and the margin M: every
 * cell's perpendicular width is at least r_hi + M (derivation: DESIGN.md 4.8).
 */
int mdh_rdf_triclinic_grid(const float *cell /* [9] */, double r_hi, int64_t n_max,
                           int32_t *nc /* [3] */, double *margin);

/*
 * Cell-list grid of one frame for any cell and drop_axis (-1, 0, 1, 2), as
 * mdh_rdf_accumulate (diagonal cell) or mdh_rdf_accumulate_triclinic (any other cell)
 * would use it; device-free.  cell, r_hi, n_max as for mdh_rdf_triclinic_grid.  Writes the
 * cells per axis (x, y, z or a, b, c; one along a dropped axis; all 0 when fewer than 3
 * fit on a kept axis) and the margin M: every cell is at least r_hi + M wide on a kept
 * axis (diagonal cells: M = 1e-5 r_hi).  MDH_EINVAL for a triclinic cell with drop_axis 0
 * or 1 (no cell list) and for drop_axis 2 with c_z < r_hi + M.  With drop_axis -1 and a
 * triclinic cell it gives what mdh_rdf_triclinic_grid gives.
 */
int mdh_rdf_cells_grid(const float *cell /* [9] */, double r_hi, int64_t n_max, int drop_axis,
                       int32_t *nc /* [3] */, double *margin);

int mdh_rdf_fetch(mdh_ctx *ctx, int64_t *counts /* [n_bins] host */);
int mdh_rdf_reset(mdh_ctx *ctx);
/* device address of the int64[n_bins] accumulator (for NCCL reductions) */
int mdh_rdf_counts_device(mdh_ctx *ctx, void **dptr);
/* pair evaluations performed so far (what the kernels computed, for rooflines) */
int mdh_rdf_pair_evaluations(mdh_ctx *ctx, int64_t *evals);

/*
 * The all-pairs kernel bins a pair from fp32 arithmetic when a rigorous error bound
 * proves the reference's fp64 distance lies in the same bin, and re-evaluates every
 * other pair with the fp64 arithmetic (rdf_filter.cu).  mode is an MDH_FILTER_*
 * value; it persists across mdh_rdf_configure calls of the context.
 */
int mdh_rdf_set_filter(mdh_ctx *ctx, int mode);
/* MDH_WRAP_* selector; persists across mdh_rdf_configure calls of the context. */
int mdh_rdf_set_prewrap(mdh_ctx *ctx, int mode);
/* stats[0] pairs-of-IPT entries re-evaluated from the deferred lists, stats[1]
 * entries re-evaluated inline (list overflow), stats[2] audit violations (must be
 * 0), stats[3] uncertain pairs seen by the audit, stats[4] frames the filter
 * declined (left to the exact kernel), stats[5] 1 if the current configuration is
 * eligible for the filter.  Since the last configure / reset. */
int mdh_rdf_filter_stats(mdh_ctx *ctx, int64_t *stats /* [6] host */);
/* frames[0] frames the all-pairs filter kernel evaluated with the half-box minimum image
 * (every coordinate difference within 1.5 box lengths), frames[1] frames it evaluated
 * with the rint form.  Since the last configure / reset. */
int mdh_rdf_filter_modes(mdh_ctx *ctx, int64_t *frames /* [2] host */);
/* frames[0] half-box frames the all-pairs filter kernel evaluated without the slot clamp
 * (its block histogram has a word for every slot the frame can reach; a subset of
 * mdh_rdf_filter_modes' frames[0]).  Since the last configure / reset. */
int mdh_rdf_filter_unclamped(mdh_ctx *ctx, int64_t *frames /* [1] host */);

/* ---- seam #2: direct-sum structure factor ------------------------------------ */

/*
 * n_total       particles per frame (all groups, concatenated in group order).
 * n_groups, group_offsets[n_groups+1]
 *               particle ranges of the groups inside a frame.
 * n_q, wavevectors[n_q][3]   fp64 wavevectors.
 * lattice_n[n_q][3], lattice_b[3]
 *               if non-NULL: wavevectors[i][k] == lattice_n[i][k] * lattice_b[k]
 *               (the reference's default reciprocal-lattice grid,
 *               structure.py:1376-1416); enables the MDH_SQ_LATTICE_* kernels.
 * n_pairs, pairs[n_pairs][2]
 *               group index pairs (j, k) per output row: row += |rho_j|^2 if
 *               j == k else 2 Re(rho_j conj(rho_k)) (structure.py:1496-1508);
 *               the pair (-1, -1) means all particles together (mode=None,
 *               structure.py:1491-1494).
 * Resets the accumulator.
 */
int mdh_sq_configure(mdh_ctx *ctx, int64_t n_total, int n_groups,
                     const int64_t *group_offsets, int n_q, const double *wavevectors,
                     const int32_t *lattice_n, const double *lattice_b, int n_pairs,
                     const int32_t *pairs, int mode);

/* Adds sum over frames of the per-frame |rho|^2 terms to the fp64 accumulator. */
int mdh_sq_accumulate(mdh_ctx *ctx, const float *pos, int64_t frame_stride, int location,
                      int n_frames);

/*
 * The same for float64 coordinates (frame_stride in doubles): what the reference sums over
 * when its position buffer is float64 -- centres of mass of residues / segments and
 * unwrapped polymer coordinates (structure.py:1468-1486, polymer.py:1076-1086).  The
 * kernels read every coordinate as float32 + float32 remainder and add the two in fp64
 * (relative error 2^-48), so rounding such positions to float32 (phase error
 * ~ |q||r| 6e-8) is avoided.
 */
int mdh_sq_accumulate_f64(mdh_ctx *ctx, const double *pos, int64_t frame_stride, int location,
                          int n_frames);

int mdh_sq_fetch(mdh_ctx *ctx, double *ssf /* [n_pairs][n_q] host */);
/* The MDH_SQ_* kernel the current configuration runs (after AUTO / fallback). */
int mdh_sq_kernel(mdh_ctx *ctx, int *mode);
/* Tiling of the MDH_SQ_LATTICE_DMMA kernel (zeros for the other kernels): stats[0] warp
 * items, stats[1] (column group, nz tile) pairs -- 64 accumulator slots each, n_q of
 * which are wavevectors --, stats[2] largest number of pairs on one warp scheduler,
 * stats[3] warp schedulers (4 per block of items). */
int mdh_sq_tiling(mdh_ctx *ctx, int64_t *stats /* [4] host */);
/* The same planning without a device or a context (host only; used by the CPU test suite):
 * stats[0..3] as mdh_sq_tiling, stats[4] consumer warps per block, stats[5] dynamic shared
 * memory per block in bytes.  coverage[q] (optional) = how many accumulator slots are
 * mapped to wavevector q -- must be 1 everywhere --, pair_rule_violations (optional) =
 * column pairs that break the bank-conflict rule of the table layout (0 unless the
 * wavevector set has columns without a compatible partner). */
int mdh_sq_plan(int n_q, const int32_t *lattice_n /* [n_q][3] */, int64_t *stats /* [6] */,
                int32_t *coverage /* [n_q] or NULL */, int32_t *pair_rule_violations);
int mdh_sq_reset(mdh_ctx *ctx);
int mdh_sq_accum_device(mdh_ctx *ctx, void **dptr);
/* rho(q) of the LAST frame of the last batch: [n_rho][n_q][2] (re, im), n_rho =
 * n_groups (or 1 for the (-1,-1) pair).  Debug / parity aid for seam #2. */
int mdh_sq_fetch_rho(mdh_ctx *ctx, double *rho);

/* ---- centres of mass (groupings="residues"/"segments") ----------------------------
 *
 * Replaces center_of_mass(group, grouping) (src/mdhelper/algorithm/molecule.py:15-310)
 * as used at structure.py:753-756 / 1485-1486 for entities that are consecutive runs of
 * atoms: entity e covers atoms starts[e] .. starts[e+1]-1 of the group.
 *   out[f][e][k] = (float)(sum_a masses[a] * pos[f][a][k] / sum_a masses[a])   (fp64,
 * atoms in index order).  out_device is a DEVICE buffer with out_frame_stride floats per
 * frame (>= 3 * n_entities; several groups can be written side by side) that can be
 * handed to mdh_rdf_accumulate / mdh_sq_accumulate with MDH_DEVICE.  Slots 0..7 hold one
 * group description each.
 */
int mdh_com_configure(mdh_ctx *ctx, int slot, int64_t n_atoms, int64_t n_entities,
                      const int64_t *starts /* [n_entities+1] host */,
                      const double *masses /* [n_atoms] host */);
int mdh_com_reduce(mdh_ctx *ctx, int slot, const float *pos, int64_t frame_stride,
                   int location, int n_frames, float *out_device, int64_t out_frame_stride);
/* The same without the final rounding to float32 (out_frame_stride in doubles): input of
 * mdh_sq_accumulate_f64. */
int mdh_com_reduce_f64(mdh_ctx *ctx, int slot, const float *pos, int64_t frame_stride,
                       int location, int n_frames, double *out_device,
                       int64_t out_frame_stride);

/*
 * Single-chain structure factor (SingleChainStructureFactor._single_frame,
 * src/mdhelper/analysis/polymer.py:1076-1099): after mdh_sq_configure with lattice
 * wavevectors, one group and the pair (-1, -1), declare the particles to be n_chains
 * consecutive chains of n_monomers.  mdh_sq_accumulate then adds, per frame,
 *   ssf[0][q] += sum over chains | sum over the chain's monomers exp(i q . r) |^2
 * and mdh_sq_fetch returns that sum (normalise by n_chains * n_monomers * n_frames).
 */
int mdh_sq_configure_chains(mdh_ctx *ctx, int64_t n_chains, int64_t n_monomers);

/* ---- intermediate scattering function F(q, t), F_s(q, t) ------------------------
 *
 * Replaces the per-frame work of IntermediateScatteringFunction._single_frame
 * (src/mdhelper/analysis/structure.py:1959-2085), which calls seam #2 once per frame
 * for rho(q, t) and, with incoherent=True, once per (frame, time lag) on the
 * displacements r(t) - r(t - lag) (:1991-1996).
 *
 * Call mdh_sq_configure first (wavevectors, groups, pairs), then mdh_isf_configure;
 * frames must be passed in time order.  n_lags time lags (0 .. n_lags-1); max_frames
 * is the total number of frames that will be passed (sizes the rho(q, t) store).
 *   cisf[lag][pair][q] = sum over t >= lag of Re(rho_j(t-lag) conj(rho_k(t)))
 *                        (+ the j <-> k term when j != k)
 *   iisf[lag][row][q]  = sum over t >= lag of Re sum_particles exp(i q.(r(t) - r(t-lag))),
 *                        row = group (or 0 for the (-1, -1) pair)
 * Un-normalised sums, as the reference accumulates them before _conclude.
 */
int mdh_isf_configure(mdh_ctx *ctx, int n_lags, int incoherent, int64_t max_frames);
int mdh_isf_accumulate(mdh_ctx *ctx, const float *pos, int64_t frame_stride, int location,
                       int n_frames);
/* float64 coordinates (centres of mass; structure.py:1927-1957 keeps them in a float64
 * buffer): positions and displacements are formed in fp64 and reach the kernels as
 * float32 + float32 remainder, as in mdh_sq_accumulate_f64.  One run is all float32 or
 * all float64 (MDH_ESTATE otherwise). */
int mdh_isf_accumulate_f64(mdh_ctx *ctx, const double *pos, int64_t frame_stride,
                           int location, int n_frames);
/* iisf may be NULL.  Synchronises. */
int mdh_isf_fetch(mdh_ctx *ctx, double *cisf /* [n_lags][n_pairs][n_q] */,
                  double *iisf /* [n_lags][n_rho][n_q] or NULL */);

/*
 * How a host batch is cut into pieces (copy of piece k+1 beside the kernels of piece k):
 * diagnostic view of the planner behind mdh_rdf_accumulate / mdh_sq_accumulate with
 * MDH_HOST, no device needed.  copy_over_kernel = measured copy time / kernel time per
 * frame (0: unknown).  Writes at most cap piece lengths (frames) and their number.
 */
int mdh_stage_plan(int n_frames, double bytes_per_frame, double copy_over_kernel,
                   int32_t *pieces, int cap, int32_t *n_pieces);

#ifdef __cplusplus
}
#endif
#endif /* MDH_B200_H */
