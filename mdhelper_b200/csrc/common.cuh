// common.cuh -- shared declarations of libmdh_b200.so (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/mdh_b200.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libmdh_b200 is written for sm_100a (B200) only"
#endif

void mdh_set_error(const char *fmt, ...);
// MDH_TRACE=1: host-side progress on stderr (where a call blocks)
bool mdh_trace_on();
#define MDH_TRACE(...)                                                          \
    do {                                                                        \
        if (mdh_trace_on()) { fprintf(stderr, "[mdh] " __VA_ARGS__); fputc('\n', stderr); } \
    } while (0)

#define MDH_CUDA(call)                                                          \
    do {                                                                        \
        cudaError_t e_ = (call);                                                \
        if (e_ != cudaSuccess) {                                                \
            mdh_set_error("%s failed at %s:%d: %s", #call, __FILE__, __LINE__,  \
                          cudaGetErrorString(e_));                              \
            return MDH_ECUDA;                                                   \
        }                                                                       \
    } while (0)

#define MDH_REQUIRE(cond, code, ...)                                            \
    do {                                                                        \
        if (!(cond)) {                                                          \
            mdh_set_error(__VA_ARGS__);                                         \
            return (code);                                                      \
        }                                                                       \
    } while (0)

// Device buffer that only ever grows; owned by the context (freed with it: a buffer
// added to a state struct cannot be forgotten in mdh_ctx_destroy).
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    int reserve(size_t bytes);
    void release();
    // take over another buffer's memory (this one must have been released)
    void adopt(DevBuf &o) { release(); p = o.p; cap = o.cap; o.p = nullptr; o.cap = 0; }
    template <typename T> T *as() const { return reinterpret_cast<T *>(p); }
};

struct FrameBox {          // per frame, device side
    double box[3];         // (double)box_f32
    double inv[3];         // (double)(float)(1.0 / (double)box_f32)
    int prewrap;           // coordinates are first moved into the cell in float32 (what the
    int pad;               // reference's grid search does, see rdf_device.cuh::ortho_pbc_f32)
};

// fp32 filter, per frame (built on the device by rdf_filter_prepare_kernel)
struct FrameFilter {
    float nbox[3];         // -box_k
    float inv[3];          // (float)(1.0 / box_k), the reference's float32 inverse box
    float offm;            // 1.5 * 2^(23-k) + off + m * 2^-k: the bin coordinate is
                           // shifted up by the window half-width m (units of 2^-k), so
                           // the uncertainty window is [0, 2m] in its fraction bits
    unsigned wlim;         // pair is uncertain iff (bits & (2^k - 1)) < wlim = 2m + 1;
                           // 0 = frame not eligible (the exact kernel handles it)
    float nhalf[3];        // -box_k / 2
    int halfbox;           // 1: the all-pairs kernel takes the half-box minimum image
                           // (every |df_k| <= 1.5 box_k; offm / wlim are from its bound)
    int unclamped;         // 1: (half-box frames only) every slot the fp32 arithmetic can
                           // produce is a word of the all-pairs kernel's histogram, so its
                           // hot loop needs no clamp (rdf_device.cuh::filter_reach)
};

struct FilterConst {       // per configuration (host)
    float scale;           // (float)(n_bins / (r_hi - r_lo))
    double offbase;        // 1.5 * 2^(23-k) + off, off a multiple of 2^-k
    unsigned cbits;        // bits of the float (1.5 * 2^(23-k)): slot 0 ("below range")
    unsigned span;         // (n_bins + 2) << k: slots 0 .. n_bins + 1
    int k;                 // fraction bits of the fixed-point bin coordinate
    int sb;                // log2(sub-bins per bin) of the cell-pair kernel's per-warp histograms
    int cb;                // all-pairs filter kernel: log2(columns per slot) of the block's histogram
    int lg;                // 2^lg >= hslots
    int lower;             // the bin coordinate can be negative (r_lo > 0 and lo == 0)
    // all-pairs filter kernel (rdf_filter.cu::filter_plan, per batch of frames); the
    // cell-list kernels keep lo = 0, hslots = n_bins + 2
    int lo;                // slot = bin + 1 + lo: the offset is shifted by lo whole slots
                           // so that the coordinate of a distance >= 0 is never negative
    int hslots;            // slots of the block histogram; slots outside
                           // [lo + 1, lo + n_bins] are scratch words, never read
    int unclamped;         // hslots covers every slot a half-box frame of the batch
                           // can reach (FrameFilter::unclamped may be set)
};

struct RdfState {
    bool configured = false;
    int64_t n1 = 0, n2 = 0;
    int same = 0, n_bins = 0, drop_axis = -1, mode = 0, hist = 0;
    int64_t excl1 = 0, excl2 = 0;
    double r_lo = 0, r_hi = 0, thr_hi = 0;
    DevBuf thr;            // double[n_bins + 2]: thresholds, then +inf
    DevBuf counts;         // unsigned long long[n_bins]
    DevBuf raw1[2], raw2[2];  // float[F][n][3] staging for host input, one per stager slot
    DevBuf pk1, pk2;       // float4[F][npad]
    DevBuf boxes;          // FrameBox[F]
    DevBuf cell[10];       // cell-list scratch, layout in rdf_cells.cu
    double cells_ws_mb = 192.0;   // working set of one group of frames (sort + pair kernel)
    int cells_chunk = 4;         // cells per work item of the cell-pair kernel
    int cells_ipt = 4;           // particles per lane of the cell-pair kernel (2 or 4)
    bool cells_debug = false;    // per-stage device times on stderr (MDH_TUNE cdbg=1)
    bool evals_dev_init = false;
    std::vector<FrameBox> h_boxes;
    FrameBox *h_boxes_pinned = nullptr;   // staging for the async box upload
    size_t h_boxes_cap = 0;
    cudaEvent_t ev_boxes = nullptr;       // previous box upload has been consumed
    int64_t evals = 0;     // all-pairs evaluations (host-side count)
    int ipt = 2;           // i-particles per thread of the all-pairs kernel
    bool fast_bins = false;  // branch-free bin guess certified for this configuration
    // fp32 filter in front of the exact arithmetic (rdf_filter.cu)
    int prewrap_mode = MDH_WRAP_AUTO;    // survives configure
    int filter_mode = MDH_FILTER_AUTO;   // survives configure
    bool filter_ok = false;  // this configuration is eligible
    int filter_occ = 2;      // blocks per SM the filter kernel is compiled for (2 or 3)
    FilterConst fc;
    FilterConst fca;       // the all-pairs filter kernel's layout for the current batch
    DevBuf ext1, ext2;     // unsigned[F][6]: coordinate extents of each frame (keys)
    DevBuf filt;           // FrameFilter[F]
    DevBuf fstats;         // unsigned long long[8], see PairParams::fstats
};

struct SqWorkItem {        // one thread's tile of the lattice kernels: two (nx, ny)
    int nx[2], ny[2];      // columns x one segment of kSqTN consecutive nz
    int nz0;
    int len[2];            // wavevectors wanted from each column (0..kSqTN)
    int pad;
};
constexpr int kSqTM = 2;   // columns per thread
constexpr int kSqTN = 8;   // nz values per thread

// Two event pairs around the copy and the kernels of the last piece of a host call; the
// next call reads them (if they have completed) to learn the ratio above.
struct RateProbe {
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    bool pending = false;
    double copy_over_kernel = 0.0;
    RateProbe() = default;
    RateProbe(const RateProbe &) = delete;
    RateProbe &operator=(const RateProbe &) = delete;
    ~RateProbe() { for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e); }
    int ensure();
    void learn();               // non-blocking
};

struct SqState {
    bool configured = false;
    int64_t n_total = 0;
    int n_groups = 0, n_q = 0, n_pairs = 0, mode = 0, n_rho = 0;
    bool lattice = false;
    int nmax[3] = {0, 0, 0};
    double b[3] = {0, 0, 0};
    int n_items = 0, block = 256;
    std::vector<int64_t> group_offsets;
    std::vector<int32_t> pairs;
    DevBuf qv;             // double[n_q][3]
    DevBuf items;          // SqWorkItem[n_items]
    DevBuf qidx;           // int[n_items][kSqTM][kSqTN]
    // DMMA lattice kernel (MDH_SQ_LATTICE_DMMA): one SqMmaItem per consumer warp
    bool mma = false;      // built and selected for this configuration
    int mma_items = 0, mma_warps = 0;   // items (padded to whole blocks), warps per block
    int mma_stats[4] = {0, 0, 0, 0};    // items, (group, tile) pairs, max scheduler load, schedulers
    DevBuf mitems;         // SqMmaItem[mma_items]
    DevBuf mqidx;          // int[mma_items][groups][tiles][8][8]
    DevBuf d_pairs;        // int[n_pairs][2]
    DevBuf chunks;         // int4[n_chunks]: {start, end, rho_row, 0}
    int n_chunks = 0, chunk_len = 0;
    DevBuf raw[2];         // float[F][n][3] (or double) staging for host input, one per stager slot
    RateProbe probe;       // copy vs kernel rate of the last host call (piece planning)
    DevBuf split;          // float[2F][n][3]: float64 input as float32 + negated remainder
    DevBuf split_vmap;     // int4[F]: {f, F + f, 0, 0}
    DevBuf tab;            // phase-factor tables of one group of frames
    DevBuf rho;            // double[F][n_rho][n_q][2]
    DevBuf ssf;            // double[n_pairs][n_q]
    int rho_frames = 0;    // frames held in rho from the last batch
    // single-chain mode (mdh_sq_configure_chains): chunks are chains, ssf[0][q]
    // accumulates sum over chains of |rho_chain(q)|^2
    int64_t n_chains = 0, n_monomers = 0;
};

constexpr int kComSlots = 8;
struct ComState {           // centres of mass of consecutive atom runs (com.cu)
    bool configured = false;
    int64_t n_atoms = 0, n_entities = 0;
    DevBuf starts;         // int64[n_entities + 1]
    DevBuf masses;         // double[n_atoms]
    DevBuf raw;            // float[F][n_atoms][3] staging for host input
};

struct IsfState {           // intermediate scattering function on top of SqState
    bool on = false;
    int n_lags = 0;
    bool incoherent = false;
    bool f64 = false;      // the window holds doubles (mdh_isf_accumulate_f64)
    int64_t max_frames = 0, n_done = 0;
    DevBuf rho_all;        // double2[max_frames][n_rho][n_q]: rho(q, t) of every frame
    DevBuf window[2];      // float (or double) [kept + batch][n_total][3], ping-pong
    int window_frames = 0, which = 0;
    DevBuf vmap;           // int4 per virtual frame: {frame, reference frame, lag, 0}
    DevBuf cisf;           // double[n_lags][n_pairs][n_q]
    DevBuf iisf;           // double[n_lags][n_rho][n_q]
};

// CUDA-event stopwatch around the hot kernels of every accumulate call, on the
// context's stream.  Pairs are recorded without synchronising; collect() sums them.
struct KernelTimer {
    std::vector<cudaEvent_t> ev;   // ev[2i] start, ev[2i+1] stop
    size_t used = 0;               // pairs recorded since the last reset / fold
    double folded_ms = 0;          // pairs folded away because the ring was full
    int64_t folded_n = 0;
    int begin(cudaStream_t s);
    int end(cudaStream_t s);
    int last(cudaStream_t s, float *ms);                       // synchronises
    int collect(cudaStream_t s, bool reset, double *ms, int64_t *n);   // synchronises
    void destroy();
};

// Host -> device staging of coordinate batches on a separate copy stream, two slots:
// the copy of piece k + 1 runs while the kernels of piece k do (accumulate calls with
// host pointers are cut into pieces for exactly this).
struct HostStager {
    cudaStream_t copy = nullptr;
    cudaEvent_t ready[2] = {nullptr, nullptr};   // slot filled (recorded on the copy stream)
    cudaEvent_t done[2] = {nullptr, nullptr};    // slot consumed (recorded on the compute stream)
    bool used[2] = {false, false};
    int turn = 0;
    int init();
    // next slot; the copy stream waits until the kernels that read it last are done
    int acquire(int *slot);
    // compute stream waits for the copies queued into `slot` since acquire()
    int publish(cudaStream_t compute, int slot);
    // to be called after the kernels reading `slot` have been launched
    int retire(cudaStream_t compute, int slot);
    void destroy();
};

// Host batches are cut into pieces so that the copy of one piece (copy stream) overlaps the
// kernels of the previous one.  The pieces grow geometrically: the first copy -- the only
// one nothing can hide -- is short (~2 MB), later ones are long enough (up to ~32 MB) for
// their kernels to run at full efficiency.
// copy_over_kernel: measured (copy time per frame) / (kernel time per frame) of an earlier
// call with the same configuration, 0 = unknown.
std::vector<int> mdh_plan_pieces(int n_frames, double bytes_per_frame,
                                 double copy_over_kernel = 0.0);


// Frame-strided copy: one contiguous transfer when the frames are adjacent on both sides
// (a 2-D copy of rows that happen to be contiguous is split by the driver), else a 2-D copy.
inline cudaError_t mdh_copy_frames(void *dst, size_t dpitch, const void *src, size_t spitch,
                                   size_t width, size_t n_frames, cudaMemcpyKind kind,
                                   cudaStream_t stream)
{
    if (dpitch == width && spitch == width)
        return cudaMemcpyAsync(dst, src, width * n_frames, kind, stream);
    return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, n_frames, kind, stream);
}

struct mdh_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    HostStager stager;
    int sm_count = 148;
    int64_t launches = 0;
    KernelTimer t_rdf, t_sq;
    RdfState rdf;
    SqState sq;
    IsfState isf;
    ComState com[kComSlots];
};

// rdf.cu
int rdf_configure_impl(mdh_ctx *c, int64_t n1, int64_t n2, int same, int n_bins,
                       const double *thr, double r_lo, double r_hi, int64_t e1, int64_t e2,
                       int drop_axis, int mode, int hist);
int rdf_accumulate_impl(mdh_ctx *c, const float *pos1, int64_t s1, const float *pos2,
                        int64_t s2, int location, const float *box, int n_frames);
// rdf_tri.cu
int rdf_accumulate_triclinic_impl(mdh_ctx *c, const float *pos1, int64_t s1, const float *pos2,
                                  int64_t s2, int location, const float *box9, int n_frames);
int rdf_triclinic_grid_impl(const float *cell9, double r_hi, int64_t n_max, int32_t *nc,
                            double *margin);
int rdf_cells_grid_impl(const float *cell9, double r_hi, int64_t n_max, int drop_axis,
                        int32_t *nc, double *margin);
// rdf_filter.cu
int rdf_filter_sqrt_error(mdh_ctx *c, double *err);
bool rdf_filter_configure(RdfState &R, const double *thr, double sqrt_err);
int rdf_filter_prepare(mdh_ctx *c, int f0, int n_frames, double sqrt_err);
// sq.cu
int sq_configure_impl(mdh_ctx *c, int64_t n_total, int n_groups, const int64_t *goff,
                      int n_q, const double *wv, const int32_t *lat_n, const double *lat_b,
                      int n_pairs, const int32_t *pairs, int mode);
int sq_accumulate_f64_impl(mdh_ctx *c, const double *pos, int64_t stride, int location,
                           int n_frames);
int sq_accumulate_impl(mdh_ctx *c, const float *pos, int64_t stride, int location,
                       int n_frames);
// com.cu
int com_configure_impl(mdh_ctx *c, int slot, int64_t n_atoms, int64_t n_entities,
                       const int64_t *starts, const double *masses);
int com_reduce_impl(mdh_ctx *c, int slot, const float *pos, int64_t stride, int location,
                    int n_frames, float *out_device, int64_t out_stride);
int com_reduce_f64_impl(mdh_ctx *c, int slot, const float *pos, int64_t stride, int location,
                        int n_frames, double *out_device, int64_t out_stride);
int sq_configure_chains_impl(mdh_ctx *c, int64_t n_chains, int64_t n_monomers);
int sq_plan_impl(int n_q, const int32_t *lat_n, int64_t *stats, int32_t *coverage,
                 int32_t *pair_rule_violations);
int isf_configure_impl(mdh_ctx *c, int n_lags, int incoherent, int64_t max_frames);
int isf_accumulate_f64_impl(mdh_ctx *c, const double *pos, int64_t stride, int location,
                            int n_frames);
int isf_accumulate_impl(mdh_ctx *c, const float *pos, int64_t stride, int location,
                        int n_frames);
int isf_fetch_impl(mdh_ctx *c, double *cisf, double *iisf);
