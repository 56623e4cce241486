// api.cu -- the C ABI declared in include/mdh_b200.h (context, fetch, errors).

#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>

#include <new>

#include "common.cuh"

static thread_local char g_err[1024] = "";

bool mdh_trace_on()
{
    static int on = -1;
    if (on < 0) { const char *e = getenv("MDH_TRACE"); on = (e && *e && *e != '0') ? 1 : 0; }
    return on == 1;
}

void mdh_set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int DevBuf::reserve(size_t bytes)
{
    if (bytes <= cap) return MDH_OK;
    if (p) {
        // the buffer may still be in use by work queued on the context's stream
        cudaError_t e = cudaDeviceSynchronize();
        if (e == cudaSuccess) e = cudaFree(p);
        if (e != cudaSuccess) {
            mdh_set_error("cudaFree failed: %s", cudaGetErrorString(e));
            return MDH_ECUDA;
        }
        p = nullptr;
        cap = 0;
    }
    const size_t want = bytes + bytes / 4 + 256;
    cudaError_t e = cudaMalloc(&p, want);
    if (e != cudaSuccess) {
        p = nullptr;
        mdh_set_error("cudaMalloc(%zu bytes) failed: %s", want, cudaGetErrorString(e));
        cudaGetLastError();
        return MDH_ENOMEM;
    }
    cap = want;
    return MDH_OK;
}

void DevBuf::release()
{
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
}

std::vector<int> mdh_plan_pieces(int n_frames, double bytes_per_frame, double copy_over_kernel)
{
    std::vector<int> out;
    const double bpf = std::max(1.0, bytes_per_frame);
    double want = 2e6;
    int done = 0;
    while (done < n_frames) {
        int nf = (int)std::max(1.0, std::floor(want / bpf));
        const int left = n_frames - done;
        if (left <= nf) {
            nf = left;
        } else if (left < nf + nf / 2) {
            // A short remainder joins the last piece (every launch costs the kernels a
            // partial round of work units) -- unless the measured rates say that the
            // copy of the merged piece would outlast the kernels of the piece before it
            // (two staging slots: a copy runs beside the previous piece's kernels only).
            // Then the remainder is cut in halves.  Seen with eight ranks on one host:
            // some GPUs get ~25 GB/s, and a merged tail of 3x its predecessor left cfg4's
            // S(q) kernels waiting 0.7 ms of a 7 ms pass.
            const int prev = out.empty() ? 0 : out.back();
            const bool fits = copy_over_kernel <= 0.0 ||
                              (double)left * copy_over_kernel <= 0.9 * (double)prev;
            nf = fits ? left : (left + 1) / 2;
        }
        out.push_back(nf);
        done += nf;
        want = std::min(32e6, want * 2.0);
    }
    return out;
}

int RateProbe::ensure()
{
    for (cudaEvent_t &e : ev)
        if (!e) MDH_CUDA(cudaEventCreate(&e));
    return MDH_OK;
}

void RateProbe::learn()
{
    if (!pending) return;
    if (cudaEventQuery(ev[1]) != cudaSuccess || cudaEventQuery(ev[3]) != cudaSuccess) {
        cudaGetLastError();                     // not ready: keep the old estimate
        return;
    }
    float tc = 0.f, tk = 0.f;
    if (cudaEventElapsedTime(&tc, ev[0], ev[1]) == cudaSuccess &&
        cudaEventElapsedTime(&tk, ev[2], ev[3]) == cudaSuccess && tk > 0.f)
        copy_over_kernel = (double)tc / (double)tk;
    else
        cudaGetLastError();
    pending = false;
}

int KernelTimer::begin(cudaStream_t s)
{
    if (used == 512) {                       // ring full: fold what has been recorded
        double ms; int64_t n;
        if (int rc = collect(s, false, &ms, &n)) return rc;
        folded_ms = ms; folded_n = n; used = 0;
    }
    while (ev.size() < 2 * (used + 1)) {
        cudaEvent_t e;
        MDH_CUDA(cudaEventCreate(&e));
        ev.push_back(e);
    }
    MDH_CUDA(cudaEventRecord(ev[2 * used], s));
    return MDH_OK;
}

int KernelTimer::end(cudaStream_t s)
{
    MDH_CUDA(cudaEventRecord(ev[2 * used + 1], s));
    ++used;
    return MDH_OK;
}

int KernelTimer::last(cudaStream_t s, float *ms)
{
    *ms = 0.f;
    if (used == 0) return MDH_OK;
    MDH_CUDA(cudaStreamSynchronize(s));
    MDH_CUDA(cudaEventElapsedTime(ms, ev[2 * used - 2], ev[2 * used - 1]));
    return MDH_OK;
}

int KernelTimer::collect(cudaStream_t s, bool reset, double *ms, int64_t *n)
{
    MDH_CUDA(cudaStreamSynchronize(s));
    double tot = folded_ms;
    for (size_t i = 0; i < used; ++i) {
        float t;
        MDH_CUDA(cudaEventElapsedTime(&t, ev[2 * i], ev[2 * i + 1]));
        tot += t;
    }
    *ms = tot;
    *n = folded_n + (int64_t)used;
    if (reset) { used = 0; folded_ms = 0; folded_n = 0; }
    return MDH_OK;
}

int HostStager::init()
{
    if (copy) return MDH_OK;
    MDH_CUDA(cudaStreamCreateWithFlags(&copy, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
        MDH_CUDA(cudaEventCreateWithFlags(&ready[i], cudaEventDisableTiming));
        MDH_CUDA(cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming));
    }
    return MDH_OK;
}

int HostStager::acquire(int *slot)
{
    if (int rc = init()) return rc;
    *slot = turn++ & 1;
    if (used[*slot]) MDH_CUDA(cudaStreamWaitEvent(copy, done[*slot], 0));
    return MDH_OK;
}

int HostStager::publish(cudaStream_t compute, int slot)
{
    MDH_CUDA(cudaEventRecord(ready[slot], copy));
    MDH_CUDA(cudaStreamWaitEvent(compute, ready[slot], 0));
    return MDH_OK;
}

int HostStager::retire(cudaStream_t compute, int slot)
{
    MDH_CUDA(cudaEventRecord(done[slot], compute));
    used[slot] = true;
    return MDH_OK;
}

void HostStager::destroy()
{
    for (int i = 0; i < 2; ++i) {
        if (ready[i]) cudaEventDestroy(ready[i]);
        if (done[i]) cudaEventDestroy(done[i]);
        ready[i] = done[i] = nullptr;
        used[i] = false;
    }
    if (copy) cudaStreamDestroy(copy);
    copy = nullptr;
}

void KernelTimer::destroy()
{
    for (cudaEvent_t e : ev) cudaEventDestroy(e);
    ev.clear();
    used = 0;
}

#define CTX_GUARD(ctx)                                                         \
    do {                                                                       \
        MDH_REQUIRE((ctx) != nullptr, MDH_EINVAL, "context is NULL");          \
        MDH_CUDA(cudaSetDevice((ctx)->device));                                \
    } while (0)

extern "C" {

int mdh_abi_version(void) { return MDH_ABI_VERSION; }

const char *mdh_last_error(void) { return g_err; }

int mdh_ctx_create(int device, void *cuda_stream, mdh_ctx **out)
{
    MDH_REQUIRE(out != nullptr, MDH_EINVAL, "out is NULL");
    *out = nullptr;
    int n_dev = 0;
    MDH_CUDA(cudaGetDeviceCount(&n_dev));
    MDH_REQUIRE(device >= 0 && device < n_dev, MDH_EINVAL, "device %d out of range (%d visible)",
                device, n_dev);
    MDH_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    MDH_CUDA(cudaGetDeviceProperties(&prop, device));
    MDH_REQUIRE(prop.major == 10, MDH_EINVAL,
                "libmdh_b200 contains sm_100a code only; device %d is sm_%d%d", device,
                prop.major, prop.minor);
    mdh_ctx *c = new (std::nothrow) mdh_ctx();
    MDH_REQUIRE(c != nullptr, MDH_ENOMEM, "out of host memory");
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    if (cuda_stream) {
        c->stream = reinterpret_cast<cudaStream_t>(cuda_stream);
    } else {
        cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
        if (e != cudaSuccess) {
            delete c;
            mdh_set_error("cudaStreamCreate failed: %s", cudaGetErrorString(e));
            return MDH_ECUDA;
        }
        c->own_stream = true;
    }
    *out = c;
    return MDH_OK;
}

int mdh_ctx_destroy(mdh_ctx *c)
{
    if (!c) return MDH_OK;
    cudaSetDevice(c->device);
    cudaStreamSynchronize(c->stream);
    RdfState &R = c->rdf;
    if (c->stager.copy) cudaStreamSynchronize(c->stager.copy);
    c->stager.destroy();
    if (R.h_boxes_pinned) cudaFreeHost(R.h_boxes_pinned);
    if (R.ev_boxes) cudaEventDestroy(R.ev_boxes);
    // every DevBuf of the state structs releases its memory in its destructor (delete c)
    c->t_rdf.destroy();
    c->t_sq.destroy();
    if (c->own_stream) cudaStreamDestroy(c->stream);
    delete c;
    return MDH_OK;
}

int mdh_sync(mdh_ctx *c)
{
    CTX_GUARD(c);
    MDH_CUDA(cudaStreamSynchronize(c->stream));
    return MDH_OK;
}

int mdh_last_kernel_ms(mdh_ctx *c, float *rdf_ms, float *sq_ms)
{
    CTX_GUARD(c);
    if (rdf_ms) if (int rc = c->t_rdf.last(c->stream, rdf_ms)) return rc;
    if (sq_ms) if (int rc = c->t_sq.last(c->stream, sq_ms)) return rc;
    return MDH_OK;
}

int mdh_kernel_time(mdh_ctx *c, int reset, double *rdf_ms, int64_t *rdf_calls, double *sq_ms,
                    int64_t *sq_calls)
{
    CTX_GUARD(c);
    MDH_REQUIRE(rdf_ms && rdf_calls && sq_ms && sq_calls, MDH_EINVAL, "NULL argument");
    if (int rc = c->t_rdf.collect(c->stream, reset != 0, rdf_ms, rdf_calls)) return rc;
    return c->t_sq.collect(c->stream, reset != 0, sq_ms, sq_calls);
}

int mdh_launch_count(mdh_ctx *c, int64_t *launches)
{
    MDH_REQUIRE(c && launches, MDH_EINVAL, "NULL argument");
    *launches = c->launches;
    return MDH_OK;
}

/* ---- seam #1 ---- */

int mdh_rdf_configure(mdh_ctx *c, int64_t n1, int64_t n2, int same_group, int n_bins,
                      const double *thresholds_sq, double r_lo, double r_hi, int64_t excl1,
                      int64_t excl2, int drop_axis, int mode, int hist)
{
    CTX_GUARD(c);
    return rdf_configure_impl(c, n1, n2, same_group, n_bins, thresholds_sq, r_lo, r_hi, excl1,
                              excl2, drop_axis, mode, hist);
}

int mdh_rdf_accumulate(mdh_ctx *c, const float *pos1, int64_t frame_stride1, const float *pos2,
                       int64_t frame_stride2, int location, const float *box, int n_frames)
{
    CTX_GUARD(c);
    return rdf_accumulate_impl(c, pos1, frame_stride1, pos2, frame_stride2, location, box,
                               n_frames);
}

int mdh_rdf_accumulate_triclinic(mdh_ctx *c, const float *pos1, int64_t frame_stride1,
                                 const float *pos2, int64_t frame_stride2, int location,
                                 const float *cell, int n_frames)
{
    CTX_GUARD(c);
    return rdf_accumulate_triclinic_impl(c, pos1, frame_stride1, pos2, frame_stride2, location,
                                         cell, n_frames);
}

int mdh_rdf_triclinic_grid(const float *cell, double r_hi, int64_t n_max, int32_t *nc,
                           double *margin)
{
    return rdf_triclinic_grid_impl(cell, r_hi, n_max, nc, margin);
}

int mdh_rdf_cells_grid(const float *cell, double r_hi, int64_t n_max, int drop_axis,
                       int32_t *nc, double *margin)
{
    return rdf_cells_grid_impl(cell, r_hi, n_max, drop_axis, nc, margin);
}

int mdh_rdf_fetch(mdh_ctx *c, int64_t *counts)
{
    CTX_GUARD(c);
    MDH_REQUIRE(c->rdf.configured, MDH_ESTATE, "rdf: fetch before configure");
    MDH_REQUIRE(counts != nullptr, MDH_EINVAL, "rdf: counts is NULL");
    MDH_CUDA(cudaMemcpyAsync(counts, c->rdf.counts.p, sizeof(int64_t) * c->rdf.n_bins,
                             cudaMemcpyDeviceToHost, c->stream));
    MDH_CUDA(cudaStreamSynchronize(c->stream));
    return MDH_OK;
}

int mdh_rdf_reset(mdh_ctx *c)
{
    CTX_GUARD(c);
    MDH_REQUIRE(c->rdf.configured, MDH_ESTATE, "rdf: reset before configure");
    MDH_CUDA(cudaMemsetAsync(c->rdf.counts.p, 0, sizeof(int64_t) * c->rdf.n_bins, c->stream));
    if (c->rdf.evals_dev_init)
        MDH_CUDA(cudaMemsetAsync(c->rdf.cell[9].p, 0, sizeof(unsigned long long), c->stream));
    if (c->rdf.fstats.p)
        MDH_CUDA(cudaMemsetAsync(c->rdf.fstats.p, 0, sizeof(unsigned long long) * 8, c->stream));
    c->rdf.evals = 0;
    return MDH_OK;
}

int mdh_rdf_counts_device(mdh_ctx *c, void **dptr)
{
    MDH_REQUIRE(c && dptr, MDH_EINVAL, "NULL argument");
    MDH_REQUIRE(c->rdf.configured, MDH_ESTATE, "rdf: not configured");
    *dptr = c->rdf.counts.p;
    return MDH_OK;
}

int mdh_rdf_pair_evaluations(mdh_ctx *c, int64_t *evals)
{
    CTX_GUARD(c);
    MDH_REQUIRE(evals != nullptr, MDH_EINVAL, "evals is NULL");
    unsigned long long dev = 0;
    if (c->rdf.evals_dev_init) {
        MDH_CUDA(cudaMemcpyAsync(&dev, c->rdf.cell[9].p, sizeof(dev), cudaMemcpyDeviceToHost,
                                 c->stream));
        MDH_CUDA(cudaStreamSynchronize(c->stream));
    }
    *evals = c->rdf.evals + (int64_t)dev;
    return MDH_OK;
}

int mdh_rdf_set_filter(mdh_ctx *c, int mode)
{
    MDH_REQUIRE(c != nullptr, MDH_EINVAL, "context is NULL");
    MDH_REQUIRE(mode >= MDH_FILTER_AUTO && mode <= MDH_FILTER_AUDIT, MDH_EINVAL,
                "rdf: invalid filter mode");
    c->rdf.filter_mode = mode;
    return MDH_OK;
}

int mdh_rdf_set_prewrap(mdh_ctx *c, int mode)
{
    MDH_REQUIRE(c != nullptr, MDH_EINVAL, "context is NULL");
    MDH_REQUIRE(mode >= MDH_WRAP_AUTO && mode <= MDH_WRAP_ALWAYS, MDH_EINVAL,
                "rdf: invalid wrap mode");
    c->rdf.prewrap_mode = mode;
    return MDH_OK;
}

int mdh_rdf_filter_stats(mdh_ctx *c, int64_t *stats)
{
    CTX_GUARD(c);
    MDH_REQUIRE(stats != nullptr, MDH_EINVAL, "stats is NULL");
    MDH_REQUIRE(c->rdf.configured, MDH_ESTATE, "rdf: not configured");
    unsigned long long h[8] = {0};
    MDH_CUDA(cudaMemcpyAsync(h, c->rdf.fstats.p, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    MDH_CUDA(cudaStreamSynchronize(c->stream));
    for (int i = 0; i < 5; ++i) stats[i] = (int64_t)h[i];
    stats[5] = c->rdf.filter_ok ? 1 : 0;
    return MDH_OK;
}

int mdh_rdf_filter_modes(mdh_ctx *c, int64_t *frames)
{
    CTX_GUARD(c);
    MDH_REQUIRE(frames != nullptr, MDH_EINVAL, "frames is NULL");
    MDH_REQUIRE(c->rdf.configured, MDH_ESTATE, "rdf: not configured");
    unsigned long long h[8] = {0};
    MDH_CUDA(cudaMemcpyAsync(h, c->rdf.fstats.p, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    MDH_CUDA(cudaStreamSynchronize(c->stream));
    frames[0] = (int64_t)h[5];
    frames[1] = (int64_t)h[6];
    return MDH_OK;
}

int mdh_rdf_filter_unclamped(mdh_ctx *c, int64_t *frames)
{
    CTX_GUARD(c);
    MDH_REQUIRE(frames != nullptr, MDH_EINVAL, "frames is NULL");
    MDH_REQUIRE(c->rdf.configured, MDH_ESTATE, "rdf: not configured");
    unsigned long long h[8] = {0};
    MDH_CUDA(cudaMemcpyAsync(h, c->rdf.fstats.p, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
    MDH_CUDA(cudaStreamSynchronize(c->stream));
    frames[0] = (int64_t)h[7];
    return MDH_OK;
}

/* ---- seam #2 ---- */

int mdh_sq_configure(mdh_ctx *c, int64_t n_total, int n_groups, const int64_t *group_offsets,
                     int n_q, const double *wavevectors, const int32_t *lattice_n,
                     const double *lattice_b, int n_pairs, const int32_t *pairs, int mode)
{
    CTX_GUARD(c);
    return sq_configure_impl(c, n_total, n_groups, group_offsets, n_q, wavevectors, lattice_n,
                             lattice_b, n_pairs, pairs, mode);
}

int mdh_sq_accumulate(mdh_ctx *c, const float *pos, int64_t frame_stride, int location,
                      int n_frames)
{
    CTX_GUARD(c);
    return sq_accumulate_impl(c, pos, frame_stride, location, n_frames);
}

int mdh_sq_accumulate_f64(mdh_ctx *c, const double *pos, int64_t frame_stride, int location,
                          int n_frames)
{
    CTX_GUARD(c);
    return sq_accumulate_f64_impl(c, pos, frame_stride, location, n_frames);
}

int mdh_sq_fetch(mdh_ctx *c, double *ssf)
{
    CTX_GUARD(c);
    MDH_REQUIRE(c->sq.configured, MDH_ESTATE, "sq: fetch before configure");
    MDH_REQUIRE(ssf != nullptr, MDH_EINVAL, "sq: ssf is NULL");
    MDH_CUDA(cudaMemcpyAsync(ssf, c->sq.ssf.p,
                             sizeof(double) * (size_t)c->sq.n_pairs * c->sq.n_q,
                             cudaMemcpyDeviceToHost, c->stream));
    MDH_CUDA(cudaStreamSynchronize(c->stream));
    return MDH_OK;
}

int mdh_sq_kernel(mdh_ctx *c, int *mode)
{
    MDH_REQUIRE(c && mode, MDH_EINVAL, "NULL argument");
    MDH_REQUIRE(c->sq.configured, MDH_ESTATE, "sq: not configured");
    *mode = c->sq.mode;
    return MDH_OK;
}

int mdh_sq_plan(int n_q, const int32_t *lattice_n, int64_t *stats, int32_t *coverage,
                int32_t *pair_rule_violations)
{
    return sq_plan_impl(n_q, lattice_n, stats, coverage, pair_rule_violations);
}

int mdh_sq_tiling(mdh_ctx *c, int64_t *stats)
{
    MDH_REQUIRE(c && stats, MDH_EINVAL, "NULL argument");
    MDH_REQUIRE(c->sq.configured, MDH_ESTATE, "sq: not configured");
    for (int i = 0; i < 4; ++i) stats[i] = c->sq.mma ? c->sq.mma_stats[i] : 0;
    return MDH_OK;
}

int mdh_sq_reset(mdh_ctx *c)
{
    CTX_GUARD(c);
    MDH_REQUIRE(c->sq.configured, MDH_ESTATE, "sq: reset before configure");
    MDH_CUDA(cudaMemsetAsync(c->sq.ssf.p, 0, sizeof(double) * (size_t)c->sq.n_pairs * c->sq.n_q,
                             c->stream));
    return MDH_OK;
}

int mdh_sq_accum_device(mdh_ctx *c, void **dptr)
{
    MDH_REQUIRE(c && dptr, MDH_EINVAL, "NULL argument");
    MDH_REQUIRE(c->sq.configured, MDH_ESTATE, "sq: not configured");
    *dptr = c->sq.ssf.p;
    return MDH_OK;
}

int mdh_sq_fetch_rho(mdh_ctx *c, double *rho)
{
    CTX_GUARD(c);
    SqState &S = c->sq;
    MDH_REQUIRE(S.configured && S.rho_frames > 0, MDH_ESTATE, "sq: no frame has been processed");
    MDH_REQUIRE(rho != nullptr, MDH_EINVAL, "sq: rho is NULL");
    const size_t per_frame = (size_t)2 * S.n_rho * S.n_q;
    MDH_CUDA(cudaMemcpyAsync(rho, S.rho.as<double>() + per_frame * (S.rho_frames - 1),
                             sizeof(double) * per_frame, cudaMemcpyDeviceToHost, c->stream));
    MDH_CUDA(cudaStreamSynchronize(c->stream));
    return MDH_OK;
}

int mdh_com_configure(mdh_ctx *c, int slot, int64_t n_atoms, int64_t n_entities,
                      const int64_t *starts, const double *masses)
{
    CTX_GUARD(c);
    return com_configure_impl(c, slot, n_atoms, n_entities, starts, masses);
}

int mdh_com_reduce(mdh_ctx *c, int slot, const float *pos, int64_t frame_stride, int location,
                   int n_frames, float *out_device, int64_t out_frame_stride)
{
    CTX_GUARD(c);
    return com_reduce_impl(c, slot, pos, frame_stride, location, n_frames, out_device,
                           out_frame_stride);
}

int mdh_com_reduce_f64(mdh_ctx *c, int slot, const float *pos, int64_t frame_stride,
                       int location, int n_frames, double *out_device,
                       int64_t out_frame_stride)
{
    CTX_GUARD(c);
    return com_reduce_f64_impl(c, slot, pos, frame_stride, location, n_frames, out_device,
                               out_frame_stride);
}

int mdh_sq_configure_chains(mdh_ctx *c, int64_t n_chains, int64_t n_monomers)
{
    CTX_GUARD(c);
    return sq_configure_chains_impl(c, n_chains, n_monomers);
}

/* ---- intermediate scattering function (on top of seam #2) ---- */

int mdh_isf_configure(mdh_ctx *c, int n_lags, int incoherent, int64_t max_frames)
{
    CTX_GUARD(c);
    return isf_configure_impl(c, n_lags, incoherent, max_frames);
}

int mdh_isf_accumulate(mdh_ctx *c, const float *pos, int64_t frame_stride, int location,
                       int n_frames)
{
    CTX_GUARD(c);
    return isf_accumulate_impl(c, pos, frame_stride, location, n_frames);
}

int mdh_isf_accumulate_f64(mdh_ctx *c, const double *pos, int64_t frame_stride, int location,
                           int n_frames)
{
    CTX_GUARD(c);
    return isf_accumulate_f64_impl(c, pos, frame_stride, location, n_frames);
}

int mdh_stage_plan(int n_frames, double bytes_per_frame, double copy_over_kernel,
                   int32_t *pieces, int cap, int32_t *n_pieces)
{
    if (n_frames < 0 || !pieces || !n_pieces || cap < 0) {
        mdh_set_error("stage_plan: invalid argument");
        return MDH_EINVAL;
    }
    const std::vector<int> p = mdh_plan_pieces(n_frames, bytes_per_frame, copy_over_kernel);
    *n_pieces = (int32_t)p.size();
    for (size_t k = 0; k < p.size() && (int)k < cap; ++k) pieces[k] = p[k];
    return MDH_OK;
}

int mdh_isf_fetch(mdh_ctx *c, double *cisf, double *iisf)
{
    CTX_GUARD(c);
    return isf_fetch_impl(c, cisf, iisf);
}

}  // extern "C"
