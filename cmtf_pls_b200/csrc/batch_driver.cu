// Host side of tpls_fit_batch (include/tpls_b200.h): limits, the per-problem working-set layout, where it lives
// (shared memory or a slot of a global workspace), staging of host inputs and results.  Kernel: batch.cu.
#include "batch.cuh"
#include "driver_internal.cuh"

namespace {

size_t up16(size_t b) { return (b + 15) & ~(size_t)15; }

long long env_ll(const char* name, long long dflt) {
    const char* v = getenv(name);
    return (v == nullptr || *v == '\0') ? dflt : atoll(v);
}

// Largest per-problem working set (MB) the batch kernel takes by default.  See DESIGN.md section 4d for the
// measurement behind it: above it one CTA per problem streams its problem at a fraction of what the streaming
// kernels of the ordinary fit reach with the whole GPU.
constexpr long long kBatchDefaultMB = 16;

int unsupported(tpls_handle h, const char* fmt, ...) {
    char buf[384];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    h->error = std::string("tpls_fit_batch: ") + buf;
    return TPLS_E_BATCH_UNSUPPORTED;
}

}  // namespace

extern "C" int tpls_fit_batch(tpls_handle h, int n_tensors, int64_t batch, const void* const* xs, const int* dtypes,
                              const int* ndims, const int64_t* const* shapes, const int64_t* x_batch_stride,
                              const double* y, int64_t m, int64_t y_batch_stride, const double* row_w, int n_components,
                              double tol, int max_iter, int flags, tpls_batch_out* out) {
    if (!h) return fail(nullptr, "NULL handle");
    const int L = n_tensors, R = n_components;
    if (L < 1 || L > TPLS_MAX_TENSORS) return fail(h, "tpls_fit_batch: n_tensors must be 1..%d", TPLS_MAX_TENSORS);
    if (batch < 1 || batch > INT32_MAX) return fail(h, "tpls_fit_batch: batch must be 1..%d", INT32_MAX);
    if (R < 1) return fail(h, "tpls_fit_batch: n_components must be >= 1");
    if (max_iter < 1 || max_iter > 4096) return fail(h, "tpls_fit_batch: max_iter must be 1..4096");
    if (!xs || !dtypes || !ndims || !shapes || !x_batch_stride || !y || !out)
        return fail(h, "tpls_fit_batch: NULL argument");
    if (m < 1) return fail(h, "tpls_fit_batch: Y needs at least one column");
    if (y_batch_stride < 0) return fail(h, "tpls_fit_batch: negative batch stride of Y");
    long long n = -1;
    for (int l = 0; l < L; ++l) {
        if (!xs[l] || !shapes[l]) return fail(h, "tpls_fit_batch: NULL X[%d]", l);
        if (dtypes[l] != TPLS_F32 && dtypes[l] != TPLS_F64) return fail(h, "tpls_fit_batch: X[%d]: dtype must be F32 or F64", l);
        if (ndims[l] < 2 || ndims[l] > TPLS_MAX_MODES) return fail(h, "tpls_fit_batch: X[%d]: ndim must be 2..%d", l, TPLS_MAX_MODES);
        if (x_batch_stride[l] < 0) return fail(h, "tpls_fit_batch: X[%d]: negative batch stride", l);
        for (int k = 0; k < ndims[l]; ++k)
            if (shapes[l][k] < 1) return fail(h, "tpls_fit_batch: X[%d] has an empty mode", l);
        if (n < 0) n = shapes[l][0];
        if (shapes[l][0] != n) return fail(h, "tpls_fit_batch: X[%d] has %lld samples, X[0] %lld", l, (long long)shapes[l][0], n);
        if (!out->W[l] || !out->x_mean[l]) return fail(h, "tpls_fit_batch: NULL output W[%d] / x_mean[%d]", l, l);
    }
    if (!out->T || !out->U || !out->Q || !out->coef || !out->r2x || !out->r2y || !out->y_mean || !out->trips ||
        !out->converged || !out->has_missing)
        return fail(h, "tpls_fit_batch: NULL output");
    if (n > (1 << 30)) return fail(h, "tpls_fit_batch: too many samples per problem");

    // ---- limits of the kernel: outside them nothing is written and the caller fits the problems one by one ----
    if (env_ll("TPLS_BATCH", 1) == 0) return unsupported(h, "batch kernel turned off (TPLS_BATCH=0)");
    if (m > kBatchMaxResp) return unsupported(h, "%lld responses (the batch kernel takes up to %d)", (long long)m, kBatchMaxResp);
    if (R > kBatchMaxComp) return unsupported(h, "%d components (the batch kernel takes up to %d)", R, kBatchMaxComp);

    BatchArgs a{};
    a.n_tensors = L;
    a.batch = (int)batch;
    a.n = (int)n;
    a.m = (int)m;
    a.R = R;
    a.y_bstride = y_batch_stride;
    a.tol = tol;
    a.max_iter = max_iter;
    a.normalize_on_break = (flags & TPLS_FIT_NORMALIZE_ON_BREAK) ? 1 : 0;
    size_t off = 0, r1_max = 0;
    for (int l = 0; l < L; ++l) {
        BatchTensor& X = a.x[l];
        const int elem = dtypes[l] == TPLS_F32 ? 4 : 8;
        long long p = 1;
        X.w_rows = 0;
        for (int k = 1; k < ndims[l]; ++k) {
            p *= shapes[l][k];
            X.w_rows += (int)shapes[l][k];
        }
        if (p > (1 << 30)) return fail(h, "tpls_fit_batch: X[%d] has too many columns", l);
        X.dtype = dtypes[l];
        X.p = (int)p;
        X.x_bstride = x_batch_stride[l];
        X.nmodes = ndims[l] - 1;
        for (int k = 0; k < X.nmodes; ++k) X.dims[k] = (int)shapes[l][k + 1];
        const size_t ws = rank1_workspace_doubles(X.nmodes, X.dims, &X.r1_nmax, &X.r1_zs, &X.r1_mt, &X.r1_tab);
        if (ws * sizeof(double) > 200 * 1024)
            return unsupported(h, "the rank-1 workspace of X[%d] (%zu KB) does not fit in shared memory", l,
                               ws * sizeof(double) / 1024);
        r1_max = std::max(r1_max, ws);
        X.off_x = off;      off = up16(off + (size_t)n * p * elem);
        X.off_mean = off;   off = up16(off + (size_t)p * 8);
        X.off_cnt = off;    off = up16(off + (size_t)p * 8);
        X.off_z = off;      off = up16(off + (size_t)p * 8);
        X.off_wk = off;     off = up16(off + (size_t)p * 8);
        X.off_fac = off;    off = up16(off + (size_t)X.w_rows * 8);
        X.off_rowcnt = off; off = up16(off + (size_t)n * 8);
    }
    a.off_y = off;  off = up16(off + (size_t)n * m * 8);
    a.off_t = off;  off = up16(off + (size_t)n * R * 8);
    a.off_u = off;  off = up16(off + (size_t)n * 8);
    a.off_r1 = off; off = up16(off + r1_max * 8);
    a.ws_bytes = off;
    const long long limit_mb = env_ll("TPLS_BATCH_MB", kBatchDefaultMB);
    if ((double)a.ws_bytes > (double)limit_mb * 1048576.0)
        return unsupported(h, "working set of %.1f MB per problem (the batch kernel takes up to %lld MB, TPLS_BATCH_MB)",
                           a.ws_bytes / 1048576.0, limit_mb);

    CK(cudaSetDevice(h->device));
    NvtxRange nvtx("tpls_fit_batch");
    cudaStream_t st = h->stream;
    const bool in_smem = env_ll("TPLS_BATCH_SMEM", 1) != 0 && a.ws_bytes <= batch_fit_smem_limit();
    const size_t smem = in_smem ? a.ws_bytes : 0;
    const int max_ctas = batch_fit_max_ctas(smem);
    if (max_ctas < 1) return fail(h, "tpls_fit_batch: no CTA of the batch kernel fits on this device");
    const int grid = (int)std::min<long long>(batch, max_ctas);

    // ---- device memory of this call: staged inputs, results for host outputs, the global working sets ----
    std::vector<void*> bufs;
    struct Release {
        tpls_handle h;
        std::vector<void*>& b;
        ~Release() {  // nothing of this call may still run on the buffers when they go back to the pool
            if (!b.empty()) cudaStreamSynchronize(h->stream);
            for (void* p : b) pool_put(h, p);
        }
    } release{h, bufs};
    auto dev_buf = [&](void** p, size_t bytes) -> int {
        TRY(pool_get(h, p, std::max<size_t>(bytes, 16)));
        bufs.push_back(*p);
        return 0;
    };
    auto stage_in = [&](const void* src, size_t bytes, const void** dst) -> int {
        if (is_device_ptr(src)) {
            *dst = src;
            return 0;
        }
        void* d = nullptr;
        TRY(dev_buf(&d, bytes));
        CK(cudaMemcpyAsync(d, src, bytes, cudaMemcpyHostToDevice, st));
        *dst = d;
        return 0;
    };
    CK(cudaEventRecord(h->ev_start, st));
    for (int l = 0; l < L; ++l) {
        const size_t elem = dtypes[l] == TPLS_F32 ? 4 : 8;
        const size_t span = ((size_t)(batch - 1) * x_batch_stride[l] + (size_t)n * a.x[l].p) * elem;
        TRY(stage_in(xs[l], span, &a.x[l].x));
    }
    {
        const void* d = nullptr;
        TRY(stage_in(y, ((size_t)(batch - 1) * y_batch_stride + (size_t)n * m) * 8, &d));
        a.y = static_cast<const double*>(d);
        if (row_w != nullptr) {
            TRY(stage_in(row_w, (size_t)batch * n * 8, &d));
            a.row_w = static_cast<const double*>(d);
        }
    }
    // results: written where they are when the caller gave device memory, else through a device buffer
    struct OutCopy {
        void* host;
        void* dev;
        size_t bytes;
    };
    std::vector<OutCopy> copies;
    auto place_out = [&](void* user, size_t bytes, void** dst) -> int {
        if (is_device_ptr(user)) {
            *dst = user;
            return 0;
        }
        TRY(dev_buf(dst, bytes));
        copies.push_back(OutCopy{user, *dst, bytes});
        return 0;
    };
    const size_t B = (size_t)batch;
    void* p = nullptr;
    TRY(place_out(out->T, B * n * R * 8, &p));           a.T = static_cast<double*>(p);
    TRY(place_out(out->U, B * n * R * 8, &p));           a.U = static_cast<double*>(p);
    TRY(place_out(out->Q, B * m * R * 8, &p));           a.Q = static_cast<double*>(p);
    TRY(place_out(out->coef, B * R * R * 8, &p));        a.coef = static_cast<double*>(p);
    TRY(place_out(out->r2x, B * L * R * 8, &p));         a.r2x = static_cast<double*>(p);
    TRY(place_out(out->r2y, B * R * 8, &p));             a.r2y = static_cast<double*>(p);
    TRY(place_out(out->y_mean, B * m * 8, &p));          a.y_mean = static_cast<double*>(p);
    TRY(place_out(out->trips, B * R * 4, &p));           a.trips = static_cast<int*>(p);
    TRY(place_out(out->converged, B * R * 4, &p));       a.conv = static_cast<int*>(p);
    TRY(place_out(out->has_missing, B * L * 4, &p));     a.has_missing = static_cast<int*>(p);
    for (int l = 0; l < L; ++l) {
        TRY(place_out(out->W[l], B * a.x[l].w_rows * R * 8, &p));
        a.x[l].W = static_cast<double*>(p);
        TRY(place_out(out->x_mean[l], B * a.x[l].p * (dtypes[l] == TPLS_F32 ? 4 : 8), &p));
        a.x[l].mean_out = p;
    }
    if (!in_smem) {
        void* g = nullptr;
        TRY(dev_buf(&g, (size_t)grid * a.ws_bytes));
        a.gws = static_cast<char*>(g);
    }
    CK(launch_batch_fit(a, grid, smem, st));
    for (const OutCopy& c : copies) CK(cudaMemcpyAsync(c.host, c.dev, c.bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(h->ev_stop, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->ev_start, h->ev_stop));
    out->fit_ms = ms;
    return 0;
}
