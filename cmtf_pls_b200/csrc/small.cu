// Small kernels -- see small.cuh.
#include "small.cuh"
#include "stream_common.cuh"

#include <cstdlib>

#include <algorithm>

namespace tpls {

bool pdl_enabled() {
    // on by default since round 2 (all GPU tests and the 1/2/8-GPU benchmark run with it); TPLS_PDL=0 turns it off
    static const bool on = [] {
        const char* v = getenv("TPLS_PDL");
        return v == nullptr || *v == '\0' || *v != '0';
    }();
    return on;
}

static thread_local bool g_pdl_hold = false;
void pdl_hold_next() { g_pdl_hold = true; }
bool pdl_take_hold() {
    const bool h = g_pdl_hold;
    g_pdl_hold = false;
    return h;
}

template <typename XT>
__global__ void finalize_mean_kernel(const double* colsum, const double* colcnt, const double* n_total, int p, int pitch,
                                     double* mean_d, XT* native_out, int* miss_flag, const double* nmiss) {
    pdl_prologue();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c == 0 && nmiss != nullptr && *nmiss > 0.0) atomicOr(miss_flag, 1);  // NaNs in rows of weight 0 count too
    if (c >= pitch) return;
    if (c >= p) {
        mean_d[c] = 0.0;
        return;
    }
    const double cnt = colcnt[c];
    const XT m = (XT)(colsum[c] / cnt);  // 0/0 -> NaN for an all-missing column, like np.nanmean
    mean_d[c] = (double)m;
    if (native_out) native_out[c] = m;
    if (cnt < *n_total) atomicOr(miss_flag, 1);
}

cudaError_t launch_finalize_mean(int dtype, const double* colsum, const double* colcnt, const double* n_total, int p,
                                 int pitch, double* mean_d, void* native_out, int* miss_flag, const double* nmiss,
                                 cudaStream_t s) {
    const int blocks = (pitch + 255) / 256;
    if (dtype == 0)
        launch_k(finalize_mean_kernel<float>, dim3(blocks), dim3(256), 0, s, colsum, colcnt, n_total, p, pitch, mean_d,
                                                           (float*)native_out, miss_flag, nmiss);
    else
        launch_k(finalize_mean_kernel<double>, dim3(blocks), dim3(256), 0, s, colsum, colcnt, n_total, p, pitch, mean_d,
                                                            (double*)native_out, miss_flag, nmiss);
    return cudaGetLastError();
}

__global__ void gather_col_kernel(const double* src, long long n, int pitch, int col, double* dst) {
    pdl_prologue();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        dst[i] = src[i * pitch + col];
}

cudaError_t launch_gather_col(const double* src, long long n, int pitch, int col, double* dst, cudaStream_t s) {
    const int blocks = (int)std::max<long long>(1, std::min<long long>(1184, (n + 255) / 256));
    launch_k(gather_col_kernel, dim3(blocks), dim3(256), 0, s, src, n, pitch, col, dst);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) normalize_q_kernel(const double* qraw, int m, int pitch, double* qcol,
                                                          double* qvec, const Ctrl* ctrl, int trip) {
    pdl_prologue();
    if (trip_is_dead(ctrl, trip)) return;
    __shared__ double red[40];
    double s = 0.0;
    for (int i = threadIdx.x; i < m; i += blockDim.x) s = fma(qraw[i], qraw[i], s);
    const double nrm = sqrt(block_sum(s, red));
    for (int i = threadIdx.x; i < pitch; i += blockDim.x) {
        const double q = i < m ? qraw[i] / nrm : 0.0;
        if (i < m) qcol[i] = q;
        qvec[i] = q;
    }
}

cudaError_t launch_normalize_q(const double* qraw, int m, int pitch, double* qcol, double* qvec, const Ctrl* ctrl,
                               int trip, cudaStream_t s) {
    launch_k(normalize_q_kernel, dim3(1), dim3(256), 0, s, qraw, m, pitch, qcol, qvec, ctrl, trip);
    return cudaGetLastError();
}

// 32 columns x 8 part-groups, the fold of reduce_cols_kernel (passes.cu) for one 32-column chunk
__global__ void __launch_bounds__(256) reduce_q_stop_kernel(const double* part, int n_parts, int stride, double* qraw, int m,
                                                            int pitch, double* qcol, double* qvec, const double* gram,
                                                            double* q_prev, Ctrl* ctrl, const LoopEnd e) {
    pdl_prologue();
    if (trip_is_dead(ctrl, 0)) return;
    // pitch <= 8 columns: 8 columns x 32 part-groups (the association order of fold_narrow)
    __shared__ double fold32[32][9];
    __shared__ double qsum[8];
    FoldSet S{part, n_parts, stride, pitch, 0};
    const double t = fold_narrow(S, fold32);
    if ((threadIdx.x >> 3) == 0 && (int)(threadIdx.x & 7) < pitch) {
        qsum[threadIdx.x & 7] = t;
        qraw[threadIdx.x & 7] = t;
    }
    __syncthreads();
    if (threadIdx.x == 0) normalize_q_stop_body(qsum, m, pitch, qcol, qvec, gram, q_prev, ctrl, e);
}

cudaError_t launch_reduce_q_stop(const double* part, int n_parts, int stride, double* qraw, int m, int pitch, double* qcol,
                                 double* qvec, const double* gram, double* q_prev, Ctrl* ctrl, const LoopEnd& e,
                                 cudaStream_t s) {
    if (pitch > 8 || m > 8) return cudaErrorInvalidValue;
    launch_k(reduce_q_stop_kernel, dim3(1), dim3(256), 0, s, part, n_parts, stride, qraw, m, pitch, qcol, qvec, gram, q_prev, ctrl, e);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) stop_kernel(Ctrl* ctrl, const double* parts, int n, const LoopEnd e) {
    pdl_prologue();
    if (trip_is_dead(ctrl, 0)) return;
    __shared__ double red[40];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) s += parts[i];
    s = block_sum(s, red);
    if (threadIdx.x == 0) ctrl_decide(ctrl, s, e);
}

cudaError_t launch_stop(Ctrl* ctrl, const double* parts, int n, const LoopEnd& e, cudaStream_t s) {
    launch_k(stop_kernel, dim3(1), dim3(256), 0, s, ctrl, parts, n, e);
    return cudaGetLastError();
}

__global__ void reset_ctrl_kernel(Ctrl* ctrl) {
    pdl_prologue();
    ctrl->done_trip = -1;
    ctrl->trips_taken = 0;
    ctrl->last_d2 = 0.0;
    ctrl->trip = 0;
    ctrl->stop = 0;
}

cudaError_t launch_reset_ctrl(Ctrl* ctrl, cudaStream_t s) {
    launch_k(reset_ctrl_kernel, dim3(1), dim3(1), 0, s, ctrl);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) multi_dot_kernel(const __grid_constant__ DotPairs d, double* part) {
    pdl_prologue();
    __shared__ double red[40];
    const int j = blockIdx.y;
    const double* a = d.a[j];
    const double* b = d.b[j];
    double s = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < d.n; i += (long long)gridDim.x * blockDim.x)
        if (d.w == nullptr || d.w[i] != 0.0) s = fma(d.w != nullptr ? a[i] * d.w[i] : a[i], b[i], s);  // NaN * 0 is NaN
    s = block_sum(s, red);
    if (threadIdx.x == 0) part[(size_t)blockIdx.x * d.npairs + j] = s;
}

cudaError_t launch_multi_dot(const DotPairs& d, double* part, int* grid_out, cudaStream_t s) {
    const int gx = (int)std::max<long long>(1, std::min<long long>(148, (d.n + 2047) / 2048));
    if (grid_out) *grid_out = gx;
    launch_k(multi_dot_kernel, dim3(gx, d.npairs), dim3(256), 0, s, d, part);
    return cudaGetLastError();
}

__global__ void solve_coef_kernel(const double* dots, double* gram, double* coef, int R, int a, const Ctrl* ctrl,
                                  int* trips_out, int* conv_out) {
    pdl_prologue();
    if (threadIdx.x != 0) return;
    const int k = a + 1;
    for (int b = 0; b < k; ++b) {
        gram[b * R + a] = dots[b];
        gram[a * R + b] = dots[b];
    }
    // Normal equations of the leading k x k block (k <= 64) on UNIT-NORM score columns: with D = diag(||t_b||),
    // (D^-1 G D^-1) (D x) = D^-1 rhs.  The scaling keeps the Cholesky factor well conditioned when a score column
    // is merely tiny (components past the rank of the data: ||t|| ~ 1e-15 ||t_0||, where the plain Gram matrix
    // loses its pivot and everything downstream turns NaN).  A column that is zero, or dependent on the earlier
    // ones to rounding, gets coefficient 0 -- the reference's lstsq (rcond = machine precision, tpls.py:110-112)
    // drops such directions too.
    double Lm[64 * 64];
    double y[64], x[64], dinv[64];
    bool drop[64];
    for (int i = 0; i < k; ++i) {
        const double g = gram[i * R + i];
        drop[i] = !(g > 0.0);
        dinv[i] = drop[i] ? 0.0 : 1.0 / sqrt(g);
    }
    for (int i = 0; i < k; ++i) {
        for (int j = 0; j <= i; ++j) {
            double s = (drop[i] || drop[j]) ? (i == j ? 1.0 : 0.0) : gram[i * R + j] * dinv[i] * dinv[j];
            for (int q = 0; q < j; ++q) s -= Lm[i * 64 + q] * Lm[j * 64 + q];
            if (i == j) {
                if (!(s > 1e-14)) {  // no independent part left in column i
                    drop[i] = true;
                    for (int q = 0; q < i; ++q) Lm[i * 64 + q] = 0.0;
                    s = 1.0;
                }
                Lm[i * 64 + i] = sqrt(s);
            } else {
                Lm[i * 64 + j] = s / Lm[j * 64 + j];
            }
        }
    }
    for (int i = 0; i < k; ++i) {
        double s = drop[i] ? 0.0 : dots[k + i] * dinv[i];
        for (int q = 0; q < i; ++q) s -= Lm[i * 64 + q] * y[q];
        y[i] = s / Lm[i * 64 + i];
    }
    for (int i = k - 1; i >= 0; --i) {
        double s = y[i];
        for (int q = i + 1; q < k; ++q) s -= Lm[q * 64 + i] * x[q];
        x[i] = drop[i] ? 0.0 : s / Lm[i * 64 + i];
    }
    for (int b = 0; b < k; ++b) coef[b * R + a] = x[b] * dinv[b];
    if (trips_out != nullptr && ctrl != nullptr) trips_out[a] = ctrl->trips_taken;
    if (conv_out != nullptr && ctrl != nullptr) conv_out[a] = ctrl->done_trip >= 0 ? 1 : 0;
}

cudaError_t launch_solve_coef(const double* dots, double* gram, double* coef, int R, int a, const Ctrl* ctrl,
                              int* trips_out, int* conv_out, cudaStream_t s) {
    launch_k(solve_coef_kernel, dim3(1), dim3(32), 0, s, dots, gram, coef, R, a, ctrl, trips_out, conv_out);
    return cudaGetLastError();
}

__global__ void lincomb_kernel(const double* T, long long n, long long ldt, const double* coef, int R, int a,
                               const double* row_w, double* out) {
    pdl_prologue();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        double s = 0.0;
        for (int b = 0; b <= a; ++b) s = fma(T[b * ldt + i], coef[b * R + a], s);
        out[i] = row_w == nullptr ? s : (row_w[i] != 0.0 ? s * row_w[i] : 0.0);  // a NaN score of a held-out row
    }
}

cudaError_t launch_lincomb(const double* T, long long n, long long ldt, const double* coef, int R, int a,
                           const double* row_w, double* out, cudaStream_t s) {
    const int blocks = (int)std::max<long long>(1, std::min<long long>(1184, (n + 255) / 256));
    launch_k(lincomb_kernel, dim3(blocks), dim3(256), 0, s, T, n, ldt, coef, R, a, row_w, out);
    return cudaGetLastError();
}

__global__ void scale_rows_kernel(double* y, long long n, int pitch, const double* w) {
    pdl_prologue();
    const long long total = n * pitch;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x)
        y[e] *= w[e / pitch];
}

cudaError_t launch_scale_rows(double* y, long long n, int pitch, const double* w, cudaStream_t s) {
    const long long total = n * pitch;
    const int blocks = (int)std::max<long long>(1, std::min<long long>(1184, (total + 255) / 256));
    launch_k(scale_rows_kernel, dim3(blocks), dim3(256), 0, s, y, n, pitch, w);
    return cudaGetLastError();
}

__global__ void transpose_out_kernel(const double* in, long long n, long long ld, int cols, double* out) {
    pdl_prologue();
    const long long total = n * cols;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        const long long i = e / cols;
        const int c = (int)(e - i * cols);
        out[e] = in[c * ld + i];
    }
}

cudaError_t launch_transpose_out(const double* in, long long n, long long ld, int cols, double* out, cudaStream_t s) {
    const long long total = n * cols;
    const int blocks = (int)std::max<long long>(1, std::min<long long>(1184, (total + 255) / 256));
    launch_k(transpose_out_kernel, dim3(blocks), dim3(256), 0, s, in, n, ld, cols, out);
    return cudaGetLastError();
}

__global__ void fill_kernel(double* p, long long n, double v) {
    pdl_prologue();
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        p[i] = v;
}

cudaError_t launch_fill(double* p, long long n, double v, cudaStream_t s) {
    const int blocks = (int)std::max<long long>(1, std::min<long long>(1184, (n + 255) / 256));
    launch_k(fill_kernel, dim3(blocks), dim3(256), 0, s, p, n, v);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) gram_rows_kernel(const double* y, long long n, int pitch, int m, double* part) {
    pdl_prologue();
    __shared__ double red[40];
    double acc[36];  // upper triangle of an 8 x 8 matrix
#pragma unroll
    for (int k = 0; k < 36; ++k) acc[k] = 0.0;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (long long)gridDim.x * blockDim.x) {
        double v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = i < m ? y[r * pitch + i] : 0.0;
        int k = 0;
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = i; j < 8; ++j) {
                acc[k] = fma(v[i], v[j], acc[k]);
                ++k;
            }
    }
    int k = 0;
    for (int i = 0; i < 8; ++i)
        for (int j = i; j < 8; ++j) {
            const double t = block_sum(acc[k++], red);
            if (threadIdx.x == 0 && i < m && j < m) {
                part[(size_t)blockIdx.x * m * m + i * m + j] = t;
                part[(size_t)blockIdx.x * m * m + j * m + i] = t;
            }
        }
}

cudaError_t launch_gram_rows(const double* y, long long n, int pitch, int m, double* part, int* grid_out, cudaStream_t s) {
    const int gx = (int)std::max<long long>(1, std::min<long long>(148, (n + 1023) / 1024));
    if (grid_out) *grid_out = gx;
    launch_k(gram_rows_kernel, dim3(gx), dim3(256), 0, s, y, n, pitch, m, part);
    return cudaGetLastError();
}

__global__ void count_rescale_kernel(double* z, const double* cnt, double n_total, int p) {
    pdl_prologue();
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < p) z[c] = cnt[c] > 0.0 ? z[c] / cnt[c] * n_total : 0.0;
}

cudaError_t launch_count_rescale(double* z, const double* cnt, double n_total, int p, cudaStream_t s) {
    launch_k(count_rescale_kernel, dim3((p + 255) / 256), dim3(256), 0, s, z, cnt, n_total, p);
    return cudaGetLastError();
}

template <typename XT>
__global__ void widen_kernel(const XT* src, double* dst, int n) {
    pdl_prologue();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = (double)src[i];
}

cudaError_t launch_widen(int dtype, const void* src, double* dst, int n, cudaStream_t s) {
    if (dtype == 0)
        launch_k(widen_kernel<float>, dim3((n + 255) / 256), dim3(256), 0, s, (const float*)src, dst, n);
    else
        launch_k(widen_kernel<double>, dim3((n + 255) / 256), dim3(256), 0, s, (const double*)src, dst, n);
    return cudaGetLastError();
}

}  // namespace tpls
