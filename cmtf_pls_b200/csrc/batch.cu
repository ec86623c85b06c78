// Batched fits, one CTA per problem -- see batch.cuh.
//
// Every step uses the arithmetic of the ordinary fit and rounds where it rounds:
//   statistics   colpass_kernel<PF_COLSTAT> + finalize_mean_kernel (weighted sums and counts, UNWEIGHTED NaN census,
//                the mean rounded to X's dtype)
//   centring     colpass_kernel<PF_DEFLATE | PF_WRITE | PF_SUMSQ>: x - mean rounded to the storage type, Sum w x^2
//   Y            centred, ||Y_c||^2 weighted, then multiplied by the 0/1 row weight (scale_rows_kernel)
//   inner loop   resident_loop_kernel: Z = Sum u x (masked: rescaled by N / n_j as the rank-1 step does), rank1_task
//                itself, the projection (masked: p / observed(row)) and the coupled average, q = Y't normalised,
//                the stop test dq^T (Y'Y) dq < tol^2 from trip 1 on, u = Y q
//   tail         solve_coef (unit-norm score columns, dependent columns get 0), the Y deflation, the X deflation
//                fused with its residual norm; after the last component the norm of the unrounded residual
// Held-out rows (weight 0) are centred, projected and deflated like the others, so their scores are transform() of
// those rows under the fold's model.  Such a score is NaN for a row without observed entries, and deflation by it
// turns that row of a dense coupled tensor NaN too; so every sum over rows skips a weight-0 row instead of
// multiplying it by 0 (NaN * 0 is NaN).  On finite data the skip gives the bits of the multiply.
#include "batch.cuh"
#include "rank1_task.cuh"

#include <algorithm>

namespace tpls {

namespace {

__device__ __forceinline__ double ldx(const void* p, int dt, size_t i) {
    return dt == 0 ? (double)static_cast<const float*>(p)[i] : static_cast<const double*>(p)[i];
}

// store in the storage type; returns the stored (rounded) value, which later steps see
__device__ __forceinline__ double stx(void* p, int dt, size_t i, double v) {
    if (dt == 0) {
        const float f = (float)v;
        static_cast<float*>(p)[i] = f;
        return (double)f;
    }
    static_cast<double*>(p)[i] = v;
    return v;
}

// Column sums over the rows of a row-major [n][p] source: thread tid takes column tid % cg of each chunk of cg
// columns and every (NTH / cg)-th row; the row groups are folded in a fixed order.  f(i, c, acc1, acc2) accumulates
// row i of column c; out(c, s1, s2) receives the folded sums.
template <typename F, typename O>
__device__ __forceinline__ void col_reduce(int n, int p, double* scr, F f, O out) {
    const int tid = threadIdx.x;
    const int cg = min(p, NTH), rg = NTH / cg;
    const int g = tid / cg;
    for (int c0 = 0; c0 < p; c0 += cg) {
        const int c = c0 + tid % cg;
        double s1 = 0.0, s2 = 0.0;
        if (g < rg && c < p)
            for (int i = g; i < n; i += rg) f(i, c, s1, s2);
        scr[tid] = s1;
        scr[NTH + tid] = s2;
        __syncthreads();
        if (tid < cg && c0 + tid < p) {
            double t1 = 0.0, t2 = 0.0;
            for (int k = 0; k < rg; ++k) {
                t1 += scr[k * cg + tid];
                t2 += scr[NTH + k * cg + tid];
            }
            out(c0 + tid, t1, t2);
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kRank1Threads, 1) batch_fit_kernel(const __grid_constant__ BatchArgs a) {
    pdl_prologue();
    extern __shared__ __align__(16) double dyn[];
    __shared__ double scr[2 * NTH];
    __shared__ double red[40];
    __shared__ double q_s[8], qp_s[8], qraw_s[8], ym_s[8], gy_s[64];
    __shared__ double gt_s[kBatchMaxComp * kBatchMaxComp], lm_s[kBatchMaxComp * kBatchMaxComp];
    __shared__ double dots_s[2 * kBatchMaxComp], ys_s[kBatchMaxComp], xs_s[kBatchMaxComp], dinv_s[kBatchMaxComp],
        drop_s[kBatchMaxComp];
    __shared__ double ss_s[kMaxTensors * (kBatchMaxComp + 1)], ssy_s[kBatchMaxComp + 1];
    __shared__ int masked_s[kMaxTensors];
    __shared__ int stop_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int L = a.n_tensors, n = a.n, M = a.m, R = a.R;
    char* const ws = a.gws != nullptr ? a.gws + (size_t)blockIdx.x * a.ws_bytes : reinterpret_cast<char*>(dyn);
    double* const Yw = reinterpret_cast<double*>(ws + a.off_y);
    double* const Tw = reinterpret_cast<double*>(ws + a.off_t);
    double* const uw = reinterpret_cast<double*>(ws + a.off_u);
    double* const r1w = reinterpret_cast<double*>(ws + a.off_r1);
    const double inv_l = 1.0 / (double)L;
    const bool pow2 = (L & (L - 1)) == 0;

    for (int prob = blockIdx.x; prob < a.batch; prob += gridDim.x) {
        const double* wr = a.row_w != nullptr ? a.row_w + (size_t)prob * n : nullptr;
        const double* ysrc = a.y + (size_t)prob * a.y_bstride;
        // sample count of the fit: the sum of the weights (the driver's multi_dot of w with itself)
        double nt = (double)n;
        if (wr != nullptr) {
            double s = 0.0;
            for (int i = tid; i < n; i += NTH) s = fma(wr[i], wr[i], s);
            nt = block_sum(s, red);
        }

        // ---- column statistics, centring, ||X_c||^2 of every tensor ----
        for (int l = 0; l < L; ++l) {
            const BatchTensor& X = a.x[l];
            const int p = X.p, dt = X.dtype;
            const void* xin = static_cast<const char*>(X.x) + (size_t)prob * X.x_bstride * (dt == 0 ? 4 : 8);
            double* mean = reinterpret_cast<double*>(ws + X.off_mean);
            double* cnt = reinterpret_cast<double*>(ws + X.off_cnt);
            int miss = 0;
            col_reduce(n, p, scr,
                       [&](int i, int c, double& s1, double& s2) {
                           const double sw = wr != nullptr ? wr[i] : 1.0;
                           double xd = ldx(xin, dt, (size_t)i * p + c);
                           const bool ob = xd == xd;
                           if (!ob) {
                               xd = 0.0;
                               miss = 1;  // the census is unweighted: NaNs in held-out rows count too
                           }
                           s1 = fma(xd, sw, s1);
                           s2 += ob ? sw : 0.0;
                       },
                       [&](int c, double s1, double s2) {
                           // 0/0 -> NaN for a column without observed entries, like np.nanmean
                           const double m = dt == 0 ? (double)(float)(s1 / s2) : s1 / s2;
                           mean[c] = m;
                           cnt[c] = s2;
                           if (dt == 0)
                               static_cast<float*>(X.mean_out)[(size_t)prob * p + c] = (float)m;
                           else
                               static_cast<double*>(X.mean_out)[(size_t)prob * p + c] = m;
                           if (s2 < nt) miss = 1;
                       });
            const int masked = __syncthreads_or(miss);
            if (tid == 0) {
                masked_s[l] = masked;
                a.has_missing[(size_t)prob * L + l] = masked;
            }
            void* xw = ws + X.off_x;
            double ss = 0.0;
            const size_t np = (size_t)n * p;
            for (size_t e = tid; e < np; e += NTH) {
                const int i = (int)(e / p), c = (int)(e - (size_t)i * p);
                const double x = ldx(xin, dt, e);
                double xd = stx(xw, dt, e, fma(-1.0, mean[c], x));  // NaN stays NaN
                if (masked && !(x == x)) xd = 0.0;
                const double sw = wr != nullptr ? wr[i] : 1.0;
                if (sw != 0.0) ss = fma(xd, xd, ss);
            }
            ss = block_sum(ss, red);
            if (tid == 0) ss_s[l * (R + 1)] = ss;
            if (masked) {
                // observed entries per row, counted after centring as transform() counts them: an entry of a column
                // without observed training entries (NaN mean) is not observed
                double* rowcnt = reinterpret_cast<double*>(ws + X.off_rowcnt);
                for (int i = warp; i < n; i += NWARP) {
                    double c = 0.0;
                    for (int j = lane; j < p; j += 32) {
                        const double v = ldx(xw, dt, (size_t)i * p + j);
                        c += v == v ? 1.0 : 0.0;
                    }
                    c = warp_sum(c);
                    if (lane == 0) rowcnt[i] = c;
                }
            }
        }
        // ---- Y: weighted mean, centring, ||Y_c||^2, held-out rows zeroed ----
        col_reduce(n, M, scr,
                   [&](int i, int c, double& s1, double& s2) {
                       const double sw = wr != nullptr ? wr[i] : 1.0;
                       double v = ysrc[(size_t)i * M + c];
                       const bool ob = v == v;
                       if (!ob) v = 0.0;
                       s1 = fma(v, sw, s1);
                       s2 += ob ? sw : 0.0;
                   },
                   [&](int c, double s1, double s2) {
                       ym_s[c] = s1 / s2;
                       a.y_mean[(size_t)prob * M + c] = s1 / s2;
                   });
        {
            double ssy = 0.0;
            for (int i = tid; i < n; i += NTH) {
                const double sw = wr != nullptr ? wr[i] : 1.0;
                double rs = 0.0;
                for (int c = 0; c < M; ++c) {
                    const double yc = fma(-1.0, ym_s[c], ysrc[(size_t)i * M + c]);
                    rs = fma(yc, yc, rs);
                    Yw[(size_t)i * M + c] = wr != nullptr ? yc * sw : yc;
                }
                ssy = fma(sw, rs, ssy);
            }
            ssy = block_sum(ssy, red);
            if (tid == 0) ssy_s[0] = ssy;
        }

        // ---- components ----
        for (int comp = 0; comp < R; ++comp) {
            // Y'Y of the current Y (the stop test: ||u_old - u_new||^2 = dq^T Y'Y dq)
            col_reduce(n, M * M, scr,
                       [&](int i, int e, double& s1, double&) {
                           const int r = e / M, c = e - r * M;
                           s1 = fma(Yw[(size_t)i * M + r], Yw[(size_t)i * M + c], s1);
                       },
                       [&](int e, double s1, double) { gy_s[e] = s1; });
            if (tid < 8) {
                q_s[tid] = tid == 0 ? 1.0 : 0.0;  // u_0 = Y e_0 (tpls.py:78)
                qp_s[tid] = q_s[tid];
            }
            __syncthreads();
            double* const Ta = Tw + (size_t)comp * n;
            int trip = 0, done_trip = -1;
            for (;;) {
                // u = Y q, then Z = X x_1 u for every tensor (tpls.py:83, 102)
                for (int i = tid; i < n; i += NTH) {
                    double u = 0.0;
                    for (int c = 0; c < M; ++c) u = fma(Yw[(size_t)i * M + c], q_s[c], u);
                    uw[i] = u;
                }
                __syncthreads();
                for (int l = 0; l < L; ++l) {
                    const BatchTensor& X = a.x[l];
                    const void* xw = ws + X.off_x;
                    const int p = X.p, dt = X.dtype;
                    double* z = reinterpret_cast<double*>(ws + X.off_z);
                    const double* cnt = reinterpret_cast<const double*>(ws + X.off_cnt);
                    const bool masked = masked_s[l] != 0;
                    col_reduce(n, p, scr,
                               [&](int i, int c, double& s1, double&) {
                                   double xd = ldx(xw, dt, (size_t)i * p + c);
                                   if (xd != xd) xd = 0.0;
                                   s1 = fma(xd, uw[i], s1);
                               },
                               [&](int c, double s1, double) {
                                   // masked: the N / n_j rescale of missingvals.py:18 with the arithmetic of the rank-1
                                   // step's (which reads the counts through the read-only cache, i.e. from global memory)
                                   z[c] = masked ? (cnt[c] > 0.0 ? s1 / cnt[c] * nt : 0.0) : s1;
                               });
                }
                // rank-1 step of every tensor (tpls.py:84-90, cmtf.py:98-104)
                for (int l = 0; l < L; ++l) {
                    const BatchTensor& X = a.x[l];
                    Rank1Task T{};
                    T.z = reinterpret_cast<const double*>(ws + X.off_z);
                    T.colcnt = nullptr;  // Z is rescaled already
                    T.n_total = nt;
                    T.p = X.p;
                    T.pitch = X.p;
                    T.nmodes = X.nmodes;
                    double* fac = reinterpret_cast<double*>(ws + X.off_fac);
                    int fo = 0;
                    for (int k = 0; k < X.nmodes; ++k) {
                        T.dims[k] = X.dims[k];
                        T.w[k] = fac + fo;
                        fo += X.dims[k];
                    }
                    T.wkron = reinterpret_cast<double*>(ws + X.off_wk);
                    T.scratch = r1w;
                    T.use_smem = a.gws == nullptr ? 1 : 0;
                    T.nmax = X.r1_nmax;
                    T.zs_len = X.r1_zs;
                    T.mt_len = X.r1_mt;
                    T.tab_cols = X.r1_tab;
                    rank1_task(T, a.tol, a.normalize_on_break, r1w);
                    __syncthreads();
                }
                // projection of every row (tpls.py:97-99; masked: missingvals.py:23-38), coupled average (cmtf.py:120)
                for (int i = warp; i < n; i += NWARP) {
                    double tl = 0.0, td = 0.0;
                    for (int l = 0; l < L; ++l) {
                        const BatchTensor& X = a.x[l];
                        const void* xw = ws + X.off_x;
                        const double* wk = reinterpret_cast<const double*>(ws + X.off_wk);
                        const int p = X.p, dt = X.dtype;
                        double v = 0.0;
                        for (int c = lane; c < p; c += 32) {
                            double xd = ldx(xw, dt, (size_t)i * p + c);
                            if (xd != xd) xd = 0.0;
                            v = fma(xd, wk[c], v);
                        }
                        if (masked_s[l]) {
                            v = warp_sum(v);
                            td += v / reinterpret_cast<const double*>(ws + X.off_rowcnt)[i] * (double)p;
                        } else {
                            tl += v;
                        }
                    }
                    tl = warp_sum(tl);
                    double ti = tl + td;
                    if (L > 1) ti = pow2 ? ti * inv_l : ti / (double)L;
                    if (lane == 0) Ta[i] = ti;
                }
                __syncthreads();
                // q = Y't / ||Y't|| and the stop test (tpls.py:100-107)
                col_reduce(n, M, scr, [&](int i, int c, double& s1, double&) {
                               const double sw = wr != nullptr ? wr[i] : 1.0;
                               if (sw != 0.0) s1 = fma(Yw[(size_t)i * M + c], Ta[i], s1);
                           },
                           [&](int c, double s1, double) { qraw_s[c] = s1; });
                if (tid == 0) {
                    double nrm = 0.0;
                    for (int c = 0; c < M; ++c) nrm = fma(qraw_s[c], qraw_s[c], nrm);
                    nrm = sqrt(nrm);
                    double dq[8];
                    for (int c = 0; c < M; ++c) {
                        const double qi = qraw_s[c] / nrm;
                        dq[c] = qp_s[c] - qi;
                        q_s[c] = qi;
                        qp_s[c] = qi;
                    }
                    double d2 = 0.0;
                    for (int r = 0; r < M; ++r)
                        for (int c = 0; c < M; ++c) d2 = fma(dq[r] * gy_s[r * M + c], dq[c], d2);
                    bool stop = false;
                    if (trip >= 1 && sqrt(fabs(d2)) < a.tol) {
                        done_trip = trip;
                        stop = true;
                    }
                    if (trip + 1 >= a.max_iter) stop = true;
                    stop_s = stop ? 1 : 0;
                }
                __syncthreads();
                ++trip;
                if (stop_s) break;
            }
            // ---- outputs of the component: u = Y q of the last trip, scores, q, loadings ----
            for (int i = tid; i < n; i += NTH) {
                double u = 0.0;
                for (int c = 0; c < M; ++c) u = fma(Yw[(size_t)i * M + c], q_s[c], u);
                uw[i] = u;
                a.U[((size_t)prob * n + i) * R + comp] = u;
                a.T[((size_t)prob * n + i) * R + comp] = Ta[i];
            }
            if (tid < M) a.Q[((size_t)prob * M + tid) * R + comp] = q_s[tid];
            for (int l = 0; l < L; ++l) {
                const BatchTensor& X = a.x[l];
                const double* fac = reinterpret_cast<const double*>(ws + X.off_fac);
                for (int r = tid; r < X.w_rows; r += NTH) X.W[((size_t)prob * X.w_rows + r) * R + comp] = fac[r];
            }
            __syncthreads();
            // ---- regression of u on the scores so far (tpls.py:110-112), the arithmetic of solve_coef ----
            const int ka = comp + 1;
            for (int j = warp; j < 2 * ka; j += NWARP) {
                const double* pa = Tw + (size_t)(j < ka ? j : j - ka) * n;
                const double* pb = j < ka ? Ta : uw;
                double s = 0.0;
#pragma unroll 1  // unrolled, this loop pushes the kernel past its 128 registers into a spill
                for (int i = lane; i < n; i += 32) {
                    const double sw = wr != nullptr ? wr[i] : 1.0;
                    if (sw != 0.0) s = fma(pa[i], pb[i], s);
                }
                s = warp_sum(s);
                if (lane == 0) dots_s[j] = s;
            }
            __syncthreads();
            if (tid == 0) {
                constexpr int LD = kBatchMaxComp;
                for (int b = 0; b < ka; ++b) {
                    gt_s[b * LD + comp] = dots_s[b];
                    gt_s[comp * LD + b] = dots_s[b];
                }
                for (int i = 0; i < ka; ++i) {
                    const double g = gt_s[i * LD + i];
                    drop_s[i] = !(g > 0.0) ? 1.0 : 0.0;
                    dinv_s[i] = drop_s[i] != 0.0 ? 0.0 : 1.0 / sqrt(g);
                }
                for (int i = 0; i < ka; ++i) {
                    for (int j = 0; j <= i; ++j) {
                        double sv = (drop_s[i] != 0.0 || drop_s[j] != 0.0) ? (i == j ? 1.0 : 0.0)
                                                                            : gt_s[i * LD + j] * dinv_s[i] * dinv_s[j];
                        for (int q = 0; q < j; ++q) sv -= lm_s[i * LD + q] * lm_s[j * LD + q];
                        if (i == j) {
                            if (!(sv > 1e-14)) {  // no independent part left in column i
                                drop_s[i] = 1.0;
                                for (int q = 0; q < i; ++q) lm_s[i * LD + q] = 0.0;
                                sv = 1.0;
                            }
                            lm_s[i * LD + i] = sqrt(sv);
                        } else {
                            lm_s[i * LD + j] = sv / lm_s[j * LD + j];
                        }
                    }
                }
                for (int i = 0; i < ka; ++i) {
                    double sv = drop_s[i] != 0.0 ? 0.0 : dots_s[ka + i] * dinv_s[i];
                    for (int q = 0; q < i; ++q) sv -= lm_s[i * LD + q] * ys_s[q];
                    ys_s[i] = sv / lm_s[i * LD + i];
                }
                for (int i = ka - 1; i >= 0; --i) {
                    double sv = ys_s[i];
                    for (int q = i + 1; q < ka; ++q) sv -= lm_s[q * LD + i] * xs_s[q];
                    xs_s[i] = drop_s[i] != 0.0 ? 0.0 : sv / lm_s[i * LD + i];
                }
                for (int i = 0; i < ka; ++i) xs_s[i] *= dinv_s[i];
                for (int i = 0; i < R; ++i) a.coef[((size_t)prob * R + i) * R + comp] = i < ka ? xs_s[i] : 0.0;
                a.trips[(size_t)prob * R + comp] = trip;
                a.conv[(size_t)prob * R + comp] = done_trip >= 0 ? 1 : 0;
            }
            __syncthreads();
            // ---- Y deflation (tpls.py:113) and ||Y||^2 ----
            {
                double ssy = 0.0;
                for (int i = tid; i < n; i += NTH) {
                    double sv = 0.0;
                    for (int b = 0; b < ka; ++b) sv = fma(Tw[(size_t)b * n + i], xs_s[b], sv);
                    const double sw = wr != nullptr ? wr[i] : 1.0;
                    if (sw == 0.0) continue;  // a held-out row of Y stays 0
                    double rs = 0.0;
                    for (int c = 0; c < M; ++c) {
                        const double yv = fma(-sv, q_s[c], Yw[(size_t)i * M + c]);
                        Yw[(size_t)i * M + c] = yv;
                        rs = fma(yv, yv, rs);
                    }
                    ssy += rs;
                }
                ssy = block_sum(ssy, red);
                if (tid == 0) ssy_s[comp + 1] = ssy;
            }
            // ---- X deflation (tpls.py:109) fused with ||X||^2; after the last component the norm alone ----
            const bool write = comp + 1 < R;
            for (int l = 0; l < L; ++l) {
                const BatchTensor& X = a.x[l];
                void* xw = ws + X.off_x;
                const double* wk = reinterpret_cast<const double*>(ws + X.off_wk);
                const int p = X.p, dt = X.dtype;
                const size_t np = (size_t)n * p;
                double ss = 0.0;
                for (size_t e = tid; e < np; e += NTH) {
                    const int i = (int)(e / p), c = (int)(e - (size_t)i * p);
                    const double x = ldx(xw, dt, e);
                    double xd = fma(-Ta[i], wk[c], x);
                    if (write) xd = stx(xw, dt, e, xd);  // NaN stays NaN
                    if (masked_s[l] && !(x == x)) xd = 0.0;
                    const double sw = wr != nullptr ? wr[i] : 1.0;
                    if (sw != 0.0) ss = fma(xd, xd, ss);
                }
                ss = block_sum(ss, red);
                if (tid == 0) ss_s[l * (R + 1) + comp + 1] = ss;
            }
            __syncthreads();
        }
        // ---- R2X / R2Y (SURVEY.md §0.4) ----
        for (int e = tid; e < (L + 1) * R; e += NTH) {
            const int l = e / R, c = e - l * R;
            if (l < L)
                a.r2x[((size_t)prob * L + l) * R + c] = 1.0 - ss_s[l * (R + 1) + c + 1] / ss_s[l * (R + 1)];
            else
                a.r2y[(size_t)prob * R + c] = 1.0 - ssy_s[c + 1] / ssy_s[0];
        }
        __syncthreads();
    }
}

}  // namespace

size_t batch_fit_smem_limit() {
    static const size_t lim = [] {
        cudaFuncAttributes fa{};
        int dev = 0, optin = 0;
        if (cudaFuncGetAttributes(&fa, batch_fit_kernel) != cudaSuccess || cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
            return (size_t)0;
        return (size_t)optin > fa.sharedSizeBytes ? (size_t)optin - fa.sharedSizeBytes : (size_t)0;
    }();
    return lim;
}

int batch_fit_max_ctas(size_t smem_bytes) {
    int dev = 0, sms = 0, per_sm = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return 0;
    if (cudaFuncSetAttribute(batch_fit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes) != cudaSuccess)
        return 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, batch_fit_kernel, kRank1Threads, smem_bytes) != cudaSuccess)
        return 0;
    return per_sm * sms;
}

cudaError_t launch_batch_fit(const BatchArgs& a, int grid, size_t smem_bytes, cudaStream_t s) {
    if (a.n_tensors < 1 || a.n_tensors > kMaxTensors || a.m < 1 || a.m > kBatchMaxResp || a.R < 1 || a.R > kBatchMaxComp ||
        grid < 1)
        return cudaErrorInvalidValue;
    cudaError_t e = cudaFuncSetAttribute(batch_fit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    if (e != cudaSuccess) return e;
    launch_k(batch_fit_kernel, dim3(grid), dim3(kRank1Threads), smem_bytes, s, a);
    return cudaGetLastError();
}

}  // namespace tpls
