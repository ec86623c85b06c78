// The single-CTA rank-1 step (rank1_task) and the block-level helpers it is built from, shared by the kernels
// that run it: rank1_kernel, cov_loop_kernel and resident_loop_kernel (rank1.cu) and batch_fit_kernel (batch.cu).
// Internal linkage: every translation unit that includes it gets its own copy of these inline device functions.
#pragma once

#include "rank1.cuh"

namespace tpls {

namespace {

constexpr int NTH = kRank1Threads;
constexpr int NWARP = NTH / 32;

__host__ __device__ inline int up4(int v) { return (v + 3) & ~3; }
__host__ __device__ inline int up8(int v) { return (v + 7) & ~7; }
// Leading dimension of a padded matrix of order v.  Orders are padded to a multiple of 8 (the fp64 MMA tile) and
// the rows by 4 more doubles: ld = 4 or 12 (mod 16), so the four k-rows x four columns a half-warp touches in one
// fragment load (address = k * ld + column) fall on 16 different bank pairs.
__host__ __device__ inline int ldp(int v) { return up8(v) + 4; }

// Workspace of the HOSVD start of one mode of a >= 3-way Z (doubles): the unfolding copy, the Gram matrix and
// the two squaring buffers, two vectors.  Every mode has its own area because the modes are worked on
// concurrently by different thread groups.
struct ModeWs {
    int n;       // order of the Gram matrix: min(dk, mk)
    int ld;      // its leading dimension
    int mt;      // doubles of the unfolding copy
    int gram;    // doubles of ONE n4 x ld matrix
    int vec;     // doubles of one work vector
    int total;
};
__host__ __device__ inline ModeWs mode_ws(int dk, int mk) {
    ModeWs w;
    w.n = dk <= mk ? dk : mk;
    w.ld = ldp(w.n);
    w.mt = up4((dk <= mk ? mk : dk) * w.ld);
    w.gram = up8(w.n) * w.ld;
    w.vec = up4(dk);
    w.total = w.mt + 3 * w.gram + 2 * w.vec;
    return w;
}

// A group of warps of the CTA that synchronises on its own named barrier: the whole CTA (barrier 0, i.e.
// __syncthreads) or one slice of it per mode during the HOSVD start.  Block-wide sums take ONE barrier: warp
// partials go to one of two alternating buffers, every thread then folds the partials itself.
struct Grp {
    int tid, nth, bar;
    double* red;  // [2][2*NWARP]
    int* ired;    // [2][NWARP]
    int flip;
    long long* dbg;  // optional diagnostics (clock64 accumulators), nullptr in normal use
    __device__ __forceinline__ void sync() const { named_bar_sync(bar, nth); }
    __device__ __forceinline__ void tick(int slot, long long t0) const {
        if (dbg != nullptr && tid == 0) dbg[slot] += clock64() - t0;
    }
};

__device__ __forceinline__ double bsum(double v, Grp& g) {
    v = warp_sum(v);
    double* r = g.red + g.flip * 2 * NWARP;
    if ((g.tid & 31) == 0) r[g.tid >> 5] = v;
    g.sync();
    double t = 0.0;
    const int nw = g.nth >> 5;
    for (int q = 0; q < nw; ++q) t += r[q];
    g.flip ^= 1;
    return t;
}

// the same for two values that only lane 0 of every warp holds (no warp-level fold needed)
__device__ __forceinline__ void bsum2_lane0(double& v1, double& v2, Grp& g) {
    double* r = g.red + g.flip * 2 * NWARP;
    if ((g.tid & 31) == 0) {
        r[g.tid >> 5] = v1;
        r[NWARP + (g.tid >> 5)] = v2;
    }
    g.sync();
    double t1 = 0.0, t2 = 0.0;
    const int nw = g.nth >> 5;
    for (int q = 0; q < nw; ++q) {
        t1 += r[q];
        t2 += r[NWARP + q];
    }
    g.flip ^= 1;
    v1 = t1;
    v2 = t2;
}

// index of the first entry with the largest |a[i]|
__device__ __forceinline__ int argmax_abs(const double* a, int n, Grp& g) {
    double bv = -1.0;
    int bi = 0x7fffffff;
    for (int i = g.tid; i < n; i += g.nth) {
        const double v = fabs(a[i]);
        if (v > bv) {
            bv = v;
            bi = i;
        }
    }
    for (int m = 16; m >= 1; m >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, bv, m);
        const int oi = __shfl_xor_sync(0xffffffffu, bi, m);
        if (ov > bv || (ov == bv && oi < bi)) {
            bv = ov;
            bi = oi;
        }
    }
    double* r = g.red + g.flip * 2 * NWARP;
    int* ir = g.ired + g.flip * NWARP;
    if ((g.tid & 31) == 0) {
        r[g.tid >> 5] = bv;
        ir[g.tid >> 5] = bi;
    }
    g.sync();
    bv = r[0];
    bi = ir[0];
    const int nw = g.nth >> 5;
    for (int q = 1; q < nw; ++q) {
        const double ov = r[q];
        const int oi = ir[q];
        if (ov > bv || (ov == bv && oi < bi)) {
            bv = ov;
            bi = oi;
        }
    }
    g.flip ^= 1;
    return bi;
}

__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c0), "+d"(c1)
                 : "d"(a), "d"(b));
}

// C = scale * Mt^T Mt on the leading n8 x n8 block (n8 % 8 == 0; Mt is krows x n8 with leading dimension ldm, C has
// leading dimension ldc).  C is symmetric: only the 8x8 tiles on or above the diagonal are computed, then mirrored.
// TRACE: returns trace(C) through one group reduction whose barrier also publishes C.  On the fp64 tensor-core path
// (mma.sync.m8n8k4.f64, SASS DMMA): one 8x8 tile on or above the diagonal per warp and round, the contraction in
// steps of 8 rows of Mt on two accumulator pairs.  A 4x4 register tile of DFMAs needs an LDS.128 per 4 FMAs and is
// bound by shared-memory issue (tools/micro/fp64_lat.cu); a DMMA does 256 FMAs for two conflict-free LDS.64, so a
// 64 x 64 squaring drops from ~7.7 k cycles to the ~2.5 k of the fp64 pipe itself.  Rows of Mt past krows are
// treated as zero; pad columns of Mt must BE zero.  Fixed association order => bit-reproducible.
template <bool TRACE>
__device__ __forceinline__ double syrk_dmma(double* __restrict__ C, int ldc, const double* __restrict__ Mt, int ldm, int krows,
                                            int n8, double scale, Grp& g) {
    const int nt = n8 >> 3;
    const int ntri = (nt * (nt + 1)) >> 1;
    const int warp = g.tid >> 5, lane = g.tid & 31, nw = g.nth >> 5;
    const int gq = lane >> 2, t4 = lane & 3;
    double tr = 0.0;
    for (int t = warp; t < ntri; t += nw) {  // warp-uniform: the MMAs stay converged
        int ti = 0, rem = t, len = nt;
        while (rem >= len) {
            rem -= len;
            --len;
            ++ti;
        }
        const int tj = ti + rem;
        // four independent accumulator pairs: with four warps per sub-partition that keeps 16 MMAs in flight
        double acc[4][2] = {{0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}, {0.0, 0.0}};
        const double* pa = Mt + 8 * ti + gq;   // A[i][k] = Mt[k][8 ti + i]
        const double* pb = Mt + 8 * tj + gq;   // B[k][j] = Mt[k][8 tj + j]
        for (int k = 0; k < krows; k += 16) {
            double av[4], bv[4];
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int kk = k + 4 * c + t4;
                const bool in = kk < krows;
                av[c] = in ? pa[kk * ldm] : 0.0;
                bv[c] = in ? pb[kk * ldm] : 0.0;
            }
#pragma unroll
            for (int c = 0; c < 4; ++c) dmma884(acc[c][0], acc[c][1], av[c], bv[c]);
        }
        const double c0 = ((acc[0][0] + acc[1][0]) + (acc[2][0] + acc[3][0])) * scale;
        const double c1 = ((acc[0][1] + acc[1][1]) + (acc[2][1] + acc[3][1])) * scale;
        // this lane holds C[8 ti + gq][8 tj + 2 t4 + {0, 1}]
        *reinterpret_cast<double2*>(C + (size_t)(8 * ti + gq) * ldc + 8 * tj + 2 * t4) = make_double2(c0, c1);
        if (ti != tj) {
            C[(size_t)(8 * tj + 2 * t4) * ldc + 8 * ti + gq] = c0;
            C[(size_t)(8 * tj + 2 * t4 + 1) * ldc + 8 * ti + gq] = c1;
        } else if (TRACE) {
            if (gq == 2 * t4) tr += c0;
            if (gq == 2 * t4 + 1) tr += c1;
        }
    }
    if (TRACE) return bsum(tr, g);
    g.sync();
    return 0.0;
}

// y[i] = sum_{j < cols} M[i*ld + j] * x[j], i < rows: 8 lanes per row
__device__ __forceinline__ void matvec8(double* y, const double* M, int ld, const double* x, int rows, int cols, const Grp& g) {
    const int part = g.tid & 7, r0 = g.tid >> 3;
    for (int rb = 0; rb < rows; rb += g.nth / 8) {
        const int i = rb + r0;
        double s = 0.0;
        if (i < rows)
            for (int j = part; j < cols; j += 8) s = fma(M[(size_t)i * ld + j], x[j], s);
        s += shfl_xor_d(s, 4);
        s += shfl_xor_d(s, 2);
        s += shfl_xor_d(s, 1);
        if (i < rows && part == 0) y[i] = s;
    }
    g.sync();
}

__device__ __forceinline__ double vec_dot(const double* a, const double* b, int n, Grp& g) {
    double s = 0.0;
    for (int i = g.tid; i < n; i += g.nth) s = fma(a[i], b[i], s);
    return bsum(s, g);
}

// dst = src / ||src||; returns ||src||
__device__ __forceinline__ double normalize_into(double* dst, const double* src, int n, Grp& g) {
    double s = 0.0;
    for (int i = g.tid; i < n; i += g.nth) s = fma(src[i], src[i], s);
    const double nv = sqrt(bsum(s, g));
    for (int i = g.tid; i < n; i += g.nth) dst[i] = src[i] / nv;
    g.sync();
    return nv;
}

// Leading eigenpair of the symmetric PSD matrix G (order n, stored up8(n) x up8(n) with zero pads, leading
// dimension ld).  A, B: work buffers of the same shape.  v (n) receives the unit eigenvector; returns the
// eigenvalue when asked for it.
__device__ __forceinline__ double lead_eig(const double* G, double* A, double* B, double* v, double* tmp, int n, int ld, Grp& g,
                                           int polish, bool want_lambda) {
    const int n8 = up8(n);
    double s = 0.0;
    for (int i = g.tid; i < n; i += g.nth) s += G[(size_t)i * ld + i];
    const double tr = bsum(s, g);
    if (!(tr > 0.0)) {
        for (int i = g.tid; i < n; i += g.nth) v[i] = 0.0;
        g.sync();
        return 0.0;
    }
    const double* src = G;
    double* dst = A;
    double* oth = B;
    double scale = (1.0 / tr) * (1.0 / tr);
    const long long c0 = g.dbg != nullptr ? clock64() : 0;
    for (int it = 0; it < 64; ++it) {
        // dst = (src / tr(src))^2; tau = its trace = sum of squared normalised eigenvalues, -> 1 at rank one
        const double tau = syrk_dmma<true>(dst, ld, src, ld, n8, n8, scale, g);
        if (g.dbg != nullptr && g.tid == 0) g.dbg[12] += 1;
        src = dst;
        double* sw = dst;
        dst = oth;
        oth = sw;
        if (1.0 - tau < 1e-7) break;
        scale = (1.0 / tau) * (1.0 / tau);
    }
    g.tick(13, c0);
    const long long c1 = g.dbg != nullptr ? clock64() : 0;
    // src ~ v v^T: take the column with the largest diagonal entry
    for (int i = g.tid; i < n; i += g.nth) tmp[i] = src[(size_t)i * ld + i];
    g.sync();
    const int bi = argmax_abs(tmp, n, g);
    for (int i = g.tid; i < n; i += g.nth) tmp[i] = src[(size_t)i * ld + bi];
    g.sync();
    normalize_into(v, tmp, n, g);
    // polish against the original matrix
    double nv = 0.0;
    for (int q = 0; q < polish; ++q) {
        matvec8(tmp, G, ld, v, n, n, g);
        nv = normalize_into(v, tmp, n, g);
    }
    g.tick(14, c1);
    if (!want_lambda) return 0.0;
    if (polish > 0) return nv;  // ||G v|| of the last step: the eigenvalue to the accuracy of v (quadratic in its error)
    matvec8(tmp, G, ld, v, n, n, g);
    return vec_dot(tmp, v, n, g);
}

__device__ __forceinline__ void flip_to_positive_peak(double* f, int n, Grp& g) {
    const int i = argmax_abs(f, n, g);
    const bool neg = f[i] < 0.0;
    g.sync();
    if (neg)
        for (int q = g.tid; q < n; q += g.nth) f[q] = -f[q];
    g.sync();
}

struct Geo {  // mode-k unfolding geometry
    int dk, mk, ik;
};

__device__ __forceinline__ Geo mode_geo(const Rank1Task& T, int k) {
    Geo g;
    g.dk = T.dims[k];
    g.ik = 1;
    for (int m = k + 1; m < T.nmodes; ++m) g.ik *= T.dims[m];
    g.mk = T.p / g.dk;
    return g;
}

// flat index of element (a, j) of the mode-k unfolding (tensorly convention: remaining modes in C order)
__device__ __forceinline__ int unf_index(const Geo& g, int a, int j) {
    const int o = j / g.ik;
    const int in = j - o * g.ik;
    return (o * g.dk + a) * g.ik + in;
}

// f[a] = sum_j Zk(a, j) * x[j]   (general mode, strided)
__device__ __forceinline__ void unf_matvec(double* f, const double* zs, const Geo& geo, const double* x, const Grp& g) {
    const int lane = g.tid & 31, w = g.tid >> 5, nw = g.nth >> 5;
    for (int a = w; a < geo.dk; a += nw) {
        double s = 0.0;
        for (int j = lane; j < geo.mk; j += 32) s = fma(zs[unf_index(geo, a, j)], x[j], s);
        s = warp_sum(s);
        if (lane == 0) f[a] = s;
    }
    g.sync();
}

// HOSVD start of ONE mode (tensorly initialize_cp, init="svd"): the leading left singular vector of the mode-k
// unfolding, sign fixed so that its largest-|entry| is positive.  Runs on the thread group g with the group's
// own workspace w; returns the singular value (wanted for mode 0 only, which carries sigma into the weights).
__device__ __forceinline__ double hosvd_mode(const double* zs, const Geo& geo, double* fk, double* w, Grp& g, bool want_sigma) {
    const ModeWs m = mode_ws(geo.dk, geo.mk);
    double* mt = w;
    double* G = mt + m.mt;
    double* A = G + m.gram;
    double* B = A + m.gram;
    double* tmp = B + m.gram;
    double* tmp2 = tmp + m.vec;
    const int n8 = up8(m.n), ld = m.ld;
    double sigma = 0.0;
    if (geo.dk <= geo.mk) {
        // Mt[j][a] = Zk(a, j): rows are the columns of the unfolding
        for (int i = g.tid; i < geo.mk * n8; i += g.nth) {
            const int j = i / n8, a = i - j * n8;
            mt[(size_t)j * ld + a] = a < geo.dk ? zs[unf_index(geo, a, j)] : 0.0;
        }
        g.sync();
        syrk_dmma<false>(G, ld, mt, ld, geo.mk, n8, 1.0, g);
        const double lam = lead_eig(G, A, B, fk, tmp, geo.dk, ld, g, 2, want_sigma);
        sigma = sqrt(lam);
    } else {
        // tall unfolding: eigenvector of the small side, then one multiplication by the unfolding
        for (int i = g.tid; i < geo.dk * n8; i += g.nth) {
            const int a = i / n8, j = i - a * n8;
            mt[(size_t)a * ld + j] = j < geo.mk ? zs[unf_index(geo, a, j)] : 0.0;
        }
        g.sync();
        syrk_dmma<false>(G, ld, mt, ld, geo.dk, n8, 1.0, g);
        lead_eig(G, A, B, tmp2, tmp, geo.mk, ld, g, 2, false);
        unf_matvec(tmp, zs, geo, tmp2, g);
        sigma = normalize_into(fk, tmp, geo.dk, g);
    }
    flip_to_positive_peak(fk, geo.dk, g);
    return sigma;
}

struct AlsIn {
    const double* zs;
    const double* zc;  // row-major copies of the unfoldings of modes 1.. (mode 0 is Z itself), up4(p) doubles each
    const unsigned short* dig_tab;
    double weight, normz2, normz, tol;
    int normalize_on_break;
    double* mode_out;  // [2][kMaxZModes] shared scratch of the renormalisation
};

// Rank-1 ALS sweeps of tensorly's parafac for an NM-way Z (NM >= 3), starting from the factors in f (norms^2 in
// nrm2_in, weight in in.weight).  One barrier per mode update and one per renormalisation:
//   * a warp per row a of the mode-k unfolding: factor[a] = weight * <Zk(a, :), prod of the other factors> / gram,
//     columns striding over the lanes (every unfolding is kept row-major, so the reads are conflict-free), the
//     other-mode indices of a column from a table;
//   * lane 0 of the warp finishes the row and keeps ||factor||^2 and <mttkrp, factor> partials, which meet in
//     one block-wide sum;
//   * cp_normalize: warp m rescales factor m and takes its new squared norm.
// NM and the mode being updated are compile-time constants, so every per-mode quantity is a register.
// Returns the number of sweeps.
template <int NM>
__device__ __forceinline__ int als_sweeps(const Rank1Task& T, double* const fb, const double* nrm2_in, const AlsIn& in, Grp& cta) {
    constexpr int DG = 4 * ((NM - 1 + 3) / 4);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    // factor m lives at fb[fo[m] ...]: ONE base pointer derived from the workspace plus integer offsets, so that
    // the compiler keeps seeing a shared-memory address (pointers kept in an array or a struct turn every factor
    // access into a generic load)
    int fo[NM];
    int dims[NM], mk[NM], tb[NM];
    double nrm2[NM];
#pragma unroll
    for (int m = 0; m < NM; ++m) {
        dims[m] = T.dims[m];
        nrm2[m] = nrm2_in[m];
    }
    fo[0] = 0;
#pragma unroll
    for (int m = 1; m < NM; ++m) fo[m] = fo[m - 1] + dims[m - 1];
    tb[0] = 0;
#pragma unroll
    for (int m = 0; m < NM; ++m) {
        mk[m] = T.p / dims[m];
        if (m + 1 < NM) tb[m + 1] = tb[m] + mk[m];
    }
    double weight = in.weight;
    double err_prev = 0.0;
    int sweeps = 0;
    for (int it = 0; it < 100; ++it) {
        ++sweeps;
        double iprod = 0.0;
#pragma unroll
        for (int k = 0; k < NM; ++k) {
            double gram = weight * weight;
#pragma unroll
            for (int m = 0; m < NM; ++m)
                if (m != k) gram *= nrm2[m];
            double s1 = 0.0, s2 = 0.0;
            const long long c0 = cta.dbg != nullptr ? clock64() : 0;
            // rows of the mode-k unfolding are contiguous: consecutive lanes read consecutive doubles
            const double* zk = k == 0 ? in.zs : in.zc + (size_t)(k - 1) * up4(T.p);
            const unsigned short* digk = in.dig_tab + (size_t)tb[k] * DG;
            for (int a = wid; a < dims[k]; a += NWARP) {
                const double* zrow = zk + (size_t)a * mk[k];
                double acc = 0.0;
#pragma unroll 4
                for (int j = lane; j < mk[k]; j += 32) {
                    unsigned short dg[DG];
                    if (DG == 4) {
                        const uint2 w = *reinterpret_cast<const uint2*>(digk + (size_t)j * DG);
                        dg[0] = (unsigned short)(w.x & 0xffffu);
                        dg[1] = (unsigned short)(w.x >> 16);
                        dg[2] = (unsigned short)(w.y & 0xffffu);
                        dg[3] = (unsigned short)(w.y >> 16);
                    } else {
                        const uint4 w = *reinterpret_cast<const uint4*>(digk + (size_t)j * DG);
                        const unsigned int ww[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            dg[2 * q] = (unsigned short)(ww[q] & 0xffffu);
                            dg[2 * q + 1] = (unsigned short)(ww[q] >> 16);
                        }
                    }
                    double pr = 1.0;
#pragma unroll
                    for (int m = 0; m < NM; ++m) {
                        if (m == k) continue;
                        const int slot = m < k ? m : m - 1;
                        pr *= fb[fo[m] + dg[slot]];
                    }
                    acc = fma(zrow[j], pr, acc);
                }
                acc = warp_sum(acc);
                if (lane == 0) {
                    const double mt_i = acc * weight;
                    const double fi = mt_i / gram;
                    fb[fo[k] + a] = fi;
                    s1 = fma(fi, fi, s1);
                    s2 = fma(mt_i, fi, s2);  // <mttkrp, factor>, wanted for the last mode only
                }
            }
            cta.tick(8, c0);
            const long long c1 = cta.dbg != nullptr ? clock64() : 0;
            bsum2_lane0(s1, s2, cta);
            cta.tick(9, c1);
            nrm2[k] = s1;
            if (k == NM - 1) iprod = s2;
        }
        const long long c2 = cta.dbg != nullptr ? clock64() : 0;
        double fn2 = weight * weight;
#pragma unroll
        for (int m = 0; m < NM; ++m) fn2 *= nrm2[m];
        const double err = sqrt(fabs(in.normz2 + fn2 - 2.0 * iprod)) / in.normz;
        const bool stop = it >= 1 && fabs(err_prev - err) < in.tol;
        err_prev = err;
        if (stop && !in.normalize_on_break) break;
        // cp_normalize: weights into factor 0, then every column norm back into the weights
        const double w_in = weight;
        double sc[NM];
        weight = 1.0;
#pragma unroll
        for (int m = 0; m < NM; ++m) {
            sc[m] = sqrt(nrm2[m]) * (m == 0 ? fabs(w_in) : 1.0);
            weight *= sc[m];
        }
        double* mo = in.mode_out + (it & 1) * kMaxZModes;  // two alternating buffers: one barrier per renormalisation
#pragma unroll
        for (int m = 0; m < NM; ++m) {
            if (wid == m) {
                const double dv = sc[m] == 0.0 ? 1.0 : sc[m];
                double q = 0.0;
                for (int i = lane; i < dims[m]; i += 32) {
                    const double v = (m == 0 ? fb[fo[m] + i] * w_in : fb[fo[m] + i]) / dv;
                    fb[fo[m] + i] = v;
                    q = fma(v, v, q);
                }
                q = warp_sum(q);
                if (lane == 0) mo[m] = q;
            }
        }
        __syncthreads();
#pragma unroll
        for (int m = 0; m < NM; ++m) nrm2[m] = mo[m];
        cta.tick(10, c2);
        if (stop) break;
    }
    return sweeps;
}

// wkron_alt: a second destination for kron(w) (the resident loop's shared-memory copy); publish = false keeps the
// task's outputs out of global memory (every CTA of the resident loop runs the task, one of them publishes).
__device__ __forceinline__ void rank1_task(const Rank1Task& T, double tol, int normalize_on_break, double* ws,
                                           double* wkron_alt = nullptr, bool publish = true) {
    __shared__ double red[(kMaxZModes + 1) * 4 * NWARP];
    __shared__ int ired[(kMaxZModes + 1) * 2 * NWARP];
    __shared__ double mode_out[2 * kMaxZModes];  // per mode: ||f||^2 of the start, sigma
    Grp cta{(int)threadIdx.x, NTH, 0, red, ired, 0, T.stamps};
    if (T.stamps != nullptr && threadIdx.x == 0)
        for (int i = 8; i < 16; ++i) T.stamps[i] = 0;
    const int p = T.p;
    const int nm = T.nmodes;
#define TPLS_STAMP(i) \
    if (T.stamps != nullptr && threadIdx.x == 0) T.stamps[i] = clock64()

    int sumd = 0, maxd = 0;
    for (int m = 0; m < nm; ++m) {
        sumd += T.dims[m];
        maxd = max(maxd, T.dims[m]);
    }

    TPLS_STAMP(0);
    if (nm == 1) {
        double* zs = ws;
        double s = 0.0;
        for (int i = threadIdx.x; i < p; i += NTH) {
            double z = T.z[i];
            if (T.colcnt != nullptr) {
                const double c = T.colcnt[i];
                z = c > 0.0 ? z / c * T.n_total : 0.0;
            }
            zs[i] = z;
            s = fma(z, z, s);
        }
        const double normz = sqrt(bsum(s, cta));
        for (int i = threadIdx.x; i < T.pitch; i += NTH) {
            const double w = i < p ? zs[i] / normz : 0.0;
            if (publish) {
                if (i < p) T.w[0][i] = w;
                T.wkron[i] = w;
            }
            if (wkron_alt != nullptr) wkron_alt[i] = w;
        }
        if (publish && threadIdx.x == 0 && T.sweeps) *T.sweeps = 0;
        return;
    }

    // workspace carve-up (doubles); see rank1_workspace_doubles
    double* zs = ws;                 // Z (nm == 2: row-padded d0 x ldp(d1))
    double* fac = zs + T.zs_len;     // the factor vectors, back to back
    double* rest = fac + up4(sumd);  // nm == 2: Z^T, Gram, squaring buffers, vector; nm >= 3: per-mode areas, tables
    // ---- load Z (with the observed-count rescaling of missingvals.py:18 when masked) ----
    const int d0 = T.dims[0], d1 = nm == 2 ? T.dims[1] : 0;
    const int ld0 = ldp(d0), ld1 = ldp(d1);
    double* mt2 = rest;  // nm == 2: padded Z^T
    double s = 0.0;
    if (nm == 2) {
        // padded row-major Z in zs and padded Z^T in mt2 (the pads up to a multiple of eight are read as zeros)
        if (up8(d1) != d1)
            for (int i = threadIdx.x; i < d0 * ld1; i += NTH) zs[i] = 0.0;
        if (up8(d0) != d0)
            for (int i = threadIdx.x; i < d1 * ld0; i += NTH) mt2[i] = 0.0;
        if (up8(d1) != d1 || up8(d0) != d0) __syncthreads();
    }
    // eight loads per thread in flight (a plain loop issued them one L2 round trip after the other)
    for (int base = 0; base < p; base += NTH * 8) {
        double zv[8], cv[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int i = base + q * NTH + (int)threadIdx.x;
            zv[q] = i < p ? T.z[i] : 0.0;  // plain load: the covariance loop rewrites Z between calls
            cv[q] = (T.colcnt != nullptr && i < p) ? __ldg(T.colcnt + i) : 1.0;
        }
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int i = base + q * NTH + (int)threadIdx.x;
            if (i >= p) continue;
            double z = zv[q];
            if (T.colcnt != nullptr) z = cv[q] > 0.0 ? z / cv[q] * T.n_total : 0.0;
            s = fma(z, z, s);
            if (nm == 2) {
                const int a = i / d1, j = i - a * d1;
                zs[(size_t)a * ld1 + j] = z;
                mt2[(size_t)j * ld0 + a] = z;
            } else {
                zs[i] = z;
            }
        }
    }
    const double normz2 = bsum(s, cta);
    const double normz = sqrt(normz2);

    TPLS_STAMP(1);
    int sweeps = 0;
    const unsigned short* dig0 = nullptr;  // nm >= 3: per column of the mode-0 unfolding, the indices of modes 1..
    if (nm == 2) {
        // ---- matrix Z: the rank-1 CP is the leading singular pair ----
        // tensorly starts ALS from the exact SVD, which is already the fixed point: its two sweeps leave
        // the pair where it is and only settle the sign -- the LAST mode keeps the "largest-|entry|
        // positive" convention of the start, mode 0 follows from Z.  So: one eigenproblem on the short
        // side, the sign rule on f1, then one power step each way (= one ALS sweep) as a polish.
        const int ks = d0 <= d1 ? 0 : 1;
        const int n = T.dims[ks], no = T.dims[1 - ks];
        const int ldg = ldp(n);
        const size_t n2 = (size_t)up8(n) * ldg;
        double* G = mt2 + T.mt_len;
        double* A = G + n2;
        double* B = A + n2;
        double* tmp = B + n2;
        // rows of Mt are the columns of the mode-ks unfolding: Z^T for ks == 0, Z for ks == 1
        const double* Mt = ks == 0 ? mt2 : zs;
        double* const f0 = fac;        // the two factor vectors, back to back
        double* const f1 = fac + d0;
        // Tiny matrices (Gram order <= 8: one 8x8 tile; vectors of <= 32 entries) run on ONE warp: every step below
        // is a short dependent chain, and with the whole CTA each of the ~35 steps paid a 16-warp barrier and a
        // 16-entry fold for work that fits one lane each (8 x 6: 13.0 -> 11.6 us; from order 16 on the 8-lane
        // matrix-vector passes and the tiles one after the other cost more than the barriers: 32 x 16 12.5 -> 15 us).
        const bool one_warp = up8(n) <= 8 && no <= 32;
        Grp w0{(int)threadIdx.x, 32, 1, red + 4 * NWARP, ired + 2 * NWARP, 0, T.stamps};
        Grp& g = one_warp ? w0 : cta;
        if (!one_warp || threadIdx.x < 32) {
            syrk_dmma<false>(G, ldg, Mt, ks == 0 ? ld0 : ld1, no, up8(n), 1.0, g);
            lead_eig(G, A, B, ks == 0 ? f0 : f1, tmp, n, ldg, g, /*polish=*/1, /*want_lambda=*/false);
            TPLS_STAMP(2);
            if (ks == 0) {
                matvec8(tmp, mt2, ld0, f0, d1, d0, g);
                normalize_into(f1, tmp, d1, g);
            }
            flip_to_positive_peak(f1, d1, g);
            matvec8(tmp, zs, ld1, f1, d0, d1, g);
            normalize_into(f0, tmp, d0, g);
            matvec8(tmp, mt2, ld0, f0, d1, d0, g);
            normalize_into(f1, tmp, d1, g);
        }
        if (one_warp) __syncthreads();
        sweeps = 2;
        TPLS_STAMP(3);
    } else {
        // ---- HOSVD start: the modes are independent, one slice of the CTA each, concurrently ----
        const int gsz = max(32, (NTH / nm) & ~31);
        const int my_mode = threadIdx.x / gsz;
        {
            int woff = 0, foff = 0;
            for (int k = 0; k < nm; ++k) {
                const Geo geo = mode_geo(T, k);
                double* const fk = fac + foff;
                if (k == my_mode) {
                    Grp g{(int)threadIdx.x - k * gsz, gsz, 1 + k, red + (1 + k) * 4 * NWARP, ired + (1 + k) * 2 * NWARP, 0,
                          k == 0 ? T.stamps : nullptr};
                    const double sigma = hosvd_mode(zs, geo, fk, rest + woff, g, k == 0);
                    const double n2k = vec_dot(fk, fk, geo.dk, g);
                    if (g.tid == 0) {
                        mode_out[2 * k] = n2k;
                        mode_out[2 * k + 1] = sigma;
                    }
                }
                woff += mode_ws(geo.dk, geo.mk).total;
                foff += geo.dk;
            }
        }
        __syncthreads();
        TPLS_STAMP(2);
        double weight = mode_out[1];
        double nrm2[kMaxZModes];
        for (int m = 0; m < kMaxZModes; ++m) nrm2[m] = m < nm ? mode_out[2 * m] : 1.0;

        // ---- for the sweeps (the per-mode areas are free again): per mode k and column j of its unfolding the
        //      indices of the other modes (16 bits each, padded to 4 or 8 per column so that one 64/128-bit load
        //      fetches them), and a row-major copy of every unfolding but the first (Z itself) -- read column-wise
        //      out of Z, the last mode's rows would put all lanes of a warp on two banks ----
        const int DG = 4 * ((nm - 1 + 3) / 4);
        unsigned short* dig_tab = reinterpret_cast<unsigned short*>(rest);
        double* zc = rest + up4((int)(((size_t)up4(T.tab_cols) * DG * 2 + 7) / 8));
        dig0 = dig_tab;
        {
            int tbase = 0;
            for (int k = 0; k < nm; ++k) {
                const Geo geo = mode_geo(T, k);
                for (int j = threadIdx.x; j < geo.mk; j += NTH) {
                    int rem = j, slot = nm - 2;
                    for (int m = nm - 1; m >= 0; --m) {
                        if (m == k) continue;
                        const int d = T.dims[m];
                        dig_tab[(size_t)(tbase + j) * DG + slot] = (unsigned short)(rem % d);
                        rem /= d;
                        --slot;
                    }
                }
                if (k > 0) {
                    double* zk = zc + (size_t)(k - 1) * up4(p);
                    for (int i = threadIdx.x; i < p; i += NTH) {
                        const int a = i / geo.mk, j = i - a * geo.mk;
                        zk[i] = zs[unf_index(geo, a, j)];
                    }
                }
                tbase += geo.mk;
            }
        }
        __syncthreads();
        TPLS_STAMP(3);

        // ---- ALS sweeps (tensorly parafac, rank 1), mode count known at compile time ----
        AlsIn in{zs, zc, dig_tab, weight, normz2, normz, tol, normalize_on_break, mode_out};
        switch (nm) {
            case 3: sweeps = als_sweeps<3>(T, fac, nrm2, in, cta); break;
            case 4: sweeps = als_sweeps<4>(T, fac, nrm2, in, cta); break;
            case 5: sweeps = als_sweeps<5>(T, fac, nrm2, in, cta); break;
            case 6: sweeps = als_sweeps<6>(T, fac, nrm2, in, cta); break;
            default: sweeps = als_sweeps<7>(T, fac, nrm2, in, cta); break;
        }
    }

    TPLS_STAMP(4);
    // ---- publish ----
    if (publish) {
        int fo = 0;
        for (int m = 0; m < nm; ++m) {
            for (int i = threadIdx.x; i < T.dims[m]; i += NTH) T.w[m][i] = fac[fo + i];
            fo += T.dims[m];
        }
    }
    const int mk0 = p / d0;
    for (int i = threadIdx.x; i < T.pitch; i += NTH) {
        double pr = 0.0;
        if (i < p) {
            // kron(w_0, w_1, ...) built the way numpy.kron nests it: ((w0 * w1) * w2) ...
            const int a = i / mk0, j = i - a * mk0;
            pr = fac[a];
            if (nm == 2) {
                pr *= fac[d0 + j];
            } else {
                const unsigned short* dg = dig0 + (size_t)j * (4 * ((nm - 1 + 3) / 4));
                int fo = d0;
                for (int m = 1; m < nm; ++m) {
                    pr *= fac[fo + dg[m - 1]];
                    fo += T.dims[m];
                }
            }
        }
        if (publish) T.wkron[i] = pr;
        if (wkron_alt != nullptr) wkron_alt[i] = pr;
    }
    if (publish && threadIdx.x == 0 && T.sweeps) *T.sweeps = sweeps;
    TPLS_STAMP(5);
}

}  // namespace

}  // namespace tpls
