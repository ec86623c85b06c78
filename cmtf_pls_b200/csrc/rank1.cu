// Single-CTA rank-1 step with on-device convergence -- see rank1.cuh.
//
//   1 mode : w = Z / ||Z||
//   >=2    : HOSVD start (leading left singular vector of every unfolding, sign
//            fixed so the largest-|entry| is positive, mode 0 carrying sigma),
//            then rank-1 ALS sweeps with tensorly's stopping rule
//            |err_{s-1} - err_s| < tol from the second sweep on, <= 100 sweeps,
//            factors renormalised at the end of every sweep that did not stop.
//
// Leading eigenvector of each (small) Gram matrix: repeated squaring of the
// trace-normalised matrix, A <- A*A / tr(A*A).  tr(A*A) -> 1 exactly when A is
// rank one, so "1 - trace < 1e-7" means the iterate just formed has a
// second-to-first eigenvalue ratio below ~1e-14: logarithmic in the spectral
// gap, one tiny reduction per step, then a polish step against the original
// Gram matrix.  Everything is fp64.  Gram matrices and squarings run on the fp64
// tensor-core path (mma.sync.m8n8k4.f64, SASS DMMA): matrices are stored with
// their order rounded up to 8 (zero pads) and a leading dimension of that + 4, so
// that every fragment load of a half-warp is conflict-free.
//
// The same file holds the two kernels that keep a whole inner loop on the device:
// cov_loop_kernel (covariance mode, one CTA per coupled tensor in a cluster) and
// resident_loop_kernel (all trips of a component in one cooperative launch, one
// CTA per SM, rows cached in shared memory -- rank1.cuh, DESIGN.md section 3b).
#include "rank1.cuh"
#include "rank1_task.cuh"

#include <cooperative_groups.h>

#include <algorithm>
#include <cstdlib>

namespace tpls {

namespace {

// SMEM = true: the workspace is the dynamic shared memory of the CTA (the compiler then emits LDS/STS
// instead of generic loads); false: it is the task's global scratch buffer.
template <bool SMEM>
__global__ void __launch_bounds__(kRank1Threads, 1) rank1_kernel(const __grid_constant__ Rank1Args a) {
    pdl_prologue();
    if (trip_is_dead(a.ctrl, a.trip)) return;
    extern __shared__ __align__(16) double dyn[];
    const Rank1Task& T = a.t[blockIdx.x];
    if (SMEM)
        rank1_task(T, a.tol, a.normalize_on_break, dyn);
    else
        rank1_task(T, a.tol, a.normalize_on_break, T.scratch);
}

// One CTA per coupled tensor, the CTAs of a fit forming ONE thread-block cluster: every CTA runs the rank-1 step of
// its own tensor, the per-tensor contributions to q = Y't (m doubles) are stored into every CTA's shared memory
// through distributed shared memory, one cluster barrier per trip, and every CTA then forms the same q (fixed
// summation order) and takes the same stop decision.  Round 1 ran the tensors one after the other on a single CTA.
template <bool SMEM>
__global__ void __launch_bounds__(kRank1Threads, 1) cov_loop_kernel(const __grid_constant__ CovLoopArgs a) {
    pdl_prologue();
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(16) double dyn[];
    __shared__ double q_last[8], q_new[8], lred[4 * NWARP];
    __shared__ double rbuf[2][kMaxTensors][8];   // [trip parity][tensor][response]: filled by the tensors' CTAs
    __shared__ int lired[2 * NWARP];
    Grp blk{(int)threadIdx.x, NTH, 0, lred, lired, 0, nullptr};
    const int M = a.m, L = a.n_tasks;
    const int l = (int)cluster.block_rank();      // this CTA's tensor
    const Rank1Task& T = a.t[l];
    const double* Cl = a.C[l];
    if (threadIdx.x < 8) q_last[threadIdx.x] = threadIdx.x == 0 ? 1.0 : 0.0;  // u_0 = Y[:, 0] = Y e_0 (tpls.py:78)
    __syncthreads();
    int trips = 0;
    bool converged = false;
    for (int trip = 0; trip < a.max_iter; ++trip) {
        trips = trip + 1;
        // Z = X x_1 u with u = Y q_last  ==  sum_m q_last[m] * C[m][:]
        double* z = const_cast<double*>(T.z);
        for (int i = threadIdx.x; i < T.p; i += NTH) {
            double v = 0.0;
            for (int m = 0; m < M; ++m) v = fma(q_last[m], Cl[(size_t)m * T.pitch + i], v);
            z[i] = v;
        }
        __syncthreads();
        if (SMEM)
            rank1_task(T, a.tol, a.normalize_on_break, dyn);
        else
            rank1_task(T, a.tol, a.normalize_on_break, T.scratch);
        __syncthreads();
        // Y't of this tensor = C'^T kron(w): the row-rescaled block when masked (missingvals.py:23-38);
        // thread 0 publishes the m values in every CTA of the cluster
        const double* Cq = Cl + (size_t)a.masked[l] * T.pitch;
        for (int m = 0; m < M; ++m) {
            double s = 0.0;
            for (int i = threadIdx.x; i < T.p; i += NTH) s = fma(Cq[(size_t)m * T.pitch + i], T.wkron[i], s);
            s = bsum(s, blk);
            if (threadIdx.x == 0)
                for (int r = 0; r < L; ++r) cluster.map_shared_rank(&rbuf[trip & 1][l][m], r)[0] = s;
        }
        cluster.sync();
        // q = Y't / ||Y't||, t = average of the tensors' projections (cmtf.py:120-122)
        if (threadIdx.x == 0) {
            double r_acc[8];
            double nrm = 0.0;
            for (int m = 0; m < M; ++m) {
                double t = 0.0;
                for (int r = 0; r < L; ++r) t += rbuf[trip & 1][r][m];
                r_acc[m] = t / (double)L;
                nrm = fma(r_acc[m], r_acc[m], nrm);
            }
            nrm = sqrt(nrm);
            for (int m = 0; m < M; ++m) q_new[m] = r_acc[m] / nrm;
        }
        __syncthreads();
        bool stop = false;
        if (trip >= 1) {
            double d2 = 0.0;
            for (int i = 0; i < M; ++i) {
                const double di = q_last[i] - q_new[i];
                for (int j = 0; j < M; ++j) d2 = fma(di * a.gram_y[i * M + j], q_last[j] - q_new[j], d2);
            }
            stop = sqrt(fabs(d2)) < a.tol;
        }
        __syncthreads();
        if (threadIdx.x < 8) q_last[threadIdx.x] = threadIdx.x < M ? q_new[threadIdx.x] : 0.0;
        __syncthreads();
        if (stop) {
            converged = true;
            break;
        }
    }
    if (l == 0) {
        for (int i = threadIdx.x; i < a.pitch_y; i += NTH) {
            const double v = i < M ? q_last[i] : 0.0;
            a.qvec[i] = v;
            if (i < M) a.q_out[i] = v;
        }
        if (threadIdx.x == 0) {
            *a.trips_out = trips;
            if (a.conv_out != nullptr) *a.conv_out = converged ? 1 : 0;
        }
    }
    cluster.sync();  // no CTA may exit while a peer can still store into its shared memory
}


// ---------------------------------------------------------------------------------------------------------------
// Resident trip loop (rank1.cuh)
// ---------------------------------------------------------------------------------------------------------------
constexpr size_t kResidentScratch = 20 * 1024;  // bytes of dynamic shared memory the non-rank-1 phases use

// Grid-wide barrier of co-resident CTAs (one per SM).  Every CTA owns a flag word on its own 128-byte line
// (bar[32 * (c + 1)]); bar[0] holds the generation the previous launch ended on.  Arriving = one release store of the
// next generation into the own flag; waiting = thread c polls the flag of CTA c (relaxed loads, one fence after the
// loop), then the CTA barrier joins them.  No atomic round trip and no counter to reset: an arrival is visible to a
// poller one store and one load after the CTA's own writes have drained.
__device__ __forceinline__ void grid_sync(unsigned int* bar, unsigned int n_ctas, unsigned int& gen) {
    __syncthreads();
    ++gen;
    if (threadIdx.x == 0)
        asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(bar + 32 * (blockIdx.x + 1)), "r"(gen) : "memory");
    if (threadIdx.x < n_ctas) {
        const unsigned int* f = bar + 32 * (threadIdx.x + 1);
        unsigned int v;
        do {
            asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(f) : "memory");
        } while ((int)(v - gen) < 0);
        __threadfence();
    }
    __syncthreads();
}

template <typename XT>
struct RVec;
template <>
struct RVec<float> {
    using type = float4;
    static constexpr int N = 4;
};
template <>
struct RVec<double> {
    using type = double2;
    static constexpr int N = 2;
};
template <typename XT>
union RPack {
    typename RVec<XT>::type v;
    XT e[RVec<XT>::N];
};

// NR rows of X times kron(w) at once: the lanes of a warp stride over the 16-byte column groups and keep H * NR
// loads in flight (a load costs its latency, not its bytes); out[i] = this LANE's share of row i's dot product (the
// caller folds the lanes once per row, after all coupled tensors).  xr[i] points at a row in the shared-memory cache
// or in global memory (generic loads).  kron(w) was written by another CTA earlier in this launch: plain loads
// (ordered by the grid barrier), never the non-coherent path.
template <typename XT, bool MASKED, int NR, int H>
__device__ __forceinline__ void resident_row_dots(const XT* const (&xr)[NR], int pitch, const double* wk, int lane, double (&out)[NR]) {
    constexpr int VEC = RVec<XT>::N;
    using V = typename RVec<XT>::type;
    double acc[NR][2];
    const XT* px[NR];  // this lane's position in every row: the pointers advance, the loads of a step use constant offsets
#pragma unroll
    for (int i = 0; i < NR; ++i) {
        acc[i][0] = acc[i][1] = 0.0;
        px[i] = xr[i] + lane * VEC;
    }
    const double* pw = wk + lane * VEC;
    int left = pitch / VEC - lane;  // column groups from this lane's first one to the end of the row
    for (; left > (H - 1) * 32; left -= H * 32) {
        RPack<XT> in[NR][H];
#pragma unroll
        for (int h = 0; h < H; ++h)
#pragma unroll
            for (int i = 0; i < NR; ++i) in[i][h].v = *reinterpret_cast<const V*>(px[i] + h * 32 * VEC);
#pragma unroll
        for (int h = 0; h < H; ++h)
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                const double w = pw[h * 32 * VEC + j];
#pragma unroll
                for (int i = 0; i < NR; ++i) {
                    XT xs = in[i][h].e[j];
                    if (MASKED && !(xs == xs)) xs = (XT)0;
                    acc[i][j & 1] = fma((double)xs, w, acc[i][j & 1]);
                }
            }
#pragma unroll
        for (int i = 0; i < NR; ++i) px[i] += H * 32 * VEC;
        pw += H * 32 * VEC;
    }
    for (; left > 0; left -= 32) {
        RPack<XT> in[NR];
#pragma unroll
        for (int i = 0; i < NR; ++i) in[i].v = *reinterpret_cast<const V*>(px[i]);
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            const double w = pw[j];
#pragma unroll
            for (int i = 0; i < NR; ++i) {
                XT xs = in[i].e[j];
                if (MASKED && !(xs == xs)) xs = (XT)0;
                acc[i][j & 1] = fma((double)xs, w, acc[i][j & 1]);
            }
        }
#pragma unroll
        for (int i = 0; i < NR; ++i) px[i] += 32 * VEC;
        pw += 32 * VEC;
    }
#pragma unroll
    for (int i = 0; i < NR; ++i) out[i] = acc[i][0] + acc[i][1];
}

// Probe builds (-DTPLS_PROBE): clock64 deltas of thread 0 of CTA 0 inside the phases of the resident loop
#ifdef TPLS_PROBE
__device__ long long g_fine[32];
#define FINE_DECL long long fine_t = clock64()
#define FINE(i)                                                         \
    do {                                                                \
        if (blockIdx.x == 0 && threadIdx.x == 0) {                      \
            const long long fine_now = clock64();                       \
            g_fine[i] += fine_now - fine_t;                             \
            fine_t = fine_now;                                          \
        }                                                               \
    } while (0)
#else
#define FINE_DECL
#define FINE(i)
#endif

// Where the rows of a CTA's block live: the first n_cached of them in shared memory, the rest in global memory.
// Rows are addressed by their index inside the block (32-bit arithmetic).
template <typename XT>
struct RowSrc {
    const XT* gbase;   // row 0 of the block in global memory
    const XT* cbase;   // row 0 of the block in the shared-memory cache
    int n_cached, pitch;
    __device__ __forceinline__ const XT* row(int k) const {
        return (k < n_cached ? cbase : gbase) + (size_t)((unsigned)k * (unsigned)pitch);
    }
};

constexpr int kResidentUChunk = 1024;  // rows of u = Y q kept in shared memory at a time

// u[k] = Y[k,:] . q for the rows [c_lo, c_hi) of the block, once per CTA (every thread of the contraction would
// otherwise form the u of each of its rows itself: m loads per row against one 16-byte load of X)
__device__ __forceinline__ void resident_u_chunk(double* u_s, const RowSrc<double>& ysrc, int m, const double* q_s, int c_lo, int c_hi) {
    __syncthreads();
    for (int k = c_lo + (int)threadIdx.x; k < c_hi; k += NTH) {
        const double* yr = ysrc.row(k);
        double ui = 0.0;
#pragma unroll
        for (int q = 0; q < 8; ++q)
            if (q < m) ui = fma(yr[q], q_s[q], ui);
        u_s[k - c_lo] = ui;
    }
    __syncthreads();
}

// n rows starting at `base` (all in shared memory or all in global memory), their u in `u`, into a thread's
// accumulators.  Every row lane takes a CONTIGUOUS run of the rows: one pointer that advances, constant offsets for the
// RU rows of a step (their loads are issued before any of them is used), u in consecutive shared-memory words.
template <typename XT, bool MASKED, int KC, int RU>
__device__ __forceinline__ void resident_contract_rows(const XT* base, const double* u, int n, int pitch, int n_cg, int lpr, int rpt,
                                                       int cl, int rl, double (&zacc)[KC][RVec<XT>::N]) {
    constexpr int VEC = RVec<XT>::N;
    using V = typename RVec<XT>::type;
    const int per = (n + rpt - 1) / rpt;
    int r = rl * per;
    const int r_end = min(n, r + per);
    if (r >= r_end) return;
    const XT* p = base + (size_t)((unsigned)r * (unsigned)pitch) + cl * VEC;
    const double* up = u + r;
    for (; r + RU <= r_end; r += RU) {
        double uu[RU];
#pragma unroll
        for (int i = 0; i < RU; ++i) uu[i] = up[i];
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            if (cl + k * lpr < n_cg) {
                RPack<XT> in[RU];
#pragma unroll
                for (int i = 0; i < RU; ++i) in[i].v = *reinterpret_cast<const V*>(p + (size_t)i * pitch + k * lpr * VEC);
#pragma unroll
                for (int i = 0; i < RU; ++i)
#pragma unroll
                    for (int j = 0; j < VEC; ++j) {
                        XT xs = in[i].e[j];
                        if (MASKED && !(xs == xs)) xs = (XT)0;
                        zacc[k][j] = fma((double)xs, uu[i], zacc[k][j]);
                    }
            }
        }
        p += (size_t)RU * pitch;
        up += RU;
    }
    if (r < r_end) {  // the last, partial step of the run: rows past its end repeat its first row with u = 0
        const int nv = r_end - r;
        double uu[RU];
#pragma unroll
        for (int i = 0; i < RU; ++i) uu[i] = i < nv ? up[i] : 0.0;
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            if (cl + k * lpr < n_cg) {
                RPack<XT> in[RU];
#pragma unroll
                for (int i = 0; i < RU; ++i)
                    in[i].v = *reinterpret_cast<const V*>(p + (i < nv ? (size_t)i * pitch : (size_t)0) + k * lpr * VEC);
#pragma unroll
                for (int i = 0; i < RU; ++i)
#pragma unroll
                    for (int j = 0; j < VEC; ++j) {
                        XT xs = in[i].e[j];
                        if (MASKED && !(xs == xs)) xs = (XT)0;
                        zacc[k][j] = fma((double)xs, uu[i], zacc[k][j]);
                    }
            }
        }
    }
}

// Z partials of this CTA's rows for one tensor: zpart_row[c] = sum_r x[r, c] * u[r], u[r] = Y[r,:] . q
// Per chunk of u: the rows still in L2 first, with twice the rows of a thread in flight (their loads are the long
// ones), then the rows in the shared-memory cache.
template <typename XT, bool MASKED, int KC>
__device__ __forceinline__ void resident_contract_kc(const ResidentTensor& X, const RowSrc<XT>& src, const RowSrc<double>& ysrc, int m,
                                                     const double* q_s, int nblk, double* u_s, int& u_lo, double* zrow, double* scr) {
    constexpr int VEC = RVec<XT>::N;
    const int n_cg = X.pitch / VEC;
    int lpr = 1;
    while (lpr < n_cg && lpr < NTH) lpr <<= 1;
    const int rpt = NTH / lpr;
    const int cl = threadIdx.x & (lpr - 1), rl = threadIdx.x / lpr;
    double zacc[KC][VEC];
#pragma unroll
    for (int k = 0; k < KC; ++k)
#pragma unroll
        for (int j = 0; j < VEC; ++j) zacc[k][j] = 0.0;
    constexpr int RU = KC <= 2 ? 8 : 4;  // rows in flight per thread: the loads of a group are issued before any of them is used
    FINE_DECL;
    for (int c_lo = 0; c_lo < nblk; c_lo += kResidentUChunk) {
        const int c_hi = min(nblk, c_lo + kResidentUChunk);
        if (u_lo != c_lo) {
            resident_u_chunk(u_s, ysrc, m, q_s, c_lo, c_hi);
            u_lo = c_lo;
        }
        FINE(8);
        const int split = min(c_hi, max(c_lo, src.n_cached));  // [c_lo, split) cached, [split, c_hi) in L2
        resident_contract_rows<XT, MASKED, KC, (KC == 1 ? 2 * RU : RU)>(src.gbase + (size_t)((unsigned)split * (unsigned)src.pitch),
                                                                        u_s + (split - c_lo), c_hi - split, src.pitch, n_cg, lpr, rpt,
                                                                        cl, rl, zacc);
        resident_contract_rows<XT, MASKED, KC, RU>(src.cbase + (size_t)((unsigned)c_lo * (unsigned)src.pitch), u_s, split - c_lo, src.pitch,
                                                   n_cg, lpr, rpt, cl, rl, zacc);
    }
    FINE(9);
    if (rpt == 1) {
#pragma unroll
        for (int k = 0; k < KC; ++k) {
            const int cg = cl + k * lpr;
            if (cg < n_cg) {
#pragma unroll
                for (int j = 0; j < VEC; ++j) zrow[cg * VEC + j] = zacc[k][j];
            }
        }
    } else {
        // fewer than NTH column groups: several row lanes per column group (then one group per thread), folded in order
        __syncthreads();
#pragma unroll
        for (int j = 0; j < VEC; ++j) scr[(size_t)threadIdx.x * VEC + j] = zacc[0][j];
        __syncthreads();
        if (rl == 0 && cl < n_cg) {
#pragma unroll
            for (int j = 0; j < VEC; ++j) {
                double t = 0.0;
                for (int q = 0; q < rpt; ++q) t += scr[((size_t)q * lpr + cl) * VEC + j];
                zrow[cl * VEC + j] = t;
            }
        }
        __syncthreads();
    }
    FINE(10);
}

template <typename XT, bool MASKED>
__device__ __forceinline__ void resident_contract_m(const ResidentTensor& X, const RowSrc<XT>& src, const RowSrc<double>& ysrc, int m,
                                                    const double* q_s, int nblk, double* u_s, int& u_lo, double* zrow, double* scr) {
    const int n_cg = X.pitch / RVec<XT>::N;
    if (n_cg <= NTH)
        resident_contract_kc<XT, MASKED, 1>(X, src, ysrc, m, q_s, nblk, u_s, u_lo, zrow, scr);
    else if (n_cg <= 2 * NTH)
        resident_contract_kc<XT, MASKED, 2>(X, src, ysrc, m, q_s, nblk, u_s, u_lo, zrow, scr);
    else
        resident_contract_kc<XT, MASKED, kResidentKc>(X, src, ysrc, m, q_s, nblk, u_s, u_lo, zrow, scr);
}

template <typename XT>
__device__ __forceinline__ void resident_contract(const ResidentTensor& X, const RowSrc<XT>& src, const RowSrc<double>& ysrc, int m,
                                                  const double* q_s, int nblk, double* u_s, int& u_lo, double* zrow, double* scr) {
    if (X.masked)
        resident_contract_m<XT, true>(X, src, ysrc, m, q_s, nblk, u_s, u_lo, zrow, scr);
    else
        resident_contract_m<XT, false>(X, src, ysrc, m, q_s, nblk, u_s, u_lo, zrow, scr);
}

// Projection of the rows [lo, hi) of a CTA's block: the rows are dealt to the warps round-robin, NR rows of a warp at
// a time with H column groups per row in flight.  Complete tensors add up per lane and are folded over the lanes once
// per row; a masked tensor is folded on its own (its rescale p / observed is per row and tensor, missingvals.py:37).
// Writes the scores, adds the rows' share of q = Y't to qacc (lane i < pitch_y: response i).
template <int NR, int H>
__device__ __forceinline__ void resident_project_rows(const ResidentArgs& a, int lo, int hi, long long r_lo, const unsigned char* cache,
                                                      int nblk, const double* w_s, const RowSrc<double>& ysrc, int warp, int lane,
                                                      double& qacc) {
    const int L = a.n_tensors;
    const double inv_l = 1.0 / (double)L;
    const bool pow2 = (L & (L - 1)) == 0;
    for (int k0 = lo + warp; k0 < hi; k0 += NR * NWARP) {
        int ks[NR];
        double tl[NR], td[NR];
#pragma unroll
        for (int i = 0; i < NR; ++i) {
            const int k = k0 + i * NWARP;
            ks[i] = k < hi ? k : k0;  // rows past the end repeat the warp's first row (results dropped)
            tl[i] = td[i] = 0.0;
        }
        size_t coff = 0;
        int woff = 0;
        for (int l = 0; l < L; ++l) {
            const ResidentTensor& X = a.x[l];
            const double* wk = w_s != nullptr ? w_s + woff : X.wkron;
            double v[NR];
            if (X.dtype == 0) {
                const RowSrc<float> src{reinterpret_cast<const float*>(X.x) + (size_t)r_lo * X.pitch,
                                        reinterpret_cast<const float*>(cache + coff), min(X.cache_rows, nblk), X.pitch};
                const float* xr[NR];
#pragma unroll
                for (int i = 0; i < NR; ++i) xr[i] = src.row(ks[i]);
                if (X.masked)
                    resident_row_dots<float, true, NR, H>(xr, X.pitch, wk, lane, v);
                else
                    resident_row_dots<float, false, NR, H>(xr, X.pitch, wk, lane, v);
                coff += (size_t)X.cache_rows * X.pitch * 4;
            } else {
                const RowSrc<double> src{reinterpret_cast<const double*>(X.x) + (size_t)r_lo * X.pitch,
                                         reinterpret_cast<const double*>(cache + coff), min(X.cache_rows, nblk), X.pitch};
                const double* xr[NR];
#pragma unroll
                for (int i = 0; i < NR; ++i) xr[i] = src.row(ks[i]);
                if (X.masked)
                    resident_row_dots<double, true, NR, H>(xr, X.pitch, wk, lane, v);
                else
                    resident_row_dots<double, false, NR, H>(xr, X.pitch, wk, lane, v);
                coff += (size_t)X.cache_rows * X.pitch * 8;
            }
            woff += X.pitch;
            if (X.masked) {
#pragma unroll
                for (int m = 16; m >= 1; m >>= 1)
#pragma unroll
                    for (int i = 0; i < NR; ++i) v[i] += __shfl_xor_sync(0xffffffffu, v[i], m);
#pragma unroll
                for (int i = 0; i < NR; ++i) td[i] += v[i] / __ldg(X.rowcnt + r_lo + ks[i]) * (double)X.p;
            } else {
#pragma unroll
                for (int i = 0; i < NR; ++i) tl[i] += v[i];
            }
        }
#pragma unroll
        for (int m = 16; m >= 1; m >>= 1)
#pragma unroll
            for (int i = 0; i < NR; ++i) tl[i] += __shfl_xor_sync(0xffffffffu, tl[i], m);
#pragma unroll
        for (int i = 0; i < NR; ++i) {
            const int k = k0 + i * NWARP;
            if (k >= hi) break;
            double ti = tl[i] + td[i];
            if (L > 1) ti = pow2 ? ti * inv_l : ti / (double)L;
            if (lane == 0) a.t_out[r_lo + k] = ti;
            if (lane < a.pitch_y) {
                const double y = ysrc.row(k)[lane];
                if (y != 0.0) qacc = fma(y, ti, qacc);  // a held-out row (Y row 0) adds nothing, even a NaN t
            }
        }
    }
}

__device__ __forceinline__ long long global_ns() {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

template <bool SMEM>
__global__ void __launch_bounds__(kRank1Threads, 1) resident_loop_kernel(const __grid_constant__ ResidentArgs a) {
    pdl_prologue();
    // diagnostics: thread 0 of CTA 0 adds the time since the previous mark to slot i
    long long t_mark = 0;
    const bool stamping = a.stamps != nullptr && blockIdx.x == 0 && threadIdx.x == 0;
    if (stamping) t_mark = global_ns();
#define RES_MARK(i)                              \
    if (stamping) {                              \
        const long long t_now = global_ns();     \
        a.stamps[i] += t_now - t_mark;           \
        t_mark = t_now;                          \
    }
    extern __shared__ __align__(16) double dyn[];
    __shared__ double q_s[8], qp_s[8], qw_s[NWARP][8];
    __shared__ int stop_s;
    __shared__ __align__(8) uint64_t cache_bar;
    __shared__ double u_s[kResidentUChunk];
    __shared__ double dq_s[8], gram_s[64];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = (int)gridDim.x, b = (int)blockIdx.x;
    const int L = a.n_tensors, M = a.m;
    const long long per = (a.n_rows + G - 1) / G;
    const long long r_lo = min(a.n_rows, (long long)b * per), r_hi = min(a.n_rows, r_lo + per);
    double* scr = dyn;  // phases other than the rank-1 step: <= kResidentScratch bytes
    // The first rows of the block live in shared memory from the first projection on: x[l].cache_rows of tensor l,
    // y_cache_rows of Y (the launcher gives narrow tensors and Y all their rows first; the widest tensor gets what is
    // left), tensor after tensor, Y last.  n_cached = the rows that EVERY tensor has in shared memory.
    unsigned char* const cache = reinterpret_cast<unsigned char*>(dyn) + a.cache_off;
    const int nblk = (int)(r_hi - r_lo);  // rows of this CTA's block
    const int n_cached = max(0, min(a.cache_rows, nblk));
    size_t y_cache_off = 0;
    bool any_cached = nblk > 0 && a.y_cache_rows > 0;
    for (int l = 0; l < L; ++l) {
        y_cache_off += (size_t)a.x[l].cache_rows * a.x[l].pitch * (a.x[l].dtype == 0 ? 4 : 8);
        any_cached = any_cached || (nblk > 0 && a.x[l].cache_rows > 0);
    }
    double* const w_reg = a.w_off != 0 ? reinterpret_cast<double*>(reinterpret_cast<unsigned char*>(dyn) + a.w_off) : nullptr;
    unsigned int bar_gen = 0;
    if (tid < 8) qp_s[tid] = tid < M ? a.q_prev[tid] : 0.0;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(bar_gen) : "l"(a.bar) : "memory");  // every thread tracks it
    if (tid == 0) {
        stop_s = 0;
        mbar_init(&cache_bar, 1);
        fence_mbar_init();
    }
    __syncthreads();
    if (tid == 0 && any_cached) {
        // one thread hands the copies to the bulk-copy engine; they land while the first fold and rank-1 step run
        unsigned int total = (unsigned int)min(a.y_cache_rows, nblk) * (unsigned int)(a.pitch_y * 8);
        for (int l = 0; l < L; ++l)
            total += (unsigned int)min(a.x[l].cache_rows, nblk) * (unsigned int)(a.x[l].pitch * (a.x[l].dtype == 0 ? 4 : 8));
        mbar_arrive_expect_tx(&cache_bar, total);
        size_t off = 0;
        for (int l = 0; l <= L; ++l) {
            const size_t row_b = l < L ? (size_t)a.x[l].pitch * (a.x[l].dtype == 0 ? 4 : 8) : (size_t)a.pitch_y * 8;
            const int rows_l = l < L ? a.x[l].cache_rows : a.y_cache_rows;
            const unsigned char* g = reinterpret_cast<const unsigned char*>(l < L ? a.x[l].x : (const void*)a.y) + (size_t)r_lo * row_b;
            const size_t bytes = (size_t)min(rows_l, nblk) * row_b;
            for (size_t o = 0; o < bytes; o += 32768)
                bulk_g2s(cache + off + o, g + o, (uint32_t)min((size_t)32768, bytes - o), &cache_bar);
            off += (size_t)rows_l * row_b;
        }
    }
    {
        // this CTA's share of Y'Y (the stop test needs dq^T Y'Y dq): entry e = (i, j) on NTH / m^2 row lanes, the lanes
        // folded in order; every CTA folds the partials of all CTAs before the first stop test
        const int MM = M * M, nl = NTH / MM;
        const int e = tid % MM, ln = tid / MM;
        double acc = 0.0;
        if (ln < nl) {
            const double* yb = a.y + (size_t)r_lo * a.pitch_y;
            const int i = e / M, j = e - i * M;
            for (int k = ln; k < nblk; k += nl) acc = fma(yb[(size_t)k * a.pitch_y + i], yb[(size_t)k * a.pitch_y + j], acc);
            scr[ln * MM + e] = acc;
        }
        __syncthreads();
        if (tid < MM) {
            double t = 0.0;
            for (int q = 0; q < nl; ++q) t += scr[q * MM + tid];
            a.grampart[(size_t)b * 64 + tid] = t;
        }
        __syncthreads();
    }
    const RowSrc<double> ysrc{a.y + (size_t)r_lo * a.pitch_y, reinterpret_cast<const double*>(cache + y_cache_off), min(a.y_cache_rows, nblk),
                              a.pitch_y};
    int trip = 0;
    double d2_last = 0.0;
    int done_trip = -1;
    for (;;) {
        // ---- Z = fold of the per-CTA partials (trip 0: the fused centring / deflation pass wrote them) ----
        {
            int chunk = b;
            for (int l = 0; l < L; ++l) {
                const ResidentTensor& X = a.x[l];
                const int nch = (X.pitch + 31) >> 5;
                const int n_parts = trip == 0 ? X.parts0 : G;
                for (; chunk < nch; chunk += G) {
                    const int c = chunk * 32 + lane;   // 32 columns x 16 part-groups
                    double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;
                    if (c < X.pitch) {
                        // a warp's share of the partials (one per CTA: ~10 rows) in ONE round of loads: rows past the end
                        // are not read and add 0 (three dependent L2 round trips with four loads at a time)
                        for (int pb = warp; pb < n_parts; pb += 12 * NWARP) {
                            double v[12];
#pragma unroll
                            for (int k = 0; k < 12; ++k) {
                                const int pk = pb + k * NWARP;
                                v[k] = pk < n_parts ? __ldcg(X.zpart + (size_t)pk * X.pitch + c) : 0.0;
                            }
#pragma unroll
                            for (int k = 0; k < 12; k += 4) {
                                t0 += v[k];
                                t1 += v[k + 1];
                                t2 += v[k + 2];
                                t3 += v[k + 3];
                            }
                        }
                    }
                    __syncthreads();
                    scr[warp * 33 + lane] = (t0 + t1) + (t2 + t3);
                    __syncthreads();
                    if (warp == 0 && c < X.pitch) {
                        double t = 0.0;
#pragma unroll
                        for (int k = 0; k < NWARP; ++k) t += scr[k * 33 + lane];
                        X.z[c] = t;
                    }
                }
                chunk -= nch;
            }
        }
        RES_MARK(0);
        grid_sync(a.bar, G, bar_gen);
        RES_MARK(5);
        // ---- rank-1 step (tpls.py:84-90, cmtf.py:98-104): on the first L CTAs, one tensor each, followed by a grid
        //      barrier -- or, when the launcher found it cheap enough (at most one coupled tensor with a Z of two or
        //      more modes), on EVERY CTA: each forms the same weights from the same Z, kron(w) lands in its own shared
        //      memory, and there is no barrier to wait at and no staging round trip (CTA 0 publishes) ----
        {
            const bool everywhere = SMEM && a.r1_everywhere != 0;
            const int l_lo = everywhere ? 0 : min(b, L), l_hi = everywhere ? L : min(b + 1, L);
            int woff = 0;
            for (int l = 0; l < l_lo; ++l) woff += a.x[l].pitch;
            for (int l = l_lo; l < l_hi; ++l) {
                rank1_task(a.r1[l], a.tol, a.normalize_on_break, SMEM ? dyn : a.r1[l].scratch, everywhere ? w_reg + woff : nullptr,
                           !everywhere || b == 0);
                woff += a.x[l].pitch;
                if (everywhere) __syncthreads();  // the next task reuses the workspace
            }
            RES_MARK(1);
            if (!everywhere) grid_sync(a.bar, G, bar_gen);
            RES_MARK(6);
        }
        // ---- projection of this CTA's rows (a warp per row), coupled average, partials of q = Y't ----
        if (trip == 0 && any_cached) mbar_wait(&cache_bar, 0);  // the cached rows have landed
        {
            double qacc = 0.0;  // lane i < pitch_y: response i
            const double* w_s = nullptr;
            if (w_reg != nullptr) {
                if (!(SMEM && a.r1_everywhere != 0)) {
                    // kron(w) of all tensors into shared memory: one L2 round trip for the CTA instead of one per warp and slice
                    int woff = 0;
                    for (int l = 0; l < L; ++l) {
                        const double* wk = a.x[l].wkron;
                        for (int i = tid; i < a.x[l].pitch; i += NTH) w_reg[woff + i] = wk[i];
                        woff += a.x[l].pitch;
                    }
                    __syncthreads();
                }
                w_s = w_reg;
            }
            FINE_DECL;
            // rows still in L2 first and with whole rows in flight (their loads are the long ones), then the cached rows
            resident_project_rows<2, 8>(a, n_cached, nblk, r_lo, cache, nblk, w_s, ysrc, warp, lane, qacc);
            FINE(0);
            resident_project_rows<4, 2>(a, 0, n_cached, r_lo, cache, nblk, w_s, ysrc, warp, lane, qacc);
            FINE(1);
            if (lane < 8) qw_s[warp][lane] = lane < a.pitch_y ? qacc : 0.0;
            __syncthreads();
            if (tid < 8) {
                double t = 0.0;
#pragma unroll
                for (int w = 0; w < NWARP; ++w) t += qw_s[w][tid];
                a.qpart[(size_t)b * 8 + tid] = t;
            }
            FINE(5);
        }
        RES_MARK(2);
        grid_sync(a.bar, G, bar_gen);
        RES_MARK(7);
        // ---- q = Y't / ||.||, stop test dq^T (Y'Y) dq (tpls.py:100-107): every CTA folds the same partials in the
        //      same order and takes the same decision; CTA 0 publishes it ----
        {
            if (trip == 0) {
                // Y'Y = sum of the CTAs' partials (written before the first grid barrier), 64 entries x 8 part-groups
                const int e = tid & 63, grp8 = tid >> 6;
                double g0 = 0.0, g1 = 0.0;
                if (e < M * M) {
                    int pb = grp8;
                    for (; pb + 8 < G; pb += 16) {
                        const double v0 = __ldcg(a.grampart + (size_t)pb * 64 + e);
                        const double v1 = __ldcg(a.grampart + (size_t)(pb + 8) * 64 + e);
                        g0 += v0;
                        g1 += v1;
                    }
                    if (pb < G) g0 += __ldcg(a.grampart + (size_t)pb * 64 + e);
                }
                u_s[grp8 * 64 + e] = g0 + g1;
                __syncthreads();
                if (tid < M * M) {
                    double t = 0.0;
#pragma unroll
                    for (int k = 0; k < 8; ++k) t += u_s[k * 64 + tid];
                    gram_s[tid] = t;
                    if (b == 0) a.gram[tid] = t;
                }
                __syncthreads();
            }
            const int col = tid & 7, grp = tid >> 3;  // 8 responses x 64 part-groups (4 per warp)
            double t0 = 0.0, t1 = 0.0;
            for (int pb = grp; pb < G; pb += 4 * (NTH / 8)) {  // (one round of loads for up to 256 CTAs)
                double v[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int pk = pb + k * (NTH / 8);
                    v[k] = pk < G ? __ldcg(a.qpart + (size_t)pk * 8 + col) : 0.0;
                }
                t0 += v[0] + v[2];
                t1 += v[1] + v[3];
            }
            double t = t0 + t1;
            t += shfl_xor_d(t, 8);
            t += shfl_xor_d(t, 16);
            if (lane < 8) qw_s[warp][lane] = t;
            __syncthreads();
            if (tid < 8) {
                // eight lanes in step: every lane folds its response, forms the same norm, divides its own entry
                double s = 0.0;
#pragma unroll
                for (int k = 0; k < NWARP; ++k) s += qw_s[k][tid];
                if (tid >= M) s = 0.0;
                double nrm = 0.0;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const double si = __shfl_sync(0xffu, s, i);
                    nrm = fma(si, si, nrm);
                }
                nrm = sqrt(nrm);
                const double qi = tid < M ? s / nrm : 0.0;
                dq_s[tid] = qp_s[tid] - qi;
                q_s[tid] = qi;
                qp_s[tid] = qi;
                __syncwarp(0xffu);
                if (tid == 0) {
                    double d2 = 0.0;
                    for (int i = 0; i < M; ++i)
                        for (int j = 0; j < M; ++j) d2 = fma(dq_s[i] * gram_s[i * M + j], dq_s[j], d2);
                    d2_last = d2;
                    bool stop = false;
                    if (trip >= 1 && sqrt(fabs(d2)) < a.tol) {
                        done_trip = trip;
                        stop = true;
                    }
                    if (trip + 1 >= a.max_iter) stop = true;
                    stop_s = stop ? 1 : 0;
                }
            }
            __syncthreads();
        }
        ++trip;
        RES_MARK(3);
        if (stop_s) break;
        // ---- contraction for the next trip: u = Y q row by row (tpls.py:102 fused into :83) ----
        {
            size_t coff = 0;
            int u_lo = -1;  // first row of the block whose u sits in u_s
            for (int l = 0; l < L; ++l) {
                const ResidentTensor& X = a.x[l];
                double* zrow = X.zpart + (size_t)b * X.pitch;
                if (X.dtype == 0) {
                    const RowSrc<float> src{reinterpret_cast<const float*>(X.x) + (size_t)r_lo * X.pitch,
                                            reinterpret_cast<const float*>(cache + coff), min(X.cache_rows, nblk), X.pitch};
                    resident_contract<float>(X, src, ysrc, M, q_s, nblk, u_s, u_lo, zrow, scr);
                    coff += (size_t)X.cache_rows * X.pitch * 4;
                } else {
                    const RowSrc<double> src{reinterpret_cast<const double*>(X.x) + (size_t)r_lo * X.pitch,
                                             reinterpret_cast<const double*>(cache + coff), min(X.cache_rows, nblk), X.pitch};
                    resident_contract<double>(X, src, ysrc, M, q_s, nblk, u_s, u_lo, zrow, scr);
                    coff += (size_t)X.cache_rows * X.pitch * 8;
                }
            }
        }
        RES_MARK(4);
        grid_sync(a.bar, G, bar_gen);
        RES_MARK(8);
    }
    if (stamping) a.stamps[9] += trip;
#undef RES_MARK
    // u = Y q of the last trip for this CTA's rows (tpls.py:102)
    for (int k = tid; k < nblk; k += NTH) {
        const double* yr = ysrc.row(k);
        double ui = 0.0;
#pragma unroll
        for (int q = 0; q < 8; ++q)
            if (q < M) ui = fma(yr[q], q_s[q], ui);
        a.u_out[r_lo + k] = ui;
    }
    // ---- the tail of the component (tpls.py:110-113), as solve_coef / lincomb / the Y deflation pass do it ----
    if (a.tail) {
        const int ka = a.comp + 1, npairs = 2 * ka, R = a.n_comp;
        __syncthreads();  // u of this CTA's rows is in global memory
        // partial dot products over the block: pair j < ka is T_j . T_a, pair ka + j is T_j . u (weighted rows)
        for (int j = warp; j < npairs; j += NWARP) {
            const double* pa = a.T + (size_t)(j < ka ? j : j - ka) * a.n_rows + r_lo;
            const double* pb = (j < ka ? a.t_out : a.u_out) + r_lo;
            double sacc = 0.0;
            for (int k = lane; k < nblk; k += 32) {
                double av = pa[k];
                if (a.row_w != nullptr) {
                    if (a.row_w[r_lo + k] == 0.0) continue;  // a held-out score can be NaN: skip, not * 0
                    av *= a.row_w[r_lo + k];
                }
                sacc = fma(av, pb[k], sacc);
            }
            sacc = warp_sum(sacc);
            if (lane == 0) a.dotpart[(size_t)b * 64 + j] = sacc;
        }
        grid_sync(a.bar, G, bar_gen);
        // every CTA: fold the partials (64 pairs x 8 part-groups), the Gram block of the scores so far into shared memory
        double* Gs = scr;            // [ka][ka]
        double* Lm = scr + 1024;     // [ka][ka] Cholesky factor
        double* dots_s = u_s + 512;  // [npairs]; then y, x, 1/||t||, dropped flags
        double* ys = u_s + 576;
        double* xs = u_s + 640;
        double* dinv = u_s + 704;
        double* drop = u_s + 768;
        {
            const int e = tid & 63, grp8 = tid >> 6;
            double g0 = 0.0, g1 = 0.0;
            if (e < npairs) {
                int pb = grp8;
                for (; pb + 8 < G; pb += 16) {
                    const double v0 = __ldcg(a.dotpart + (size_t)pb * 64 + e);
                    const double v1 = __ldcg(a.dotpart + (size_t)(pb + 8) * 64 + e);
                    g0 += v0;
                    g1 += v1;
                }
                if (pb < G) g0 += __ldcg(a.dotpart + (size_t)pb * 64 + e);
            }
            u_s[grp8 * 64 + e] = g0 + g1;
            for (int i = tid; i < ka * ka; i += NTH) {
                const int r = i / ka, c = i - r * ka;
                Gs[i] = (r == a.comp || c == a.comp) ? 0.0 : a.gram_t[r * R + c];
            }
            __syncthreads();
            if (tid < npairs) {
                double t = 0.0;
#pragma unroll
                for (int k = 0; k < 8; ++k) t += u_s[k * 64 + tid];
                dots_s[tid] = t;
            }
            __syncthreads();
            if (tid < ka) {
                Gs[tid * ka + a.comp] = dots_s[tid];
                Gs[a.comp * ka + tid] = dots_s[tid];
                if (b == 0) {
                    a.gram_t[tid * R + a.comp] = dots_s[tid];
                    a.gram_t[a.comp * R + tid] = dots_s[tid];
                }
            }
            __syncthreads();
        }
        if (tid == 0) {
            // normal equations on unit-norm score columns; a column that is zero or dependent on the earlier ones gets
            // the coefficient 0, like the reference's lstsq (small.cu: solve_coef_kernel, same arithmetic)
            for (int i = 0; i < ka; ++i) {
                const double g = Gs[i * ka + i];
                drop[i] = !(g > 0.0) ? 1.0 : 0.0;
                dinv[i] = drop[i] != 0.0 ? 0.0 : 1.0 / sqrt(g);
            }
            for (int i = 0; i < ka; ++i) {
                for (int j = 0; j <= i; ++j) {
                    double sv = (drop[i] != 0.0 || drop[j] != 0.0) ? (i == j ? 1.0 : 0.0) : Gs[i * ka + j] * dinv[i] * dinv[j];
                    for (int q = 0; q < j; ++q) sv -= Lm[i * ka + q] * Lm[j * ka + q];
                    if (i == j) {
                        if (!(sv > 1e-14)) {  // no independent part left in column i
                            drop[i] = 1.0;
                            for (int q = 0; q < i; ++q) Lm[i * ka + q] = 0.0;
                            sv = 1.0;
                        }
                        Lm[i * ka + i] = sqrt(sv);
                    } else {
                        Lm[i * ka + j] = sv / Lm[j * ka + j];
                    }
                }
            }
            for (int i = 0; i < ka; ++i) {
                double sv = drop[i] != 0.0 ? 0.0 : dots_s[ka + i] * dinv[i];
                for (int q = 0; q < i; ++q) sv -= Lm[i * ka + q] * ys[q];
                ys[i] = sv / Lm[i * ka + i];
            }
            for (int i = ka - 1; i >= 0; --i) {
                double sv = ys[i];
                for (int q = i + 1; q < ka; ++q) sv -= Lm[q * ka + i] * xs[q];
                xs[i] = drop[i] != 0.0 ? 0.0 : sv / Lm[i * ka + i];
            }
            for (int i = 0; i < ka; ++i) xs[i] *= dinv[i];  // the coefficients of this component
            if (b == 0) {
                for (int i = 0; i < ka; ++i) a.coef[i * R + a.comp] = xs[i];
                a.trips_out[a.comp] = trip;
                a.conv_out[a.comp] = done_trip >= 0 ? 1 : 0;
            }
        }
        __syncthreads();
        // Y deflation of this CTA's rows (tpls.py:113) and their share of the residual norm of Y
        double ssy = 0.0;
        for (int k = tid; k < nblk; k += NTH) {
            const long long r = r_lo + k;
            double sv = 0.0;
            for (int bb = 0; bb < ka; ++bb) sv = fma(a.T[(size_t)bb * a.n_rows + r], xs[bb], sv);
            double sw = 1.0;
            if (a.row_w != nullptr) {
                sw = a.row_w[r];
                if (sw == 0.0) continue;  // a held-out row of Y stays 0 (its score can be NaN)
                sv *= sw;
            }
            double* yr = a.y_rw + (size_t)r * a.pitch_y;
            double rs = 0.0;
#pragma unroll
            for (int c = 0; c < 8; ++c)
                if (c < M) {
                    const double yv = fma(-sv, q_s[c], yr[c]);
                    yr[c] = yv;
                    rs = fma(yv, yv, rs);
                }
            ssy = fma(sw, rs, ssy);
        }
        ssy = warp_sum(ssy);
        if (lane == 0) qw_s[warp][0] = ssy;
        __syncthreads();
        if (tid == 0) {
            double t = 0.0;
#pragma unroll
            for (int w = 0; w < NWARP; ++w) t += qw_s[w][0];
            a.sspart_y[b] = t;
        }
    }
    if (b == 0) {
        if (tid < a.pitch_y) a.qvec[tid] = tid < M ? q_s[tid] : 0.0;
        if (tid < M) {
            a.qcol[tid] = q_s[tid];
            a.q_prev[tid] = q_s[tid];
        }
        if (tid == 0) {
            a.bar[0] = bar_gen;  // the generation this launch ends on (every CTA has passed its last barrier)
            a.ctrl->done_trip = done_trip;
            a.ctrl->trips_taken = trip;
            a.ctrl->last_d2 = d2_last;
            a.ctrl->trip = trip;
            a.ctrl->stop = 1;
        }
    }
}

}  // namespace

cudaError_t launch_cov_loop(const CovLoopArgs& a, size_t smem_bytes, bool use_smem, cudaStream_t s) {
    if (a.n_tasks < 1 || a.n_tasks > 8 || a.m > 8) return cudaErrorInvalidValue;
    auto kern = (use_smem && smem_bytes > 0) ? cov_loop_kernel<true> : cov_loop_kernel<false>;
    const size_t smem = (use_smem && smem_bytes > 0) ? smem_bytes : 0;
    if (smem > 0) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(a.n_tasks);
    cfg.blockDim = dim3(kRank1Threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = a.n_tasks;
    at[0].val.clusterDim.y = 1;
    at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at;
    cfg.numAttrs = (pdl_enabled() && !pdl_take_hold()) ? 2 : 1;
    return cudaLaunchKernelEx(&cfg, kern, a);
}

size_t resident_min_smem() { return kResidentScratch; }

int resident_fine_stamps(long long* out32) {
#ifdef TPLS_PROBE
    if (cudaMemcpyFromSymbol(out32, g_fine, sizeof(long long) * 32) != cudaSuccess) return 0;
    long long z[32] = {};
    cudaMemcpyToSymbol(g_fine, z, sizeof z);
    return 1;
#else
    (void)out32;
    return 0;
#endif
}

cudaError_t launch_resident_loop(const ResidentArgs& a_in, int n_ctas, size_t r1_smem_bytes, cudaStream_t s) {
    ResidentArgs a = a_in;
    if (a.n_tensors < 1 || a.n_tensors > kMaxTensors || a.m > 8 || a.pitch_y > 8 || n_ctas < a.n_tensors || n_ctas > kRank1Threads) return cudaErrorInvalidValue;
    const bool in_smem = a.r1_in_smem != 0 && r1_smem_bytes > 0;
    auto kern = in_smem ? resident_loop_kernel<true> : resident_loop_kernel<false>;
    // dynamic shared memory: [rank-1 workspace or the scratch of the other phases | row cache]
    const size_t front = (std::max(in_smem ? r1_smem_bytes : (size_t)0, kResidentScratch) + 127) & ~(size_t)127;
    static const size_t dyn_max[2] = {
        [] {
            cudaFuncAttributes fa{};
            int dev = 0, optin = 0;
            if (cudaFuncGetAttributes(&fa, resident_loop_kernel<false>) != cudaSuccess || cudaGetDevice(&dev) != cudaSuccess ||
                cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
                return (size_t)0;
            return (size_t)optin > fa.sharedSizeBytes ? (size_t)optin - fa.sharedSizeBytes : (size_t)0;
        }(),
        [] {
            cudaFuncAttributes fa{};
            int dev = 0, optin = 0;
            if (cudaFuncGetAttributes(&fa, resident_loop_kernel<true>) != cudaSuccess || cudaGetDevice(&dev) != cudaSuccess ||
                cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
                return (size_t)0;
            return (size_t)optin > fa.sharedSizeBytes ? (size_t)optin - fa.sharedSizeBytes : (size_t)0;
        }()};
    static const bool cache_on = [] {
        const char* v = getenv("TPLS_RESIDENT_CACHE");  // =0: every pass reads its rows from L2 (A/B switch)
        return v == nullptr || *v != '0';
    }();
    size_t w_bytes = 0;
    int n_big = 0;  // coupled tensors whose Z has two or more modes (their rank-1 step is the expensive kind)
    for (int l = 0; l < a.n_tensors; ++l) {
        w_bytes += (size_t)a.x[l].pitch * sizeof(double);
        n_big += a.r1[l].nmodes >= 2 ? 1 : 0;
    }
    // kron(w) of all tensors in shared memory, behind the rank-1 workspace, when it is at most kResidentScratch bytes
    w_bytes = w_bytes <= kResidentScratch ? ((w_bytes + 127) & ~(size_t)127) : 0;
    a.w_off = w_bytes ? (unsigned)front : 0u;
    static const bool everywhere_on = [] {
        const char* v = getenv("TPLS_RESIDENT_R1_ALL");  // =0: the rank-1 step on the first L CTAs only (A/B switch)
        return v == nullptr || *v != '0';
    }();
    a.r1_everywhere = (everywhere_on && in_smem && w_bytes != 0 && n_big <= 1) ? 1 : 0;
    const size_t head = front + w_bytes;
    const long long per = (a.n_rows + n_ctas - 1) / n_ctas;
    const size_t room = dyn_max[in_smem ? 1 : 0] > head ? dyn_max[in_smem ? 1 : 0] - head : 0;
    // Who gets the room: Y and the narrow tensors all rows of the block first (a few KB buy a whole L2 round trip per
    // pass: their rows past the cached ones would be fetched behind the wide tensor's), the widest tensor what is left.
    size_t left = cache_on ? room : 0;
    a.y_cache_rows = (int)std::min<long long>(per, (long long)(left / ((size_t)a.pitch_y * 8)));
    left -= (size_t)a.y_cache_rows * a.pitch_y * 8;
    int order[kMaxTensors];
    for (int l = 0; l < a.n_tensors; ++l) order[l] = l;
    std::sort(order, order + a.n_tensors, [&](int p, int q) {
        const size_t bp = (size_t)a.x[p].pitch * (a.x[p].dtype == 0 ? 4 : 8), bq = (size_t)a.x[q].pitch * (a.x[q].dtype == 0 ? 4 : 8);
        return bp != bq ? bp < bq : p < q;
    });
    a.cache_rows = (int)per;  // rows that every tensor has in shared memory
    size_t cached_bytes = (size_t)a.y_cache_rows * a.pitch_y * 8;
    for (int i = 0; i < a.n_tensors; ++i) {
        ResidentTensor& X = a.x[order[i]];
        const size_t rb = (size_t)X.pitch * (X.dtype == 0 ? 4 : 8);
        X.cache_rows = (int)std::min<long long>(per, (long long)(left / rb));
        left -= (size_t)X.cache_rows * rb;
        cached_bytes += (size_t)X.cache_rows * rb;
        a.cache_rows = std::min(a.cache_rows, X.cache_rows);
    }
    a.cache_off = (unsigned)head;
    const size_t smem = head + cached_bytes;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    // A cooperative launch: the CTAs spin on each other at the grid barriers, so all of them must be resident at once
    // (the driver checks it and schedules them together; a plain launch would also fit -- one CTA per SM -- unless
    // another stream holds SMs).  TPLS_RESIDENT_COOP=0 launches it as an ordinary kernel.
    static const bool coop = [] {
        const char* v = getenv("TPLS_RESIDENT_COOP");
        return v == nullptr || *v != '0';
    }();
    if (!coop) {
        launch_k(kern, dim3(n_ctas), dim3(kRank1Threads), smem, s, a);
        return cudaGetLastError();
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(n_ctas);
    cfg.blockDim = dim3(kRank1Threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeCooperative;
    at[0].val.cooperative = 1;
    cfg.attrs = at;
    cfg.numAttrs = 1;
    pdl_take_hold();
    return cudaLaunchKernelEx(&cfg, kern, a);
}

size_t rank1_workspace_doubles(int nmodes, const int* dims, int* nmax_out, int* zs_len_out, int* mt_len_out,
                               int* tab_cols_out) {
    long long p = 1;
    int sumd = 0, maxd = 0;
    for (int m = 0; m < nmodes; ++m) {
        p *= dims[m];
        sumd += dims[m];
        maxd = std::max(maxd, dims[m]);
    }
    long long nmax = 1, zs_len = (p + 3) & ~3ll, mt_len = 0, rest = 0, tab_cols = 0;
    if (nmodes == 2) {
        // [Z padded | factors | Z^T padded | Gram, two squaring buffers | vector]
        nmax = std::min(dims[0], dims[1]);
        zs_len = ((long long)dims[0] * ldp(dims[1]) + 3) & ~3ll;
        mt_len = ((long long)dims[1] * ldp(dims[0]) + 3) & ~3ll;
        rest = mt_len + 3ll * up8((int)nmax) * ldp((int)nmax) + up4(maxd);
    } else if (nmodes >= 3) {
        // [Z | factors | per-mode HOSVD areas, reused afterwards for the index table and the unfolding copies]
        long long areas = 0;
        for (int m = 0; m < nmodes; ++m) {
            const long long dk = dims[m], mk = p / dims[m];
            nmax = std::max(nmax, std::min(dk, mk));
            areas += mode_ws((int)dk, (int)mk).total;
            tab_cols += mk;
        }
        const long long tc4 = (tab_cols + 3) & ~3ll;
        // after the HOSVD start the areas hold the index table (4 or 8 shorts per column, rounded up to whole
        // doubles) and the row-major copies of the unfoldings of modes 1..
        const long long dgd = (tc4 * 4 * ((nmodes - 1 + 3) / 4) * 2 + 7) / 8;
        const long long tables = ((dgd + 3) & ~3ll) + (long long)(nmodes - 1) * ((p + 3) & ~3ll);
        rest = std::max(areas, tables);
        mt_len = rest;
    }
    if (nmax_out) *nmax_out = (int)nmax;
    if (zs_len_out) *zs_len_out = (int)zs_len;
    if (mt_len_out) *mt_len_out = (int)mt_len;
    if (tab_cols_out) *tab_cols_out = (int)tab_cols;
    return (size_t)(zs_len + up4(sumd) + rest + 16);
}

cudaError_t launch_rank1(const Rank1Args& a, size_t smem_bytes, cudaStream_t s) {
    if (smem_bytes > 0 && a.t[0].use_smem) {
        cudaError_t e =
            cudaFuncSetAttribute(rank1_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
        if (e != cudaSuccess) return e;
        launch_k(rank1_kernel<true>, dim3(a.n_tasks), dim3(kRank1Threads), smem_bytes, s, a);
    } else {
        launch_k(rank1_kernel<false>, dim3(a.n_tasks), dim3(kRank1Threads), 0, s, a);
    }
    return cudaGetLastError();
}

}  // namespace tpls
