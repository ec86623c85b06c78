// Streaming column/row passes over an X (or Y) shard -- see passes.cuh.
#include "passes.cuh"
#include "stream_common.cuh"

#include <algorithm>
#include <cstdlib>

namespace tpls {

// ---------------------------------------------------------------------------
// geometry
// ---------------------------------------------------------------------------
// Tuning overrides for experiments (tools/opbench.py): TPLS_TILE_KB, TPLS_SMEM_KB (per-CTA staging budget),
// TPLS_CTAS_PER_SM.  Unset in normal use.
int tune_env(const char* name, int dflt) {
    const char* v = getenv(name);
    return (v != nullptr && *v) ? atoi(v) : dflt;
}

static int pow2_ceil(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

PassGeom make_geom(long long n_rows, int p, int pitch, int elem_size, int sm_count, int y_row_bytes) {
    PassGeom g{};
    const int vec = 16 / elem_size;
    g.n_rows = n_rows;
    g.p = p;
    g.pitch = pitch;
    g.elem_size = elem_size;
    const int cg_total = pitch / vec;
    const int max_cg = kConsumers * kMaxCpt;
    g.n_slabs = (cg_total + max_cg - 1) / max_cg;
    const int slab_cg = (cg_total + g.n_slabs - 1) / g.n_slabs;
    g.slab_w = slab_cg * vec;
    // as few lanes per row as kMaxCpt groups per lane allow: more work per thread and row
    g.lpr = std::min(kConsumers, pow2_ceil((slab_cg + kMaxCpt - 1) / kMaxCpt));
    if (slab_cg % kConsumers == 0 && (slab_cg / kConsumers == 1 || slab_cg / kConsumers == 2))
        g.lpr = kConsumers;  // exact fit: the compile-time FULL path applies
    {
        const int need = (slab_cg + g.lpr - 1) / g.lpr;
        g.cpt = need <= 1 ? 1 : (need <= 2 ? 2 : 4);
    }
    g.rpt = kConsumers / g.lpr;
    const long long row_bytes = (long long)(g.n_slabs == 1 ? pitch : g.slab_w) * elem_size;
    long long tr = std::max<long long>(1, ((long long)tune_env("TPLS_TILE_KB", 32) * 1024) / row_bytes);
    tr = std::min<long long>(tr, std::max<long long>(1, n_rows));
    tr = std::min<long long>(tr, 4096);
    if (y_row_bytes > 0) tr = std::min<long long>(tr, std::max<long long>(2, 16384 / y_row_bytes));  // staged rows of Y <= 16 KB
    g.tile_rows = (int)tr;
    const long long stage_bytes = tr * (row_bytes + y_row_bytes);
    g.stages = (int)std::max<long long>(2, std::min<long long>(kMaxStages, ((long long)tune_env("TPLS_SMEM_KB", 100) * 1024) / stage_bytes));
    const long long n_tiles = (n_rows + tr - 1) / tr;
    const long long want = std::max(1, (sm_count * tune_env("TPLS_CTAS_PER_SM", 2)) / g.n_slabs);
    g.grid_x = (int)std::max<long long>(1, std::min<long long>(n_tiles, want));
#ifdef TPLS_PROBE
    g.dbg = tune_env("TPLS_DBG", 0);
#endif
    return g;
}

static size_t stage_bytes_of(const PassGeom& g) {
    return (size_t)g.tile_rows * (g.n_slabs == 1 ? g.pitch : g.slab_w) * g.elem_size;
}

size_t colpass_smem(const PassGeom& g, int pitch_y) {
    const size_t tiles = g.stages * (stage_bytes_of(g) + (size_t)g.tile_rows * pitch_y * sizeof(double));
    const size_t red = (size_t)kConsumers * g.cpt * (16 / g.elem_size) * sizeof(double);  // row-lane fold
    return std::max(tiles, red) + 256;  // + barriers (128) + q (kMaxFusedResp doubles)
}

// ---------------------------------------------------------------------------
// column pass
// ---------------------------------------------------------------------------
// FULL: one slab, every thread owns CPT valid column groups of every row (pitch == kConsumers * VEC * CPT,
// e.g. 4096 fp32 columns): layout constants fold at compile time and the row loop carries no bounds checks.
template <typename XT, int CPT, bool MASKED, int FLAGS, bool FULL>
__global__ void __launch_bounds__(kThreads, 2) colpass_kernel(const __grid_constant__ ColPassArgs a) {
    pdl_prologue();
    constexpr int VEC = VecOf<XT>::N;
    constexpr bool DEFLATE = (FLAGS & PF_DEFLATE) != 0;
    constexpr bool WRITE = (FLAGS & PF_WRITE) != 0;
    constexpr bool CONTRACT = (FLAGS & PF_CONTRACT) != 0;
    constexpr bool SUMSQ = (FLAGS & PF_SUMSQ) != 0;
    constexpr bool COLSTAT = (FLAGS & PF_COLSTAT) != 0;
    constexpr bool ZACC = CONTRACT || COLSTAT;

    if (trip_is_dead(a.ctrl, a.trip)) return;

    extern __shared__ __align__(128) unsigned char smem[];
    const PassGeom& g = a.g;
    const int c0 = blockIdx.y * g.slab_w;
    const int slab_cols = min(g.slab_w, g.pitch - c0);
    const int lpr = FULL ? kConsumers : g.lpr;
    const int rpt = FULL ? 1 : g.rpt;
    const int srow = FULL ? kConsumers * VecOf<XT>::N * CPT : ((g.n_slabs == 1) ? g.pitch : g.slab_w);
    const size_t stage_elems = (size_t)g.tile_rows * srow;
    XT* tiles = reinterpret_cast<XT*>(smem);
    // u = Y q formed here (CONTRACT with a.y): the rows of Y are staged behind the X tiles of the ring
    const bool use_y = CONTRACT && a.y != nullptr;
    const int pitch_y = use_y ? a.pitch_y : 0;
    const size_t ystage = (size_t)g.tile_rows * pitch_y;
    double* ytiles = reinterpret_cast<double*>(smem + (size_t)g.stages * stage_elems * sizeof(XT));
    const size_t tile_area = max((size_t)g.stages * (stage_elems * sizeof(XT) + ystage * sizeof(double)),
                                 (size_t)kConsumers * CPT * VEC * sizeof(double));
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + tile_area);
    uint64_t* empty = full + kMaxStages;
    double* qs = reinterpret_cast<double*>(smem + tile_area + 128);

    if (threadIdx.x == 0) {
        for (int s = 0; s < g.stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kConsumers / 32);
        }
        fence_mbar_init();
    }
    if (use_y && threadIdx.x < kMaxFusedResp) qs[threadIdx.x] = (int)threadIdx.x < pitch_y ? a.q[threadIdx.x] : 0.0;
    __syncthreads();

    if (threadIdx.x >= kConsumers) {
        if (threadIdx.x == kConsumers)
            produce_tiles<XT>(g, reinterpret_cast<const XT*>(a.x_in), tiles, full, empty, c0, slab_cols, srow,
                              use_y ? a.y : nullptr, pitch_y, ytiles);
        return;
    }

    const int tid = threadIdx.x;
    const int cl = tid & (lpr - 1);
    const int rl = tid / lpr;
    const int lane = tid & 31;

    double wreg[CPT][VEC];
    double zacc[CPT][VEC];
    double cacc[CPT][VEC];
    bool cvalid[CPT];
#pragma unroll
    for (int k = 0; k < CPT; ++k) {
        const int cg = cl + k * lpr;
        cvalid[k] = FULL ? true : (cg * VEC < slab_cols);
#pragma unroll
        for (int j = 0; j < VEC; ++j) {
            zacc[k][j] = 0.0;
            cacc[k][j] = 0.0;
            wreg[k][j] = (DEFLATE && cvalid[k]) ? a.col_w[c0 + cg * VEC + j] : 0.0;
        }
    }
    double ss = 0.0;
    int nmiss = 0;  // COLSTAT: unobserved entries seen by this thread, whatever the row weights

    XT* xo = reinterpret_cast<XT*>(a.x_out);
    const TileWalk tw = tile_walk(g);
    const long long n_tiles = (g.n_rows + g.tile_rows - 1) / g.tile_rows;
    RingPos rp;
    for (long long tile = tw.first; tile < tw.end; tile += tw.step, rp.advance(g.stages)) {
        const int s = rp.idx;
        const long long r0 = tile * g.tile_rows;
        int rows = tile_rows_of(g, tile, n_tiles);
        mbar_wait(&full[s], rp.phase);
#ifdef TPLS_PROBE
        if (g.dbg & 16) rows = 0;  // data movement only
#endif
        const XT* tp = tiles + s * stage_elems;
        const double* yp = ytiles + s * ystage;
        for (int r = rl; r < rows; r += rpt) {
            const long long grow = r0 + r;
            double ar = 1.0, ur = 0.0;
            if (DEFLATE && a.row_a != nullptr) ar = __ldg(a.row_a + grow);
            // a NaN score: the row has a tensor without observed entries, so its later scores are NaN whatever it
            // holds; left as it is, it keeps NaN out of the sums over rows (NaN * 0 is NaN)
            if (DEFLATE && !(ar == ar)) ar = 0.0;
            if (CONTRACT) {
                if (use_y) {
                    // (a compile-time unrolled variant with two chains was measured against this loop on one box:
                    //  1 % slower, although it executes ~25 % fewer instructions -- the pass waits on the copy barrier)
                    const double2* yr = reinterpret_cast<const double2*>(yp + (size_t)r * pitch_y);
                    for (int m = 0; m < pitch_y; m += 2) {
                        const double2 yv = yr[m >> 1];
                        ur = fma(yv.x, qs[m], ur);
                        ur = fma(yv.y, qs[m + 1], ur);
                    }
                } else {
                    ur = __ldg(a.row_u + grow);
                }
            }
            // optional 0/1 sample weights (cross-validation folds): weighted column statistics and
            // weighted residual norm; the row's own sum of squares is folded in once per row
            const double sw = ((COLSTAT || SUMSQ) && a.row_sw != nullptr) ? __ldg(a.row_sw + grow) : 1.0;
            // the row's sum of squares in two chains, folded into ss (times the row weight) once per row.  (Measured on
            // one box against a single chain: no difference -- the read-only residual pass is held back by its three
            // conversions per element, fp32 -> fp64, to the storage type and back, not by the dependent DFMAs.)
            double rs[2] = {0.0, 0.0};
#pragma unroll
            for (int k = 0; k < CPT; ++k) {
                if (!FULL && !cvalid[k]) continue;
                const int cg = cl + k * lpr;
                Pack<XT> in, out;
                in.v = *reinterpret_cast<const typename VecOf<XT>::type*>(tp + (size_t)r * srow + cg * VEC);
#pragma unroll
                for (int j = 0; j < VEC; ++j) {
                    const XT xs = in.e[j];
                    double xd = (double)xs;
                    if (DEFLATE) {
                        xd = fma(-ar, wreg[k][j], xd);
                        if (WRITE) {
                            out.e[j] = (XT)xd;       // NaN stays NaN
                            xd = (double)out.e[j];   // later passes see the stored (rounded) value
                        }
                        // (the read-only residual pass after the last component stores nothing: it sums the squares
                        // of the unrounded values -- for fp32 storage that differs from the sum over the would-be
                        // stored values by ~6e-8 / sqrt(elements) relative, and saves two of its three conversions
                        // per element, which are what bounds it)
                    }
                    // observed after centring, as transform() counts: an entry of a column whose mean is NaN (no
                    // observed training entry) is missing
                    const bool ob = MASKED ? (xd == xd) : true;
                    if (MASKED && !ob) xd = 0.0;
                    if (CONTRACT) zacc[k][j] = fma(xd, ur, zacc[k][j]);
                    if (COLSTAT) {
                        zacc[k][j] = fma(xd, sw, zacc[k][j]);
                        cacc[k][j] += ob ? sw : 0.0;
                        nmiss += ob ? 0 : 1;
                    }
                    if (SUMSQ) rs[j & 1] = fma(xd, xd, rs[j & 1]);
                }
                if (WRITE) {
                    __stcs(reinterpret_cast<typename VecOf<XT>::type*>(xo + grow * g.pitch + c0 + cg * VEC), out.v);
                }
            }
            if (SUMSQ) {
                if (sw != 0.0) ss = fma(sw, rs[0] + rs[1], ss);  // a held-out row adds nothing, even a NaN
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
    }

    // ---- epilogue: fold row lanes, publish this CTA's column partials ----
    if (ZACC) {
        double* red = reinterpret_cast<double*>(smem);
        // red[row lane][column group slot k][lane column][element]: kConsumers * CPT * VEC doubles in total
        const int wcols = lpr * VEC;
        for (int pass = 0; pass < (COLSTAT ? 2 : 1); ++pass) {
            double(*acc)[VEC] = pass == 0 ? zacc : cacc;
            double* outp = (pass == 0 ? a.zpart : a.cntpart) + (size_t)blockIdx.x * g.pitch + c0;
            if (rpt > 1) {
                named_bar_sync(1, kConsumers);
#pragma unroll
                for (int k = 0; k < CPT; ++k)
#pragma unroll
                    for (int j = 0; j < VEC; ++j) red[((size_t)rl * CPT + k) * wcols + cl * VEC + j] = acc[k][j];
                named_bar_sync(1, kConsumers);
                // every thread folds a share of the (column, element) pairs over the row lanes
                for (int e = tid; e < CPT * wcols; e += kConsumers) {
                    const int k = e / wcols, ce = e - k * wcols;       // ce = cl * VEC + j
                    const int cg = ce / VEC + k * lpr;
                    if (cg * VEC >= slab_cols) continue;
                    double t = 0.0;
                    for (int q = 0; q < rpt; ++q) t += red[((size_t)q * CPT + k) * wcols + ce];
                    outp[cg * VEC + (ce % VEC)] = t;
                }
            } else {
#pragma unroll
                for (int k = 0; k < CPT; ++k) {
                    if (!cvalid[k]) continue;
                    const int cg = cl + k * lpr;
#pragma unroll
                    for (int j = 0; j < VEC; ++j) outp[cg * VEC + j] = acc[k][j];
                }
            }
        }
    }
    if (SUMSQ || (COLSTAT && a.sspart != nullptr)) {
        double* red = reinterpret_cast<double*>(smem);
        if (COLSTAT) ss = (double)nmiss;
        named_bar_sync(1, kConsumers);
        ss = warp_sum(ss);
        if (lane == 0) red[tid >> 5] = ss;
        named_bar_sync(1, kConsumers);
        if (tid == 0) {
            double t = 0.0;
            for (int w = 0; w < kConsumers / 32; ++w) t += red[w];
            a.sspart[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = t;
        }
    }
}

// ---------------------------------------------------------------------------
// small finishing kernels
// ---------------------------------------------------------------------------
// 32 columns x 8 part-groups per CTA: each thread folds every 8th partial of its column (coalesced 256-byte
// rows, several loads in flight), the 8 groups meet in shared memory.  Fixed order => bit-reproducible.
__global__ void __launch_bounds__(256) reduce_cols_kernel(const ReduceArgs a) {
    pdl_prologue();
    if (trip_is_dead(a.ctrl, a.trip)) return;
    __shared__ double fold[8][33];
    __shared__ double red[40];
    const int cl = threadIdx.x & 31, q = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + cl;
    double t0 = 0.0, t1 = 0.0, t2 = 0.0, t3 = 0.0;
    if (c < a.n_cols) {
        int b = q;
        for (; b + 24 < a.n_parts; b += 32) {
            t0 += a.part[(size_t)(b + 0) * a.stride + c];
            t1 += a.part[(size_t)(b + 8) * a.stride + c];
            t2 += a.part[(size_t)(b + 16) * a.stride + c];
            t3 += a.part[(size_t)(b + 24) * a.stride + c];
        }
        for (; b < a.n_parts; b += 8) t0 += a.part[(size_t)b * a.stride + c];
    }
    fold[q][cl] = (t0 + t1) + (t2 + t3);
    __syncthreads();
    if (q == 0 && c < a.n_cols) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += fold[k][cl];
        a.out[c] = t;
    }
    if (a.ss_out != nullptr && blockIdx.x == 0) {
        double t = 0.0;
        for (int i = threadIdx.x; i < a.n_ss; i += blockDim.x) t += a.sspart[i];
        t = block_sum(t, red);
        if (threadIdx.x == 0) a.ss_out[0] = t;
    }
}

cudaError_t launch_reduce_cols(const ReduceArgs& a, cudaStream_t s) {
    const int blocks = std::max(1, (a.n_cols + 31) / 32);
    launch_k(reduce_cols_kernel, dim3(blocks), dim3(256), 0, s, a);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) fold_sets_kernel(const __grid_constant__ FoldArgs a) {
    pdl_prologue();
    if (trip_is_dead(a.ctrl, 0)) return;
    __shared__ double fold[8][37];  // 8 x 37 >= 32 x 9: doubles as the [32][9] area of fold_narrow
    const int cl = threadIdx.x & 31, q = threadIdx.x >> 5;
    int c_base = 0;
    const FoldSet& S = a.sets[fold_locate(a.sets, a.n_sets, blockIdx.x, &c_base)];
    if (S.n_cols <= 8) {  // narrow set: 32 part-groups per column
        const double t = fold_narrow(S, reinterpret_cast<double(*)[9]>(&fold[0][0]));
        if ((threadIdx.x >> 3) == 0 && (int)(threadIdx.x & 7) < S.n_cols) a.out[S.off + (threadIdx.x & 7)] = t;
        return;
    }
    const int c = c_base + cl;
    fold[q][cl] = fold_share(S, c, q);
    __syncthreads();
    if (q == 0 && c < S.n_cols) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) t += fold[k][cl];
        a.out[S.off + c] = t;
    }
}

cudaError_t launch_fold_sets(const FoldArgs& a, cudaStream_t s) {
    if (a.n_sets < 1 || a.n_sets > kMaxFoldSets) return cudaErrorInvalidValue;
    const int blocks = std::max(1, fold_chunks(a.sets, a.n_sets));
    launch_k(fold_sets_kernel, dim3(blocks), dim3(256), 0, s, a);
    return cudaGetLastError();
}

__global__ void __launch_bounds__(256) row_finish_kernel(const RowFinishArgs a) {
    pdl_prologue();
    if (trip_is_dead(a.ctrl, a.trip)) return;
    __shared__ double red[40];
    double d2 = 0.0;
    double qacc[kMaxFusedResp];
#pragma unroll
    for (int m = 0; m < kMaxFusedResp; ++m) qacc[m] = 0.0;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r < a.n_rows;
         r += (long long)gridDim.x * blockDim.x) {
        double v = 0.0, cnt = 0.0;
        for (int s = 0; s < a.n_slabs; ++s) {
            v += a.tpart[(size_t)s * a.n_rows + r];
            if (a.cpart != nullptr) cnt += a.cpart[(size_t)s * a.n_rows + r];
        }
        if (a.rowcnt != nullptr) {
            if (a.cpart != nullptr) {
                cnt -= a.pads;
                a.rowcnt[r] = cnt;
            } else {
                cnt = a.rowcnt[r];
            }
            v = v / cnt * a.p_total;
        }
        const double old = a.t_out[r];
        double nv = v;
        if (a.epi == 1) nv = old + v;
        if (a.epi == 2) nv = (old + v) / a.div;
        a.t_out[r] = nv;
        const double d = old - nv;
        d2 = fma(d, d, d2);
        if (a.qpart != nullptr) {
#pragma unroll
            for (int m = 0; m < kMaxFusedResp; ++m)
                if (m < a.pitch_y) {
                    const double y = a.y[r * a.pitch_y + m];
                    if (y != 0.0) qacc[m] = fma(y, nv, qacc[m]);  // a held-out row (Y row 0) adds nothing, even a NaN t
                }
        }
    }
    if (a.d2part != nullptr) {
        d2 = block_sum(d2, red);
        if (threadIdx.x == 0) a.d2part[blockIdx.x] = d2;
    }
    if (a.qpart != nullptr) {
#pragma unroll
        for (int m = 0; m < kMaxFusedResp; ++m) {
            const double t = block_sum(qacc[m], red);
            if (threadIdx.x == 0) a.qpart[(size_t)blockIdx.x * kMaxFusedResp + m] = t;
        }
    }
}

int row_finish_grid(long long n_rows) {
    return (int)std::max<long long>(1, std::min<long long>(296, (n_rows + 255) / 256));
}

cudaError_t launch_row_finish(const RowFinishArgs& a, int* grid_out, cudaStream_t s) {
    const int blocks = row_finish_grid(a.n_rows);
    if (grid_out) *grid_out = blocks;
    launch_k(row_finish_kernel, dim3(blocks), dim3(256), 0, s, a);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------
// dispatch
// ---------------------------------------------------------------------------
template <typename XT, int CPT, bool MASKED, int FLAGS, bool FULL>
static cudaError_t run_colpass_impl(const ColPassArgs& a, cudaStream_t s) {
    auto kern = colpass_kernel<XT, CPT, MASKED, FLAGS, FULL>;
    size_t smem = colpass_smem(a.g, ((FLAGS & PF_CONTRACT) && a.y != nullptr) ? a.pitch_y : 0);
#ifdef TPLS_PROBE
    smem += (size_t)tune_env("TPLS_DBG_COLPAD_KB", 0) * 1024;  // unused tail: does the footprint alone matter?
#endif
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    dim3 grid(a.g.grid_x, a.g.n_slabs);
    launch_k(kern, dim3(grid), dim3(kThreads), smem, s, a);
    return cudaGetLastError();
}

template <typename XT, int CPT, bool MASKED, int FLAGS>
static cudaError_t run_colpass(const ColPassArgs& a, cudaStream_t s) {
    const bool full = a.g.n_slabs == 1 && a.g.lpr == kConsumers && a.g.cpt == CPT &&
                      a.g.pitch == kConsumers * (16 / (int)sizeof(XT)) * CPT;
    return full ? run_colpass_impl<XT, CPT, MASKED, FLAGS, true>(a, s) : run_colpass_impl<XT, CPT, MASKED, FLAGS, false>(a, s);
}

template <typename XT, int CPT, bool MASKED>
static cudaError_t colpass_flags(int flags, const ColPassArgs& a, cudaStream_t s) {
    switch (flags) {
        case PF_COLSTAT:
            return run_colpass<XT, CPT, true, PF_COLSTAT>(a, s);
        case PF_CONTRACT:
            return run_colpass<XT, CPT, MASKED, PF_CONTRACT>(a, s);
        case PF_DEFLATE | PF_WRITE | PF_CONTRACT | PF_SUMSQ:
            return run_colpass<XT, CPT, MASKED, PF_DEFLATE | PF_WRITE | PF_CONTRACT | PF_SUMSQ>(a, s);
        case PF_DEFLATE | PF_WRITE | PF_SUMSQ:
            return run_colpass<XT, CPT, MASKED, PF_DEFLATE | PF_WRITE | PF_SUMSQ>(a, s);
        case PF_DEFLATE | PF_SUMSQ:
            return run_colpass<XT, CPT, MASKED, PF_DEFLATE | PF_SUMSQ>(a, s);
        default:
            return cudaErrorInvalidValue;
    }
}

template <typename XT>
static cudaError_t colpass_cpt(bool masked, int flags, const ColPassArgs& a, cudaStream_t s) {
#define TPLS_CP(C)                                                  \
    return masked ? colpass_flags<XT, C, true>(flags, a, s) : colpass_flags<XT, C, false>(flags, a, s)
    switch (a.g.cpt) {
        case 1:
            TPLS_CP(1);
        case 2:
            TPLS_CP(2);
        default:
            TPLS_CP(4);
    }
#undef TPLS_CP
}

cudaError_t launch_colpass(int dtype, bool masked, int flags, const ColPassArgs& a, cudaStream_t s) {
    return dtype == 0 ? colpass_cpt<float>(masked, flags, a, s) : colpass_cpt<double>(masked, flags, a, s);
}

}  // namespace tpls
