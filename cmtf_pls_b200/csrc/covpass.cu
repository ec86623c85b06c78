// Cross-covariance pass (SURVEY.md §8f n4): ONE read (+ write) of an X shard that
//   * centres or deflates it in place:   xn = x - a[row] * w[col]           (tpls.py:71, :109)
//   * accumulates the residual norm:      ss += xn^2                          (util.py:7-15)
//   * accumulates the cross-covariance with EVERY response column at once:
//         C[m][col] = sum_rows xn[row, col] * Y[row, m]          m < M
//     and, for a masked tensor, a second block with the rows rescaled by P / (observed entries
//     of the row), which is what the masked projection needs (missingvals.py:23-38):
//         C[M + m][col] = sum_rows xn[row, col] * Y[row, m] * P / cnt[row]
// Z = X x_1 u and q = Y't are linear in u = Y q and in the weight vector, so with C in hand the
// whole NIPALS inner iteration runs on (P x M)-sized data (rank1.cu: cov_loop_kernel) and X is
// streamed ~2.5 times per component instead of twice per inner trip.
//
// Same staging as colpass (passes.cu): producer warp, 1-D bulk async copies, mbarrier ring.  A thread
// owns ONE 16-byte column group and MR accumulators per column; column slabs along gridDim.y.
#include "passes.cuh"
#include "stream_common.cuh"

#include <algorithm>

namespace tpls {

PassGeom make_cov_geom(long long n_rows, int p, int pitch, int elem_size, int sm_count) {
    PassGeom g{};
    const int vec = 16 / elem_size;
    g.n_rows = n_rows;
    g.p = p;
    g.pitch = pitch;
    g.elem_size = elem_size;
    const int cg_total = pitch / vec;
    g.n_slabs = (cg_total + kConsumers - 1) / kConsumers;
    const int slab_cg = (cg_total + g.n_slabs - 1) / g.n_slabs;
    g.slab_w = slab_cg * vec;
    g.cpt = 1;
    g.lpr = 1;
    while (g.lpr < slab_cg) g.lpr <<= 1;
    g.lpr = std::min(g.lpr, kConsumers);
    g.rpt = kConsumers / g.lpr;
    const long long row_bytes = (long long)(g.n_slabs == 1 ? pitch : g.slab_w) * elem_size;
    long long tr = std::max<long long>(1, (24 * 1024) / row_bytes);
    tr = std::min<long long>(tr, std::max<long long>(1, n_rows));
    tr = std::min<long long>(tr, 1024);
    g.tile_rows = (int)tr;
    g.stages = 3;
    const long long n_tiles = (n_rows + tr - 1) / tr;
    const long long want = std::max(1, (sm_count * 2) / g.n_slabs);
    g.grid_x = (int)std::max<long long>(1, std::min<long long>(n_tiles, want));
    return g;
}

static size_t cov_stage_bytes(const PassGeom& g) {
    return (size_t)g.tile_rows * (g.n_slabs == 1 ? g.pitch : g.slab_w) * g.elem_size;
}

static size_t cov_ystage_bytes(const PassGeom& g, int pitch_y) { return (size_t)g.tile_rows * pitch_y * sizeof(double); }

size_t covpass_smem(const PassGeom& g, int pitch_y, int mr) {
    const size_t tiles = g.stages * (cov_stage_bytes(g) + cov_ystage_bytes(g, pitch_y));
    const size_t red = (size_t)kConsumers * (16 / g.elem_size) * mr * sizeof(double);  // row-lane fold (rpt > 1)
    return std::max(tiles, red) + 128;
}

template <typename XT, bool MASKED, int MR>
__global__ void __launch_bounds__(kThreads, 2) covpass_kernel(const __grid_constant__ CovPassArgs a) {
    pdl_prologue();
    constexpr int VEC = VecOf<XT>::N;
    constexpr int MY = MASKED ? MR / 2 : MR;  // response columns actually read

    extern __shared__ __align__(128) unsigned char smem[];
    const PassGeom& g = a.g;
    const int c0 = blockIdx.y * g.slab_w;
    const int slab_cols = min(g.slab_w, g.pitch - c0);
    const int srow = (g.n_slabs == 1) ? g.pitch : g.slab_w;
    const size_t stage_elems = (size_t)g.tile_rows * srow;
    const size_t ystage = (size_t)g.tile_rows * a.pitch_y;
    XT* tiles = reinterpret_cast<XT*>(smem);
    double* ytiles = reinterpret_cast<double*>(smem + (size_t)g.stages * stage_elems * sizeof(XT));
    const size_t tile_area = max((size_t)g.stages * (stage_elems * sizeof(XT) + ystage * sizeof(double)),
                                 (size_t)kConsumers * VEC * MR * sizeof(double));
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + tile_area);
    uint64_t* empty = full + kMaxStages;

    if (threadIdx.x == 0) {
        for (int s = 0; s < g.stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kConsumers / 32);
        }
        fence_mbar_init();
    }
    __syncthreads();
    const long long n_tiles = (g.n_rows + g.tile_rows - 1) / g.tile_rows;

    if (threadIdx.x >= kConsumers) {
        if (threadIdx.x == kConsumers) {
            // producer: the X tile (contiguous, or one row segment per row) and the matching rows of Y
            const XT* x = reinterpret_cast<const XT*>(a.x_in);
            RingPos rp;
            for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, rp.advance(g.stages)) {
                const int s = rp.idx;
                if (rp.wrapped) mbar_wait(&empty[s], rp.phase ^ 1u);
                const long long r0 = tile * g.tile_rows;
                const int rows = tile_rows_of(g, tile, n_tiles);
                XT* dst = tiles + s * stage_elems;
                const XT* src = x + r0 * g.pitch + c0;
                const uint32_t ybytes = (uint32_t)((size_t)rows * a.pitch_y * sizeof(double));
                if (g.n_slabs == 1) {
                    const uint32_t bytes = (uint32_t)((size_t)rows * g.pitch * sizeof(XT));
                    mbar_arrive_expect_tx(&full[s], bytes + ybytes);
                    bulk_g2s(dst, src, bytes, &full[s]);
                } else {
                    const uint32_t rb = (uint32_t)(slab_cols * sizeof(XT));
                    mbar_arrive_expect_tx(&full[s], rb * rows + ybytes);
                    for (int r = 0; r < rows; ++r)
                        bulk_g2s(dst + (size_t)r * srow, src + (size_t)r * g.pitch, rb, &full[s]);
                }
                bulk_g2s(ytiles + s * ystage, a.y + r0 * a.pitch_y, ybytes, &full[s]);
            }
        }
        return;
    }

    const int tid = threadIdx.x;
    const int cl = tid & (g.lpr - 1);
    const int rl = tid / g.lpr;
    const int lane = tid & 31;
    const bool cvalid = cl * VEC < slab_cols;
    double wreg[VEC];
    double acc[VEC][MR];
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
        wreg[j] = cvalid ? a.col_w[c0 + cl * VEC + j] : 0.0;
#pragma unroll
        for (int m = 0; m < MR; ++m) acc[j][m] = 0.0;
    }
    double ss = 0.0;
    XT* xo = reinterpret_cast<XT*>(a.x_out);
    const double p_total = (double)g.p;

    RingPos rp;
    for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, rp.advance(g.stages)) {
        const int s = rp.idx;
        const long long r0 = tile * g.tile_rows;
        const int rows = tile_rows_of(g, tile, n_tiles);
        mbar_wait(&full[s], rp.phase);
        const XT* tp = tiles + s * stage_elems;
        const double* yp = ytiles + s * ystage;
        if (cvalid) {
            for (int r = rl; r < rows; r += g.rpt) {
                const long long grow = r0 + r;
                double ar = a.row_a != nullptr ? __ldg(a.row_a + grow) : 1.0;
                if (!(ar == ar)) ar = 0.0;  // a NaN score: leave the row as it is (see col_pass)
                const double sw = a.row_sw != nullptr ? __ldg(a.row_sw + grow) : 1.0;
                double yv[MR];
#pragma unroll
                for (int m = 0; m < MY; ++m) yv[m] = m < a.m ? yp[(size_t)r * a.pitch_y + m] : 0.0;
                if (MASKED) {
                    // second block: rows rescaled by P / (observed entries of the row); an all-missing row
                    // gives inf * 0 = NaN exactly like the reference's 0/0 (missingvals.py:37)
                    const double sc = p_total / __ldg(a.rowcnt + grow);
#pragma unroll
                    for (int m = 0; m < MY; ++m) yv[MY + m] = yv[m] * sc;
                }
                if (sw == 0.0) {  // a held-out row adds nothing (its rescale can be inf: 0 * inf is NaN)
#pragma unroll
                    for (int m = 0; m < MR; ++m) yv[m] = 0.0;
                }
                Pack<XT> in, out;
                in.v = *reinterpret_cast<const typename VecOf<XT>::type*>(tp + (size_t)r * srow + cl * VEC);
                double rs = 0.0;
#pragma unroll
                for (int j = 0; j < VEC; ++j) {
                    const XT xs = in.e[j];
                    double xd = fma(-ar, wreg[j], (double)xs);
                    out.e[j] = (XT)xd;      // NaN stays NaN
                    xd = (double)out.e[j];  // later passes see the stored (rounded) value
                    const bool ob = MASKED ? (xd == xd) : true;  // observed after centring (NaN mean: missing)
                    if (MASKED && !ob) xd = 0.0;
#pragma unroll
                    for (int m = 0; m < MR; ++m) acc[j][m] = fma(xd, yv[m], acc[j][m]);
                    rs = fma(xd, xd, rs);
                }
                if (sw != 0.0) ss = fma(sw, rs, ss);
                __stcs(reinterpret_cast<typename VecOf<XT>::type*>(xo + grow * g.pitch + c0 + cl * VEC), out.v);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(&empty[s]);
    }

    // ---- epilogue: fold the row lanes, publish this CTA's partial of C (layout [m][pitch]) and of ss ----
    double* red = reinterpret_cast<double*>(smem);
    double* outp = a.cpart + (size_t)blockIdx.x * a.c_stride;
    if (g.rpt > 1) {
        const int wcols = g.lpr * VEC;
        named_bar_sync(1, kConsumers);
#pragma unroll
        for (int j = 0; j < VEC; ++j)
#pragma unroll
            for (int m = 0; m < MR; ++m) red[((size_t)rl * MR + m) * wcols + cl * VEC + j] = acc[j][m];
        named_bar_sync(1, kConsumers);
        if (rl == 0 && cvalid) {
#pragma unroll
            for (int j = 0; j < VEC; ++j)
#pragma unroll
                for (int m = 0; m < MR; ++m) {
                    double t = 0.0;
                    for (int q = 0; q < g.rpt; ++q) t += red[((size_t)q * MR + m) * wcols + cl * VEC + j];
                    outp[(size_t)m * g.pitch + c0 + cl * VEC + j] = t;
                }
        }
    } else if (cvalid) {
#pragma unroll
        for (int j = 0; j < VEC; ++j)
#pragma unroll
            for (int m = 0; m < MR; ++m) outp[(size_t)m * g.pitch + c0 + cl * VEC + j] = acc[j][m];
    }
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

template <typename XT, bool MASKED, int MR>
static cudaError_t run_cov(const CovPassArgs& a, cudaStream_t s) {
    auto kern = covpass_kernel<XT, MASKED, MR>;
    const size_t smem = covpass_smem(a.g, a.pitch_y, MR);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    dim3 grid(a.g.grid_x, a.g.n_slabs);
    launch_k(kern, dim3(grid), dim3(kThreads), smem, s, a);
    return cudaGetLastError();
}

template <typename XT>
static cudaError_t cov_dispatch(bool masked, int mr, const CovPassArgs& a, cudaStream_t s) {
    if (masked) {
        switch (mr) {
            case 2:
                return run_cov<XT, true, 2>(a, s);
            case 4:
                return run_cov<XT, true, 4>(a, s);
            case 8:
                return run_cov<XT, true, 8>(a, s);
            default:
                return cudaErrorInvalidValue;
        }
    }
    switch (mr) {
        case 1:
            return run_cov<XT, false, 1>(a, s);
        case 2:
            return run_cov<XT, false, 2>(a, s);
        case 4:
            return run_cov<XT, false, 4>(a, s);
        case 8:
            return run_cov<XT, false, 8>(a, s);
        default:
            return cudaErrorInvalidValue;
    }
}

cudaError_t launch_covpass(int dtype, bool masked, int mr, const CovPassArgs& a, cudaStream_t s) {
    return dtype == 0 ? cov_dispatch<float>(masked, mr, a, s) : cov_dispatch<double>(masked, mr, a, s);
}

}  // namespace tpls
