// Row pass: t[i] = sum_c x[i,c] * w[c]  (projection, reference cmtf_pls/tpls.py:97-99,
// masked variant missingvals.py:23-38; also u = Y q, tpls.py:102) -- see passes.cuh.
//
// Warp roles in one CTA (kRowThreads = 320):
//   warps 0..7  consumers  each thread owns up to 4 sixteen-byte column groups of the
//                          slab, keeps w for them in registers, and for every staged
//                          row writes ONE fp64 partial into a shared-memory slot ring;
//   warp  8     producer   one lane streams row tiles in with 1-D bulk async copies;
//   warp  9     reducer    folds the per-thread partials of a tile into t[row], applies
//                          the epilogue (coupled average, masked rescaling, ||dt||^2).
// Consumers never meet at a CTA-wide barrier: tiles and slots are handed over with
// mbarriers only.  Rows narrower than 32 column groups skip the slot ring and reduce
// with sub-warp shuffles instead.
#include "passes.cuh"
#include "stream_common.cuh"

#include <algorithm>

namespace tpls {

constexpr int kRowThreads = kConsumers + 64;
constexpr int kSlots = 3;
#ifndef TPLS_RP_RPI
#define TPLS_RP_RPI 1   // row iterations whose loads are issued together when a thread owns more than 8 elements of a row
#endif

static int pow2_ceil_i(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

static size_t row_stage_bytes(const PassGeom& g) {
    return (size_t)g.tile_rows * (g.n_slabs == 1 ? g.pitch : g.slab_w) * g.elem_size;
}

static size_t row_slot_doubles(const PassGeom& g, bool masked) {
    return g.lpr >= 32 ? (size_t)g.tile_rows * g.lpr * (masked ? 2 : 1) : 0;
}

PassGeom make_row_geom(long long n_rows, int p, int pitch, int elem_size, int sm_count, bool masked) {
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
    if (slab_cg < 32) {
        g.lpr = pow2_ceil_i(slab_cg);
        g.cpt = 1;
    } else {
        g.lpr = std::min(kConsumers, std::max(32, pow2_ceil_i((slab_cg + kMaxCpt - 1) / kMaxCpt)));
        const int need = (slab_cg + g.lpr - 1) / g.lpr;
        g.cpt = need <= 1 ? 1 : (need <= 2 ? 2 : 4);
    }
    g.rpt = kConsumers / g.lpr;
    const long long row_bytes = (long long)(g.n_slabs == 1 ? pitch : g.slab_w) * elem_size;
    // budget: stages * tile + kSlots * slot <= ~108 KB so that two CTAs share an SM
    const double slot_per_tile_byte = g.lpr >= 32 ? (masked ? 2.0 : 1.0) / (2.0 * g.cpt) : 0.0;
    const double budget = tune_env("TPLS_SMEM_KB", 108) * 1024.0;
    long long tile_max = (long long)(budget / (3.0 * (1.0 + slot_per_tile_byte)));
    tile_max = std::min<long long>(tile_max, (long long)tune_env("TPLS_TILE_KB", 32) * 1024);
    long long tr = std::max<long long>(1, tile_max / row_bytes);
    tr = std::min<long long>(tr, std::max<long long>(1, n_rows));
    tr = std::min<long long>(tr, 4096);
    g.tile_rows = (int)tr;
#ifdef TPLS_PROBE
    g.dbg = tune_env("TPLS_DBG", 0);
#endif
    const size_t slots = kSlots * row_slot_doubles(g, masked) * sizeof(double);
    const long long stage = (long long)row_stage_bytes(g);
    g.stages = (int)std::max<long long>(2, std::min<long long>(kMaxStages, ((long long)budget - (long long)slots) / stage));
    const long long n_tiles = (n_rows + tr - 1) / tr;
    const long long want = std::max(1, (sm_count * tune_env("TPLS_CTAS_PER_SM", 2)) / g.n_slabs);
    g.grid_x = (int)std::max<long long>(1, std::min<long long>(n_tiles, want));
#ifdef TPLS_PROBE
    g.dbg = tune_env("TPLS_DBG", 0);
#endif
    return g;
}

size_t rowpass_smem(const PassGeom& g, bool masked) {
    return g.stages * row_stage_bytes(g) + 256 + kSlots * row_slot_doubles(g, masked) * sizeof(double) + 1024;
}

// `old` = previous t[row]; only read by the caller when the epilogue needs it (coupled accumulation, ||dt||^2)
__device__ __forceinline__ bool epilogue_needs_old(const RowPassArgs& a) { return a.epi != 0 || a.d2part != nullptr; }

__device__ __forceinline__ double row_epilogue(const RowPassArgs& a, long long grow, double v, double old, double& d2) {
    double* tp = a.t_out + grow;
    double nv = v;
    if (a.epi == 1) nv = old + v;
    if (a.epi == 2) nv = a.inv_div != 0.0 ? (old + v) * a.inv_div : (old + v) / a.div;
#ifdef TPLS_PROBE
    if (!(a.g.dbg & 1) || nv == 1.2345e301)
#endif
    *tp = nv;
    if (a.d2part != nullptr) {
        const double d = old - nv;
        d2 = fma(d, d, d2);
    }
    return nv;
}

// q = Y't fused into the projection (tpls.py:100): qacc[m] += Y[row, m] * t[row] for the row's FINAL t
__device__ __forceinline__ void q_accumulate(double (&qacc)[kMaxFusedResp], const double (&yv)[kMaxFusedResp], double t) {
#pragma unroll
    for (int m = 0; m < kMaxFusedResp; ++m)
        if (yv[m] != 0.0) qacc[m] = fma(yv[m], t, qacc[m]);  // a held-out row (Y row 0) adds nothing, even a NaN t
}

__device__ __forceinline__ void load_y_row(const RowPassArgs& a, long long grow, double (&yv)[kMaxFusedResp]) {
    const double2* yr = reinterpret_cast<const double2*>(a.y + grow * a.pitch_y);
#pragma unroll
    for (int m = 0; m < kMaxFusedResp; m += 2) {
        double2 t = make_double2(0.0, 0.0);
        if (m < a.pitch_y) t = yr[m >> 1];
        yv[m] = t.x;
        yv[m + 1] = t.y;
    }
}

// MODE 0: dense.  MODE 1: masked, per-row observed counts read from a.rowcnt (they are constant
// during a fit).  MODE 2: masked and counting -- the first masked pass over a tensor; writes a.rowcnt.
// FULL: one slab, every consumer thread owns CPT valid column groups of every row (see colpass_kernel).
template <typename XT, int CPT, int MODE, bool FULL>
__global__ void __launch_bounds__(kRowThreads, 2) rowpass_kernel(const __grid_constant__ RowPassArgs a) {
    pdl_prologue();
    constexpr int VEC = VecOf<XT>::N;
    constexpr bool MASKED = MODE != 0;
    constexpr bool COUNT = MODE == 2;
    const double pads = (double)(a.g.pitch - a.g.p);  // zero-filled pad columns look "observed"
    if (trip_is_dead(a.ctrl, a.trip)) return;

    extern __shared__ __align__(128) unsigned char smem[];
    const PassGeom& g = a.g;
    const int c0 = blockIdx.y * g.slab_w;
    const int slab_cols = min(g.slab_w, g.pitch - c0);
    const int lpr = FULL ? kConsumers : g.lpr;
    const int rpt = FULL ? 1 : g.rpt;
    const int srow = FULL ? kConsumers * VEC * CPT : ((g.n_slabs == 1) ? g.pitch : g.slab_w);
    const size_t stage_elems = (size_t)g.tile_rows * srow;
    XT* tiles = reinterpret_cast<XT*>(smem);
    const size_t tile_area = (size_t)g.stages * stage_elems * sizeof(XT);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + tile_area);
    uint64_t* empty = full + kMaxStages;
    uint64_t* red_full = empty + kMaxStages;
    uint64_t* red_empty = red_full + kSlots;
    double* slots = reinterpret_cast<double*>(smem + tile_area + 256);
    const bool use_slots = FULL ? true : (g.lpr >= 32);
    const size_t slot_doubles = use_slots ? (size_t)g.tile_rows * lpr * (COUNT ? 2 : 1) : 0;
    const bool slabbed = g.n_slabs > 1;
    const double p_total = (double)g.p;

    if (threadIdx.x == 0) {
        for (int s = 0; s < g.stages; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], kConsumers / 32);
        }
        for (int s = 0; s < kSlots; ++s) {
            mbar_init(&red_full[s], kConsumers / 32);
            mbar_init(&red_empty[s], 1);
        }
        fence_mbar_init();
    }
    __syncthreads();

    const TileWalk tw = tile_walk(g);
    const long long n_tiles = (g.n_rows + g.tile_rows - 1) / g.tile_rows;
    const int tid = threadIdx.x;
#ifdef TPLS_PROBE
    const int dbg = g.dbg;  // 1: no store of t   2: reducer skips its fold   4: no slot ring   8: contiguous tile runs   16: no compute
#else
    constexpr int dbg = 0;
#endif
    const int lane = tid & 31;

    // ------------------------------------------------------------------ producer
    if (tid >= kConsumers && tid < kConsumers + 32) {
        if (tid == kConsumers) {
#ifdef TPLS_PROBE
            if (dbg & 32)  // a second, tiny bulk copy per tile (as the column pass has with the rows of Y): does it matter?
                produce_tiles<XT>(g, reinterpret_cast<const XT*>(a.x_in), tiles, full, empty, c0, slab_cols, srow,
                                  reinterpret_cast<const double*>(a.x_in), 4, slots + (size_t)kSlots * slot_doubles);
            else
#endif
            produce_tiles<XT>(g, reinterpret_cast<const XT*>(a.x_in), tiles, full, empty, c0, slab_cols, srow);
        }
        return;
    }

    // ------------------------------------------------------------------ reducer
    if (tid >= kConsumers + 32) {
        if (!use_slots || (dbg & 4)) return;
        // G lanes cooperate on one row; 32/G rows per round
        int G = 32;
        while (G > 1 && (32 / G) * 2 <= g.tile_rows) G >>= 1;  // as many rows per round as the tile has
        if (G > lpr) G = lpr;
        const int rows_per_round = 32 / G;
        const int rg = lane / G, gl = lane - rg * G;
        const bool need_old = epilogue_needs_old(a);
        const bool want_q = a.qpart != nullptr && !slabbed;
        double d2 = 0.0;
        double qacc[kMaxFusedResp], y_pf[kMaxFusedResp];
#pragma unroll
        for (int m = 0; m < kMaxFusedResp; ++m) qacc[m] = y_pf[m] = 0.0;
        RingPos sp_pos;
        for (long long tile = tw.first; tile < tw.end; tile += tw.step, sp_pos.advance(kSlots)) {
            const int sl = sp_pos.idx;
            const uint32_t ph = sp_pos.phase;
            const long long r0 = tile * g.tile_rows;
            int rows = tile_rows_of(g, tile, n_tiles);
            if (dbg & (2 | 16)) rows = 0;
            // what the first round's epilogue reads from global memory is requested BEFORE the wait, so that
            // its latency (microseconds while the HBM is saturated) overlaps the consumers' work on the tile
            double old_pf = 0.0, cnt_pf = 1.0;
            if (gl == 0 && rg < rows && !slabbed) {
                // (t is read before it is written even when the epilogue does not use the old value: measured on
                //  several B200s the first projection of a trip, whose stores missed in L2, took 2.50 ms per 16.4 GB
                //  and 2.23 ms with this load in front of the store; on other boxes it made no difference)
                asm volatile("ld.global.f64 %0, [%1];" : "=d"(old_pf) : "l"(a.t_out + r0 + rg));
                if (MASKED && !COUNT) cnt_pf = a.rowcnt[r0 + rg];
                if (want_q) load_y_row(a, r0 + rg, y_pf);
            }
            mbar_wait(&red_full[sl], ph);
            const double* sp = slots + (size_t)sl * slot_doubles;
            const double* cp = sp + (size_t)g.tile_rows * lpr;
            for (int rb = 0; rb < rows; rb += rows_per_round) {
                const int r = rb + rg;
                double v = 0.0, cnt = 0.0;
                if (r < rows) {
                    const double* rowp = sp + (size_t)r * lpr;
                    const double* rowc = cp + (size_t)r * lpr;
                    const int skew = (G * rg) & (lpr - 1);
                    // lpr / G partials per lane: four independent chains
                    double v1 = 0.0, v2 = 0.0, v3 = 0.0;
                    int i = gl;
                    for (; i + 3 * G < lpr; i += 4 * G) {
                        v += rowp[(i + skew) & (lpr - 1)];
                        v1 += rowp[(i + G + skew) & (lpr - 1)];
                        v2 += rowp[(i + 2 * G + skew) & (lpr - 1)];
                        v3 += rowp[(i + 3 * G + skew) & (lpr - 1)];
                        if (COUNT)
                            cnt += (rowc[(i + skew) & (lpr - 1)] + rowc[(i + G + skew) & (lpr - 1)]) +
                                   (rowc[(i + 2 * G + skew) & (lpr - 1)] + rowc[(i + 3 * G + skew) & (lpr - 1)]);
                    }
                    for (; i < lpr; i += G) {
                        const int col = (i + skew) & (lpr - 1);
                        v += rowp[col];
                        if (COUNT) cnt += rowc[col];
                    }
                    v = (v + v1) + (v2 + v3);
                }
                for (int m = G >> 1; m >= 1; m >>= 1) {
                    v += shfl_xor_d(v, m);
                    if (COUNT) cnt += shfl_xor_d(cnt, m);
                }
                if (r < rows && gl == 0) {
                    const long long grow = r0 + r;
                    if (slabbed) {
                        a.tpart[(size_t)blockIdx.y * g.n_rows + grow] = v;
                        if (COUNT) a.cpart[(size_t)blockIdx.y * g.n_rows + grow] = cnt;
                    } else {
                        if (MASKED) {
                            if (COUNT) {
                                cnt -= pads;
                                if (a.rowcnt != nullptr) a.rowcnt[grow] = cnt;
                            } else {
                                cnt = rb == 0 ? cnt_pf : a.rowcnt[grow];
                            }
                            v = v / cnt * p_total;  // missingvals.py:37: (dot / n_obs) * P, NaN if n_obs == 0
                        }
                        const double old = !need_old ? 0.0 : (rb == 0 ? old_pf : a.t_out[grow]);
                        const double nv = row_epilogue(a, grow, v, old, d2);
                        if (want_q) {
                            if (rb != 0) load_y_row(a, grow, y_pf);
                            q_accumulate(qacc, y_pf, nv);
                        }
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&red_empty[sl]);
        }
        if (a.d2part != nullptr && !slabbed) {
            d2 = warp_sum(d2);
            if (lane == 0) a.d2part[blockIdx.x] = d2;
        }
        if (want_q) {
#pragma unroll
            for (int m = 0; m < kMaxFusedResp; ++m) {
                const double t = warp_sum(qacc[m]);
                if (lane == 0) a.qpart[(size_t)blockIdx.x * kMaxFusedResp + m] = t;
            }
        }
        return;
    }

    // ------------------------------------------------------------------ consumers
    const int cl = tid & (lpr - 1);
    const int rl = tid / lpr;
    double wreg[CPT][VEC];
    bool cvalid[CPT];
    int goff[CPT];  // element offset of the thread's k-th column group in a staged row; a group past the end of the row
                    // reads the row's first group with weights 0 (no branch per group in the row loop)
#pragma unroll
    for (int k = 0; k < CPT; ++k) {
        const int cg = cl + k * lpr;
        cvalid[k] = FULL ? true : (cg * VEC < slab_cols);
        goff[k] = cvalid[k] ? cg * VEC : 0;
#pragma unroll
        for (int j = 0; j < VEC; ++j) wreg[k][j] = cvalid[k] ? a.col_w[c0 + cg * VEC + j] : 0.0;
    }
    double d2 = 0.0;
    // (rows narrower than 32 column groups always have CPT == 1, see make_row_geom: wider layouts never take this path)
    const bool want_q = CPT == 1 && !use_slots && a.qpart != nullptr && !slabbed;
    double qacc[kMaxFusedResp];
#pragma unroll
    for (int m = 0; m < kMaxFusedResp; ++m) qacc[m] = 0.0;

    const bool ring = use_slots && !(dbg & 4);
    RingPos st_pos, sl_pos;
    for (long long tile = tw.first; tile < tw.end; tile += tw.step, st_pos.advance(g.stages), sl_pos.advance(kSlots)) {
        const int s = st_pos.idx;
        const long long r0 = tile * g.tile_rows;
        int rows = tile_rows_of(g, tile, n_tiles);
        if (dbg & 16) rows = 0;
        const int sl = sl_pos.idx;
        double* sp = slots + (size_t)sl * slot_doubles;
        double* cp = sp + (size_t)g.tile_rows * lpr;
        // the slot must have been folded by the reducer before it is written again.  (Waiting for it only right before
        // the first partial of the tile is stored was measured too: 1769 against 1775-1784 ms per fit, within the noise.)
        if (ring && sl_pos.wrapped) mbar_wait(&red_empty[sl], sl_pos.phase ^ 1u);
        mbar_wait(&full[s], st_pos.phase);
        const XT* tp = tiles + s * stage_elems;
        // every lane of a row group walks the same number of rounds so that the shuffles stay converged.
        // The stage goes back to the producer as soon as the LAST rows of the tile sit in registers, before their
        // arithmetic: what a consumer holds a stage for is then loads only, as in the column pass.  RPI row iterations
        // are loaded together (two when a thread owns at most 8 elements of a row; for 16 elements two were measured
        // slower inside the fit: 1814 against 1775 ms).
        constexpr int RPI = (CPT * VEC <= 8) ? 2 : TPLS_RP_RPI;
        bool released = false;
        for (int rb = 0; rb < rows; rb += rpt * RPI) {
            Pack<XT> in[RPI][CPT];
            bool live[RPI];
#pragma unroll
            for (int i = 0; i < RPI; ++i) {
                const int r = rb + i * rpt + rl;
                live[i] = r < rows;
                if (live[i]) {
#pragma unroll
                    for (int k = 0; k < CPT; ++k) {
                        const int cg = cl + k * lpr;
                        in[i][k].v = *reinterpret_cast<const typename VecOf<XT>::type*>(tp + (size_t)r * srow + (FULL ? cg * VEC : goff[k]));
                    }
                }
            }
            if (rb + rpt * RPI >= rows) {
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[s]);
                released = true;
            }
#pragma unroll
            for (int i = 0; i < RPI; ++i) {
                const int r = rb + i * rpt + rl;
                if (RPI > 1 && rb + i * rpt >= rows) break;  // (uniform over the warp)
                double v = 0.0, cnt = 0.0;
                int icnt = 0;
                if (live[i]) {
                    // one accumulator per (column group, element): CPT * VEC independent chains instead of
                    // one chain of CPT * VEC dependent fp64 FMAs
                    double acc[CPT][VEC];
#pragma unroll
                    for (int k = 0; k < CPT; ++k) {
#pragma unroll
                        for (int j = 0; j < VEC; ++j) {
                            const XT xs = in[i][k].e[j];
                            if (MASKED) {
                                const bool ob = (xs == xs);
                                const XT xc = ob ? xs : (XT)0;  // select in the storage type, convert once
                                acc[k][j] = (double)xc * wreg[k][j];
                                // counting: the weights are the column means, and an entry of a column whose mean is
                                // NaN (no observed training entry) is missing after centring, as transform() counts
                                if (COUNT) icnt += (ob && wreg[k][j] == wreg[k][j] && (FULL || cvalid[k])) ? 1 : 0;
                            } else {
                                acc[k][j] = (double)xs * wreg[k][j];
                            }
                        }
                    }
                    // fixed-shape tree
#pragma unroll
                    for (int k = 0; k < CPT; ++k) {
                        double t = acc[k][0];
#pragma unroll
                        for (int j = 1; j < VEC; ++j) t += acc[k][j];
                        v += t;
                    }
                }
                if (COUNT) cnt = (double)icnt;
                if (use_slots) {
                    if (live[i] && (ring || v == 1.2345e301)) {
                        sp[(size_t)r * lpr + cl] = v;
                        if (COUNT) cp[(size_t)r * lpr + cl] = cnt;
                    }
                } else {
                    for (int m = lpr >> 1; m >= 1; m >>= 1) {
                        v += shfl_xor_d(v, m);
                        if (COUNT) cnt += shfl_xor_d(cnt, m);
                    }
                    if (live[i] && cl == 0) {
                        const long long grow = r0 + r;
                        if (slabbed) {
                            a.tpart[(size_t)blockIdx.y * g.n_rows + grow] = v;
                            if (COUNT) a.cpart[(size_t)blockIdx.y * g.n_rows + grow] = cnt;
                        } else {
                            if (MASKED) {
                                if (COUNT) {
                                    cnt -= pads;
                                    if (a.rowcnt != nullptr) a.rowcnt[grow] = cnt;
                                } else {
                                    cnt = a.rowcnt[grow];
                                }
                                v = v / cnt * p_total;  // missingvals.py:37: (dot / n_obs) * P, NaN if n_obs == 0
                            }
                            const double nv = row_epilogue(a, grow, v, epilogue_needs_old(a) ? a.t_out[grow] : 0.0, d2);
                            if (want_q) {
                                double yv[kMaxFusedResp];
                                load_y_row(a, grow, yv);
                                q_accumulate(qacc, yv, nv);
                            }
                        }
                    }
                }
            }
        }
        __syncwarp();
        if (lane == 0) {
            if (!released) mbar_arrive(&empty[s]);
            if (ring) mbar_arrive(&red_full[sl]);
        }
    }

    if (!use_slots && a.d2part != nullptr && !slabbed) {
        double* r2 = reinterpret_cast<double*>(smem);  // tiles are drained
        named_bar_sync(1, kConsumers);
        d2 = warp_sum(d2);
        if (lane == 0) r2[tid >> 5] = d2;
        named_bar_sync(1, kConsumers);
        if (tid == 0) {
            double t = 0.0;
            for (int w = 0; w < kConsumers / 32; ++w) t += r2[w];
            a.d2part[blockIdx.x] = t;
        }
    }
    if (want_q) {
        double* r2 = slots;  // no slot ring on this path: the 1 KB scratch behind the barriers; [warp][kMaxFusedResp]
        named_bar_sync(1, kConsumers);
#pragma unroll
        for (int m = 0; m < kMaxFusedResp; ++m) {
            const double t = warp_sum(qacc[m]);
            if (lane == 0) r2[(tid >> 5) * kMaxFusedResp + m] = t;
        }
        named_bar_sync(1, kConsumers);
        if (tid < kMaxFusedResp) {
            double t = 0.0;
            for (int w = 0; w < kConsumers / 32; ++w) t += r2[w * kMaxFusedResp + tid];
            a.qpart[(size_t)blockIdx.x * kMaxFusedResp + tid] = t;
        }
    }
}

// ---------------------------------------------------------------------------
// dispatch
// ---------------------------------------------------------------------------
template <typename XT, int CPT, int MODE, bool FULL>
static cudaError_t run_rowpass_impl(const RowPassArgs& a, cudaStream_t s) {
    auto kern = rowpass_kernel<XT, CPT, MODE, FULL>;
    const size_t smem = rowpass_smem(a.g, MODE == 2);
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    dim3 grid(a.g.grid_x, a.g.n_slabs);
    int threads = kRowThreads;
#ifdef TPLS_PROBE
    if (a.g.dbg & 4) threads -= 32;  // no slot ring: no reducer warp either
#endif
    launch_k(kern, dim3(grid), dim3(threads), smem, s, a);
    return cudaGetLastError();
}

template <typename XT, int CPT, int MODE>
static cudaError_t run_rowpass(const RowPassArgs& a, cudaStream_t s) {
    const bool full = a.g.n_slabs == 1 && a.g.lpr == kConsumers && a.g.cpt == CPT &&
                      a.g.pitch == kConsumers * (16 / (int)sizeof(XT)) * CPT;
    return full ? run_rowpass_impl<XT, CPT, MODE, true>(a, s) : run_rowpass_impl<XT, CPT, MODE, false>(a, s);
}

template <typename XT>
static cudaError_t rowpass_cpt(int mode, const RowPassArgs& a, cudaStream_t s) {
#define TPLS_RP(C)                                                                                     \
    return mode == 0 ? run_rowpass<XT, C, 0>(a, s) : (mode == 1 ? run_rowpass<XT, C, 1>(a, s) : run_rowpass<XT, C, 2>(a, s))
    switch (a.g.cpt) {
        case 1:
            TPLS_RP(1);
        case 2:
            TPLS_RP(2);
        default:
            TPLS_RP(4);
    }
#undef TPLS_RP
}

cudaError_t launch_rowpass(int dtype, int mode, const RowPassArgs& a, cudaStream_t s) {
    if (mode == 1 && a.rowcnt == nullptr) return cudaErrorInvalidValue;
    return dtype == 0 ? rowpass_cpt<float>(mode, a, s) : rowpass_cpt<double>(mode, a, s);
}

}  // namespace tpls
