// Host side of the C ABI (include/tpls_b200.h): device state of one fit, the
// NIPALS driver that enqueues the passes, and NCCL all-reduces of the small
// replicated quantities (SURVEY.md §8e).  No CPU arithmetic on the data path.
// transform / predict live in transform.cu, the single-operator entry points in ops.cu.
#include "driver_internal.cuh"

namespace tpls_drv {

std::string g_error;
NcclApi g_nccl;

int fail(tpls_handle h, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (h)
        h->error = buf;
    else
        g_error = buf;
    return 1;
}

bool is_device_ptr(const void* p) {
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged;
}


// Per-fit buffers are carved out of ONE cached slab (cudaMalloc / cudaFree cost milliseconds each once
// NCCL has enabled peer access; a fit needs ~60 buffers).  `track == &h->fit_allocs` selects the slab:
// a dry run adds up the sizes, the real run hands out 256-byte aligned pieces.  Any other `track` is a
// list of pool buffers the caller returns with pool_put.
int dev_alloc(tpls_handle h, void** out, size_t bytes, std::vector<void*>* track) {
    *out = nullptr;
    if (track == &h->fit_allocs) {
        const size_t al = (std::max<size_t>(bytes, 16) + 255) & ~(size_t)255;
        if (h->slab_dry) {
            h->slab_need += al;
            *out = reinterpret_cast<void*>(256);
            return 0;
        }
        if (h->slab_off + al > h->slab_cap) return fail(h, "fit slab overflow (internal error)");
        *out = h->slab + h->slab_off;
        h->slab_off += al;
        return 0;
    }
    TRY(pool_get(h, out, bytes));
    if (track) track->push_back(*out);
    return 0;
}

void pool_trim(tpls_handle h) {
    std::vector<tpls_ctx::PoolBuf> keep;
    for (auto& b : h->pool) {
        if (b.used)
            keep.push_back(b);
        else
            cudaFree(b.p);
    }
    h->pool.swap(keep);
}

int pool_get(tpls_handle h, void** out, size_t bytes) {
    bytes = std::max<size_t>(bytes, 256);
    for (auto& b : h->pool)
        if (!b.used && b.bytes >= bytes && b.bytes <= bytes + bytes / 4 + (1u << 20)) {
            b.used = true;
            *out = b.p;
            return 0;
        }
    cudaError_t e = cudaMalloc(out, bytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        pool_trim(h);
        CK(cudaMalloc(out, bytes));
    }
    h->pool.push_back({*out, bytes, true});
    return 0;
}

void pool_put(tpls_handle h, void* p) {
    for (auto& b : h->pool)
        if (b.p == p) b.used = false;
}

void free_fit(tpls_handle h) {
    h->fit_allocs.clear();
    h->slab_off = 0;
    h->fitted = false;
}

void free_tensor(tpls_handle h, Tensor& t) {
    if (t.owned) pool_put(h, t.owned);
    if (t.owned2) pool_put(h, t.owned2);
    t = Tensor();
}


// ---- per-class timing ----
cudaEvent_t prof_event(tpls_handle h) {
    cudaEvent_t e = nullptr;
    if (!h->ev_pool.empty()) {
        e = h->ev_pool.back();
        h->ev_pool.pop_back();
    } else {
        cudaEventCreate(&e);
    }
    return e;
}


// Sums the launch records of every profiled fit since the last collection (event queries cost a few
// microseconds each, so they are made when the profile is asked for, not inside the fit).
void prof_collect(tpls_handle h) {
    h->prof_sum = tpls_profile{};
    // TPLS_PROFILE_TRACE=<file>: one line "class ms bytes" per profiled launch, in launch order (tools/trace_classes.py)
    const char* trace_path = getenv("TPLS_PROFILE_TRACE");
    FILE* trace = (trace_path != nullptr && *trace_path) ? fopen(trace_path, "a") : nullptr;
    for (auto& r : h->prof) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, r.a, r.b);
        if (trace != nullptr) fprintf(trace, "%d %.6f %.0f\n", r.cls, ms, r.bytes);
        // A streaming launch that "moved" its bytes faster than 20 TB/s did not run: the host-enqueued loop works one
        // trip ahead of the stop flag, so the last trip of a component is followed by kernels that return at once
        // (trip_is_dead).  They must not count as launches or bytes of their class -- in round 1 and early round 2
        // they did, which overstated the per-class rates by the share of dead launches (one trip in ~17).
        const bool dead = r.bytes > 0.0 && r.bytes > 20e12 * (double)ms * 1e-3;
        h->prof_sum.ms[r.cls] += ms;
        if (!dead) {
            h->prof_sum.launches[r.cls] += 1;
            h->prof_sum.bytes[r.cls] += r.bytes;
        }
        h->ev_pool.push_back(r.a);
        h->ev_pool.push_back(r.b);
    }
    if (trace != nullptr) fclose(trace);
    h->prof.clear();
}

int allreduce_nccl(tpls_handle h, double* buf, size_t count) {
    if (h->world <= 1 || count == 0) return 0;
    if (h->capturing) return fail(h, "internal error: an NCCL all-reduce inside the captured fit");
    ProfScope ps(h, TPLS_K_NCCL, 0.0);
    CKN(g_nccl.AllReduce(buf, buf, count, kNcclFloat64, kNcclSum, h->comm, h->stream));
    h->stats.collectives++;
    return 0;
}

// fills the communicator part of an exchange and launches it (never skipped: see xchg.cuh)
int xchg_launch(tpls_handle h, XchgArgs& a) {
    ProfScope ps(h, TPLS_K_XCHG, 0.0);
    a.cap = h->xchg_cap;
    a.rank = h->rank;
    a.world = h->world;
    for (int r = 0; r < h->world; ++r) {
        char* base = static_cast<char*>(h->xchg_peer[r]);
        a.flags[r] = reinterpret_cast<unsigned long long*>(base);
        a.data[r] = reinterpret_cast<double*>(base + kXchgHeaderBytes);
    }
    char* mine = static_cast<char*>(h->xchg_buf);
    a.done_ctr = reinterpret_cast<unsigned int*>(mine + 512);
    a.err = reinterpret_cast<int*>(mine + 520);
    a.seq_ctr = reinterpret_cast<unsigned long long*>(mine + 528);
    a.diag = reinterpret_cast<unsigned long long*>(mine + 536);
    CK(launch_xchg(a, h->stream));
    h->stats.kernel_launches++;
    h->stats.collectives++;
    return 0;
}

static bool xchg_fits(tpls_handle h, size_t count) { return h->xchg_ready && count <= (size_t)h->xchg_cap; }

// Sum of a small replicated vector over the ranks: the one-shot peer-memory exchange when it is set up
// (and the vector fits its slots), NCCL otherwise.
int allreduce(tpls_handle h, double* buf, size_t count) {
    if (h->world <= 1 || count == 0) return 0;
    if (!xchg_fits(h, count)) return allreduce_nccl(h, buf, count);
    XchgArgs a{};
    a.in = buf;
    a.out = buf;
    a.count = (int)count;
    return xchg_launch(h, a);
}

static int fold_sum_tail(tpls_handle h, const SetList& sl, size_t base_off, size_t count, const Ctrl* ctrl, bool local_only,
                         XchgArgs* tail) {
    double* base = h->arena + base_off;
    if (h->world > 1 && !local_only && xchg_fits(h, count)) {
        XchgArgs xa{};
        if (tail) xa = *tail;
        xa.n_sets = sl.n;
        for (int i = 0; i < sl.n; ++i) xa.sets[i] = sl.s[i];
        xa.out = base;
        xa.count = (int)count;
        return xchg_launch(h, xa);
    }
    FoldArgs f{};
    f.n_sets = sl.n;
    for (int i = 0; i < sl.n; ++i) f.sets[i] = sl.s[i];
    f.out = base;
    f.ctrl = ctrl;
    {
        ProfScope ps(h, TPLS_K_OTHER, 0.0);
        CK(launch_fold_sets(f, h->stream));
        h->stats.kernel_launches++;
    }
    if (h->world > 1 && !local_only) TRY(allreduce_nccl(h, base, count));
    return 0;
}

int fold_sum(tpls_handle h, const SetList& sl, size_t base_off, size_t count, const Ctrl* ctrl, bool local_only) {
    return fold_sum_tail(h, sl, base_off, count, ctrl, local_only, nullptr);
}

// ---- pass wrappers that keep the launch / byte counters ----
int col_pass(tpls_handle h, int dtype, bool masked, int flags, ColPassArgs& a, int cls) {
    const double bytes = (double)a.g.n_rows * a.g.pitch * a.g.elem_size * ((flags & PF_WRITE) ? 2.0 : 1.0);
    if (cls < 0) {
        cls = TPLS_K_OTHER;
        if (flags == PF_COLSTAT) cls = TPLS_K_COLSTAT;
        if (flags == PF_CONTRACT) cls = TPLS_K_CONTRACT;
        if (flags == (PF_DEFLATE | PF_WRITE | PF_CONTRACT | PF_SUMSQ)) cls = TPLS_K_DEFLATE_CONTRACT;
        if (flags == (PF_DEFLATE | PF_SUMSQ)) cls = TPLS_K_RESIDUAL;
    }
    ProfScope ps(h, cls, bytes);
    CK(launch_colpass(dtype, masked, flags, a, h->stream));
    h->stats.kernel_launches++;
    if (cls != TPLS_K_YSIDE) h->stats.streamed_bytes += bytes;
    return 0;
}

// mode: 0 dense, 1 masked with known row counts (a.rowcnt), 2 masked and counting (fills a.rowcnt)
int row_pass(tpls_handle h, int dtype, int mode, RowPassArgs& a, int cls) {
    const double bytes = (double)a.g.n_rows * a.g.pitch * a.g.elem_size;
    {
        int ex = 0;
        a.inv_div = (a.div > 0.0 && std::frexp(a.div, &ex) == 0.5) ? 1.0 / a.div : 0.0;  // exact only for powers of two
    }
    ProfScope ps(h, cls, bytes);
    CK(launch_rowpass(dtype, mode, a, h->stream));
    h->stats.kernel_launches++;
    if (cls != TPLS_K_YSIDE) h->stats.streamed_bytes += bytes;
    if (a.g.n_slabs > 1) {
        RowFinishArgs f{};
        f.n_rows = a.g.n_rows;
        f.n_slabs = a.g.n_slabs;
        f.tpart = a.tpart;
        f.cpart = mode == 2 ? a.cpart : nullptr;
        f.rowcnt = mode != 0 ? a.rowcnt : nullptr;
        f.pads = (double)(a.g.pitch - a.g.p);
        f.p_total = (double)a.g.p;
        f.t_out = a.t_out;
        f.epi = a.epi;
        f.div = a.div;
        f.d2part = a.d2part;
        f.y = a.y;
        f.pitch_y = a.pitch_y;
        f.qpart = a.qpart;
        f.ctrl = a.ctrl;
        f.trip = a.trip;
        CK(launch_row_finish(f, nullptr, h->stream));
        h->stats.kernel_launches++;
    }
    return 0;
}

int reduce_cols(tpls_handle h, const double* part, double* out, int n_cols, int stride, int n_parts,
                const double* sspart, double* ss_out, int n_ss, const Ctrl* ctrl, int trip) {
    ReduceArgs r{};
    r.part = part;
    r.out = out;
    r.n_cols = n_cols;
    r.stride = stride;
    r.n_parts = n_parts;
    r.sspart = sspart;
    r.ss_out = ss_out;
    r.n_ss = n_ss;
    r.ctrl = ctrl;
    r.trip = trip;
    ProfScope ps(h, TPLS_K_OTHER, 0.0);
    CK(launch_reduce_cols(r, h->stream));
    h->stats.kernel_launches++;
    return 0;
}

int d2_grid(const PassGeom& g) { return g.n_slabs > 1 ? row_finish_grid(g.n_rows) : g.grid_x; }

int copy_out_transposed(tpls_handle h, const double* colmajor, long long rows, int cols, double* out) {
    CK(cudaSetDevice(h->device));
    if (is_device_ptr(out)) {
        CK(launch_transpose_out(colmajor, rows, rows, cols, out, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        return 0;
    }
    const size_t need = sizeof(double) * std::max<long long>(1, rows * cols);
    if (need > h->tmp_cap) {
        if (h->tmp_buf) pool_put(h, h->tmp_buf);
        h->tmp_buf = nullptr;
        h->tmp_cap = 0;
        TRY(pool_get(h, &h->tmp_buf, need));
        h->tmp_cap = need;
    }
    double* tmp = static_cast<double*>(h->tmp_buf);
    CK(launch_transpose_out(colmajor, rows, rows, cols, tmp, h->stream));
    CK(cudaMemcpyAsync(out, tmp, sizeof(double) * rows * cols, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

void drop_graph(tpls_handle h) {
    if (h->graph_exec) cudaGraphExecDestroy(h->graph_exec);
    if (h->graph) cudaGraphDestroy(h->graph);
    h->graph_exec = nullptr;
    h->graph = nullptr;
    h->graph_key = 0;
}

}  // namespace tpls_drv

// ===========================================================================
// C ABI
// ===========================================================================
extern "C" {

int tpls_version(void) { return 100; }

const char* tpls_last_error(tpls_handle h) { return h ? h->error.c_str() : g_error.c_str(); }

int tpls_create(tpls_handle* out, int device, void* cuda_stream) {
    tpls_handle h = nullptr;
    if (!out) return fail(nullptr, "tpls_create: out is NULL");
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(nullptr, "tpls_create: no CUDA device is visible (this library has no CPU path)");
    }
    if (device < 0 || device >= count) return fail(nullptr, "tpls_create: device %d out of range (%d visible)", device, count);
    cudaDeviceProp prop{};
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return fail(nullptr, "cudaGetDeviceProperties failed");
    if (prop.major != 10)
        return fail(nullptr, "tpls_create: device %d is sm_%d%d; this build carries sm_100a code only", device, prop.major,
                    prop.minor);
    h = new tpls_ctx();
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    cudaSetDevice(device);
    if (cuda_stream) {
        h->stream = (cudaStream_t)cuda_stream;
    } else {
        if (cudaStreamCreateWithFlags(&h->private_stream, cudaStreamNonBlocking) != cudaSuccess) {
            delete h;
            return fail(nullptr, "cudaStreamCreate failed");
        }
        h->stream = h->private_stream;
    }
    cudaEventCreate(&h->ev_start);
    cudaEventCreate(&h->ev_stop);
    for (auto& e : h->ev_trip) cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    cudaMallocHost((void**)&h->h_done, sizeof(int) * 4096);
    *out = h;
    return 0;
}

int tpls_destroy(tpls_handle h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    free_fit(h);
    for (auto& t : h->x) free_tensor(h, t);
    if (h->y_src) pool_put(h, h->y_src);
    if (h->y_work) pool_put(h, h->y_work);
    if (h->row_w) pool_put(h, h->row_w);
    if (h->slab) pool_put(h, h->slab);
    if (h->tmp_buf) pool_put(h, h->tmp_buf);
    pool_trim(h);
    drop_graph(h);
    if (h->cap_stream) cudaStreamDestroy(h->cap_stream);
    if (h->body_stream) cudaStreamDestroy(h->body_stream);
    if (h->xchg_buf) {
        for (int r = 0; r < kXchgMaxRanks; ++r)
            if (h->xchg_peer[r] && h->xchg_peer[r] != h->xchg_buf) cudaIpcCloseMemHandle(h->xchg_peer[r]);
        cudaFree(h->xchg_buf);
    }
    if (h->comm) g_nccl.CommDestroy(h->comm);
    if (h->h_done) cudaFreeHost(h->h_done);
    for (int q = 0; q < 2; ++q) {
        if (h->bounce[q]) cudaFreeHost(h->bounce[q]);
        if (h->bounce_ev[q]) cudaEventDestroy(h->bounce_ev[q]);
    }
    cudaEventDestroy(h->ev_start);
    cudaEventDestroy(h->ev_stop);
    for (auto& e : h->ev_trip) cudaEventDestroy(e);
    for (auto& e : h->ev_pool) cudaEventDestroy(e);
    for (auto& r : h->prof) {  // launch records of profiled fits that were never collected
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    if (h->private_stream) cudaStreamDestroy(h->private_stream);
    delete h;
    return 0;
}

int tpls_set_stream(tpls_handle h, void* cuda_stream) {
    if (!h) return fail(nullptr, "NULL handle");
    CK(cudaSetDevice(h->device));
    cudaStream_t next = (cudaStream_t)cuda_stream;
    if (next == nullptr) {
        if (!h->private_stream) CK(cudaStreamCreateWithFlags(&h->private_stream, cudaStreamNonBlocking));
        next = h->private_stream;
    }
    if (next == h->stream) return 0;
    CK(cudaStreamSynchronize(h->stream));
    h->stream = next;
    return 0;
}

int tpls_comm_unique_id(void* id128) {
    const char* why = "";
    if (!g_nccl.load(&why)) return fail(nullptr, "tpls_comm_unique_id: %s", why);
    NcclUniqueId id;
    int r = g_nccl.GetUniqueId(&id);
    if (r != 0) return fail(nullptr, "ncclGetUniqueId -> %s", g_nccl.GetErrorString(r));
    memcpy(id128, &id, sizeof id);
    return 0;
}

int tpls_comm_init(tpls_handle h, const void* id128, int rank, int world) {
    if (!h) return fail(nullptr, "NULL handle");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    drop_graph(h);
    if (h->comm) {  // re-initialisation: release the previous communicator and exchange set-up
        g_nccl.CommDestroy(h->comm);
        h->comm = nullptr;
    }
    h->xchg_ready = false;
    if (world <= 1) {
        h->rank = 0;
        h->world = 1;
        return 0;
    }
    const char* why = "";
    if (!g_nccl.load(&why)) return fail(h, "tpls_comm_init: %s", why);
    NcclUniqueId id;
    memcpy(&id, id128, sizeof id);
    CKN(g_nccl.CommInitRank(&h->comm, world, id, rank));
    h->rank = rank;
    h->world = world;
    return 0;
}

int tpls_comm_xchg_handle(tpls_handle h, void* handle64) {
    if (!h) return fail(nullptr, "NULL handle");
    if (h->world <= 1) return fail(h, "tpls_comm_xchg_handle: no communicator (call tpls_comm_init first)");
    if (h->world > kXchgMaxRanks) return fail(h, "tpls_comm_xchg_handle: at most %d ranks", kXchgMaxRanks);
    CK(cudaSetDevice(h->device));
    if (!h->xchg_buf) {
        h->xchg_cap = 1 << 17;  // doubles per slot (1 MiB): Z of all coupled tensors fits
        const size_t bytes = kXchgHeaderBytes + 2 * sizeof(double) * (size_t)h->xchg_cap;
        CK(cudaMalloc(&h->xchg_buf, bytes));
        CK(cudaMemset(h->xchg_buf, 0, bytes));
        CK(cudaDeviceSynchronize());
    }
    cudaIpcMemHandle_t hnd;
    CK(cudaIpcGetMemHandle(&hnd, h->xchg_buf));
    static_assert(sizeof(hnd) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(handle64, &hnd, sizeof hnd);
    return 0;
}

int tpls_comm_xchg_open(tpls_handle h, const void* handles) {
    if (!h) return fail(nullptr, "NULL handle");
    if (handles == nullptr) {  // switch the exchange off again (every rank must do the same)
        h->xchg_ready = false;
        return 0;
    }
    if (!h->xchg_buf) return fail(h, "tpls_comm_xchg_open: call tpls_comm_xchg_handle first");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    drop_graph(h);  // a captured fit holds the old peer addresses
    for (int r = 0; r < kXchgMaxRanks; ++r) {  // mappings of an earlier set-up
        if (h->xchg_peer[r] && h->xchg_peer[r] != h->xchg_buf) cudaIpcCloseMemHandle(h->xchg_peer[r]);
        h->xchg_peer[r] = nullptr;
    }
    // flags, counters and the sequence number start from zero on every rank (the caller's all-gather of the
    // "opened" verdicts orders this before any peer's first exchange)
    CK(cudaMemset(h->xchg_buf, 0, kXchgHeaderBytes));
    for (int r = 0; r < h->world; ++r) {
        if (r == h->rank) {
            h->xchg_peer[r] = h->xchg_buf;
            continue;
        }
        cudaIpcMemHandle_t hnd;
        memcpy(&hnd, static_cast<const char*>(handles) + 64 * (size_t)r, sizeof hnd);
        CK(cudaIpcOpenMemHandle(&h->xchg_peer[r], hnd, cudaIpcMemLazyEnablePeerAccess));
    }
    h->xchg_ready = true;
    return 0;
}

int tpls_set_x(tpls_handle h, int index, const void* x, int dtype, int ndim, const int64_t* shape, int flags) {
    if (!h) return fail(nullptr, "NULL handle");
    if (index < 0 || index >= TPLS_MAX_TENSORS) return fail(h, "tpls_set_x: index %d out of range", index);
    if (ndim < 2 || ndim > TPLS_MAX_MODES) return fail(h, "tpls_set_x: X must have 2..%d modes, got %d", TPLS_MAX_MODES, ndim);
    if (dtype != TPLS_F32 && dtype != TPLS_F64) return fail(h, "tpls_set_x: dtype must be TPLS_F32 or TPLS_F64");
    CK(cudaSetDevice(h->device));
    Tensor& t = h->x[index];
    free_tensor(h, t);
    t.dtype = dtype;
    t.elem = dtype == TPLS_F32 ? 4 : 8;
    t.ndim = ndim;
    long long p = 1;
    for (int k = 0; k < ndim; ++k) {
        if (shape[k] <= 0) return fail(h, "tpls_set_x: empty mode %d", k);
        if (k && ndim > 3 && shape[k] > 65535)  // the rank-1 kernel keeps per-mode indices of a >= 3-way Z in 16 bits
            return fail(h, "tpls_set_x: mode %d of a %d-way X has %lld entries, at most 65535 are supported", k, ndim, (long long)shape[k]);
        t.shape[k] = shape[k];
        if (k) p *= shape[k];
    }
    if (p > (1ll << 30)) return fail(h, "tpls_set_x: trailing size %lld too large", p);
    t.n = shape[0];
    t.p = (int)p;
    const int vec = 16 / t.elem;
    t.pitch = (int)((p + vec - 1) / vec * vec);
    const size_t bytes = (size_t)t.n * t.pitch * t.elem;
    const bool dev = is_device_ptr(x);
    if (dev && t.pitch == t.p && ((uintptr_t)x % 16 == 0)) {
        t.src = x;
        if (flags & TPLS_X_MAY_OVERWRITE) {
            t.work = const_cast<void*>(x);
        } else {
            TRY(pool_get(h, &t.owned, bytes));
            t.work = t.owned;
        }
    } else {
        TRY(pool_get(h, &t.owned, bytes));
        if (t.pitch != t.p) CK(cudaMemsetAsync(t.owned, 0, bytes, h->stream));
        CK(cudaMemcpy2DAsync(t.owned, (size_t)t.pitch * t.elem, x, (size_t)t.p * t.elem, (size_t)t.p * t.elem, t.n,
                             cudaMemcpyDefault, h->stream));
        if (!dev) h->h2d_bytes += (double)t.n * t.p * t.elem;
        t.src = t.owned;
        t.work = t.owned;
    }
    t.set = true;
    h->fitted = false;
    return 0;
}

int tpls_set_y(tpls_handle h, const double* y, int64_t n, int64_t m) {
    if (!h) return fail(nullptr, "NULL handle");
    if (n <= 0 || m <= 0) return fail(h, "tpls_set_y: empty Y");
    CK(cudaSetDevice(h->device));
    if (h->y_src) pool_put(h, h->y_src);
    if (h->y_work) pool_put(h, h->y_work);
    h->y_src = h->y_work = nullptr;
    h->n = n;
    h->m = (int)m;
    h->pitch_y = (int)((m + 1) / 2 * 2);
    const size_t bytes = (size_t)n * h->pitch_y * sizeof(double);
    TRY(pool_get(h, (void**)&h->y_src, bytes));
    TRY(pool_get(h, (void**)&h->y_work, bytes));
    if (h->pitch_y != m) CK(cudaMemsetAsync(h->y_src, 0, bytes, h->stream));
    CK(cudaMemcpy2DAsync(h->y_src, (size_t)h->pitch_y * 8, y, (size_t)m * 8, (size_t)m * 8, n, cudaMemcpyDefault,
                         h->stream));
    if (!is_device_ptr(y)) h->h2d_bytes += (double)n * m * 8;
    h->fitted = false;
    return 0;
}

// ---------------------------------------------------------------------------
// fit
// ---------------------------------------------------------------------------
static int layout_fit(tpls_handle h, int L, int R);

static int alloc_fit(tpls_handle h, int L, int R) {
    free_fit(h);
    h->slab_dry = true;
    h->slab_need = 0;
    TRY(layout_fit(h, L, R));
    h->slab_dry = false;
    if (h->slab_need > h->slab_cap) {
        if (h->slab) pool_put(h, h->slab);
        h->slab = nullptr;
        h->slab_cap = 0;
        void* p = nullptr;
        TRY(pool_get(h, &p, h->slab_need));
        h->slab = static_cast<char*>(p);
        h->slab_cap = h->slab_need;
    }
    CK(cudaMemsetAsync(h->slab, 0, h->slab_need, h->stream));
    h->slab_off = 0;
    return layout_fit(h, L, R);
}

static int layout_fit(tpls_handle h, int L, int R) {
    auto* tr = &h->fit_allocs;
    const long long n = h->n;
    h->L = L;
    h->R = R;
    h->gy = make_geom(n, h->m, h->pitch_y, 8, h->sm_count);
    h->gy_row = make_row_geom(n, h->m, h->pitch_y, 8, h->sm_count, false);
    // up to kMaxFusedResp responses the Y side of a trip rides on the X passes: the contraction stages the rows of Y
    const int y_row_bytes = h->pitch_y <= kMaxFusedResp ? h->pitch_y * 8 : 0;
    // arena layout
    size_t off = 0;
    for (int l = 0; l < L; ++l) {
        Tensor& t = h->x[l];
        t.g = make_geom(n, t.p, t.pitch, t.elem, h->sm_count, y_row_bytes);
        t.off_colsum = off;
        off += t.pitch;
        t.off_colcnt = off;
        off += t.pitch;
    }
    h->off_ysum = off;
    off += h->pitch_y;
    h->off_ycnt = off;
    off += h->pitch_y;
    h->off_n = off;
    off += 1;
    h->off_nmiss = off;
    off += L;
    h->off_stats_end = off;
    off = (off + 1) / 2 * 2;
    h->off_zcat = off;
    for (int l = 0; l < L; ++l) {
        h->x[l].off_z = off;
        off += h->x[l].pitch;
    }
    h->zcat_len = off - h->off_zcat;
    h->off_q = off;
    off += h->pitch_y;
    h->off_d2 = off;
    off += 2;
    h->off_dots = off;
    off += 64;
    h->off_ss = off;
    for (int l = 0; l < L; ++l) {
        h->x[l].off_ss = off;
        off += R + 1;
    }
    off += R + 1;  // Y
    h->ss_len = off - h->off_ss;
    // covariance mode: C of every tensor followed by Y'Y, one all-reduce per component
    off = (off + 1) / 2 * 2;
    h->off_cov = off;
    if (h->cov_alloc) {
        const int mr_alloc = h->m <= 1 ? 2 : (h->m <= 2 ? 4 : 8);  // room for the masked (row-rescaled) block when m <= 4
        for (int l = 0; l < L; ++l) {
            h->x[l].off_c = off;
            off += (size_t)mr_alloc * h->x[l].pitch;
        }
    }
    h->off_gram_y = off;
    off += 64;
    h->cov_len = off - h->off_cov;
    h->arena_doubles = off;
    TRY(dev_alloc(h, (void**)&h->arena, off * sizeof(double), tr));

    TRY(dev_alloc(h, (void**)&h->T, sizeof(double) * n * R, tr));
    TRY(dev_alloc(h, (void**)&h->U, sizeof(double) * n * R, tr));
    TRY(dev_alloc(h, (void**)&h->Q, sizeof(double) * h->m * R, tr));
    TRY(dev_alloc(h, (void**)&h->coef, sizeof(double) * R * R, tr));
    TRY(dev_alloc(h, (void**)&h->gram, sizeof(double) * R * R, tr));
    TRY(dev_alloc(h, (void**)&h->qvec, sizeof(double) * h->pitch_y, tr));
    TRY(dev_alloc(h, (void**)&h->svec, sizeof(double) * n, tr));
    TRY(dev_alloc(h, (void**)&h->ymean_d, sizeof(double) * h->pitch_y, tr));
    TRY(dev_alloc(h, (void**)&h->zpart_y, sizeof(double) * h->gy.grid_x * h->pitch_y, tr));
    TRY(dev_alloc(h, (void**)&h->cntpart_y, sizeof(double) * h->gy.grid_x * h->pitch_y, tr));
    TRY(dev_alloc(h, (void**)&h->sspart_y, sizeof(double) * std::max(h->gy.grid_x * h->gy.n_slabs, h->sm_count), tr));
    TRY(dev_alloc(h, (void**)&h->d2part, sizeof(double) * 2048, tr));
    TRY(dev_alloc(h, (void**)&h->dotpart, sizeof(double) * 148 * 64, tr));
    TRY(dev_alloc(h, (void**)&h->grampart, sizeof(double) * std::max(148, h->sm_count) * 64, tr));
    TRY(dev_alloc(h, (void**)&h->q_prev, sizeof(double) * 8, tr));
    TRY(dev_alloc(h, (void**)&h->qpart, sizeof(double) * 2048 * kMaxFusedResp, tr));
    TRY(dev_alloc(h, (void**)&h->res_bar, sizeof(unsigned int) * 32 * (h->sm_count + 1), tr));  // (the slab is zeroed when it is laid out)
    h->res_stamps = nullptr;
    if (tune_env("TPLS_RESIDENT_STAMPS", 0)) TRY(dev_alloc(h, (void**)&h->res_stamps, sizeof(long long) * 16, tr));
    TRY(dev_alloc(h, (void**)&h->e0vec, sizeof(double) * kMaxFusedResp, tr));
    TRY(dev_alloc(h, (void**)&h->nloc, sizeof(double) * 2, tr));
    TRY(dev_alloc(h, (void**)&h->conv_dev, sizeof(int) * R, tr));
    TRY(dev_alloc(h, (void**)&h->scratch_ss, sizeof(double) * 8, tr));
    TRY(dev_alloc(h, (void**)&h->trips_dev, sizeof(int) * R, tr));
    TRY(dev_alloc(h, (void**)&h->ymiss_flag, sizeof(int) * 4, tr));
    TRY(dev_alloc(h, (void**)&h->ctrl, sizeof(Ctrl), tr));

    for (int l = 0; l < L; ++l) {
        Tensor& t = h->x[l];
        const size_t gp = (size_t)t.g.grid_x * t.pitch;
        // (the resident trip loop writes one row of partials per CTA, one CTA per SM)
        TRY(dev_alloc(h, (void**)&t.zpart, sizeof(double) * (size_t)std::max(t.g.grid_x, h->sm_count) * t.pitch, tr));
        TRY(dev_alloc(h, (void**)&t.cntpart, sizeof(double) * gp, tr));
        TRY(dev_alloc(h, (void**)&t.sspart, sizeof(double) * t.g.grid_x * t.g.n_slabs, tr));
        TRY(dev_alloc(h, (void**)&t.mean_d, sizeof(double) * t.pitch, tr));
        TRY(dev_alloc(h, &t.mean_native, (size_t)t.elem * t.pitch, tr));
        TRY(dev_alloc(h, (void**)&t.wkron, sizeof(double) * t.pitch * R, tr));
        TRY(dev_alloc(h, (void**)&t.rowcnt, sizeof(double) * n, tr));
        t.rowcnt_ready = false;
        if (h->cov_alloc) {
            const int mr_alloc = h->m <= 1 ? 2 : (h->m <= 2 ? 4 : 8);
            t.gc = make_cov_geom(n, t.p, t.pitch, t.elem, h->sm_count);
            TRY(dev_alloc(h, (void**)&t.covpart, sizeof(double) * (size_t)t.gc.grid_x * mr_alloc * t.pitch, tr));
            TRY(dev_alloc(h, (void**)&t.sspart_cov, sizeof(double) * (size_t)t.gc.grid_x * t.gc.n_slabs, tr));
            TRY(dev_alloc(h, (void**)&t.zscratch, sizeof(double) * t.pitch, tr));
        }
        if (t.g.n_slabs > 1) {
            TRY(dev_alloc(h, (void**)&t.tpart, sizeof(double) * n * t.g.n_slabs, tr));
            TRY(dev_alloc(h, (void**)&t.cpart, sizeof(double) * n * t.g.n_slabs, tr));
        }
        for (int k = 1; k < t.ndim; ++k) {
            TRY(dev_alloc(h, (void**)&t.W[k], sizeof(double) * t.shape[k] * R, tr));
        }
        TRY(dev_alloc(h, (void**)&t.miss_flag, sizeof(int) * 4, tr));
        TRY(dev_alloc(h, (void**)&t.sweeps, sizeof(int) * 4, tr));
        int dims[kMaxZModes];
        for (int k = 1; k < t.ndim; ++k) dims[k - 1] = (int)t.shape[k];
        t.r1_ws = rank1_workspace_doubles(t.ndim - 1, dims, &t.r1_nmax, &t.r1_zs, &t.r1_mt, &t.r1_tab);
        TRY(dev_alloc(h, (void**)&t.r1_scratch, sizeof(double) * t.r1_ws, tr));
    }
    return 0;
}

static void fill_rank1_task(tpls_handle h, Tensor& t, int a, Rank1Task& k, bool use_smem) {
    k.z = h->arena + t.off_z;
    k.colcnt = t.masked ? h->arena + t.off_colcnt : nullptr;
    k.n_total = h->n_total;
    k.p = t.p;
    k.pitch = t.pitch;
    k.nmodes = t.ndim - 1;
    for (int m = 1; m < t.ndim; ++m) {
        k.dims[m - 1] = (int)t.shape[m];
        k.w[m - 1] = t.W[m] + (size_t)a * t.shape[m];
    }
    k.wkron = t.wkron + (size_t)a * t.pitch;
    k.scratch = t.r1_scratch;
    k.use_smem = use_smem ? 1 : 0;
    k.nmax = t.r1_nmax;
    k.zs_len = t.r1_zs;
    k.mt_len = t.r1_mt;
    k.tab_cols = t.r1_tab;
    k.sweeps = t.sweeps;
}


// Regression of u_a on the scores so far and the Y deflation that follows (tpls.py:110-113), shared by the
// streaming and the covariance component loops.  stream_mode: the trip count comes from the control block.
static int component_tail(tpls_handle h, int R, int a, double* ss_y, bool stream_mode) {
    cudaStream_t st = h->stream;
    const long long n = h->n;
    double* A = h->arena;
    double* Ta = h->T + (size_t)a * n;
    double* Ua = h->U + (size_t)a * n;
    // ---- regression on the scores so far (tpls.py:110-112) ----
    {
        DotPairs d{};
        d.n = n;
        d.npairs = 2 * (a + 1);
        d.w = h->row_w;
        for (int b = 0; b <= a; ++b) {
            d.a[b] = h->T + (size_t)b * n;
            d.b[b] = Ta;
            d.a[a + 1 + b] = h->T + (size_t)b * n;
            d.b[a + 1 + b] = Ua;
        }
        int gx = 1;
        {
            ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
            CK(launch_multi_dot(d, h->dotpart, &gx, st));
            h->stats.kernel_launches++;
        }
        {
            SetList sl;
            sl.add(h->dotpart, gx, d.npairs, d.npairs, 0);
            TRY(fold_sum(h, sl, h->off_dots, d.npairs, nullptr));
        }
        {
            ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
            CK(launch_solve_coef(A + h->off_dots, h->gram, h->coef, R, a, h->ctrl, stream_mode ? h->trips_dev : nullptr,
                                 stream_mode ? h->conv_dev : nullptr, st));
            h->stats.kernel_launches++;
        }
    }
    // ---- Y deflation (tpls.py:113) + ||Y||^2 for R2Y ----
    {
        {
            ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
            CK(launch_lincomb(h->T, n, n, h->coef, R, a, h->row_w, h->svec, st));
            h->stats.kernel_launches++;
        }
        ColPassArgs c{};
        c.g = h->gy;
        c.x_in = h->y_work;
        c.x_out = h->y_work;
        c.row_a = h->svec;
        c.col_w = h->qvec;
        c.sspart = h->sspart_y;
        c.row_sw = h->row_w;
        TRY(col_pass(h, TPLS_F64, false, PF_DEFLATE | PF_WRITE | PF_SUMSQ, c, TPLS_K_YSIDE));
        // the residual norm of Y is folded together with the norms of the X pass that follows (see fit_streaming)
        if (!stream_mode) {
            SetList sl;
            sl.add(h->sspart_y, h->gy.grid_x * h->gy.n_slabs, 1, 1, 0);
            TRY(fold_sum(h, sl, (size_t)(ss_y + a + 1 - A), 1, nullptr, true));
        }
    }
    return 0;
}

// ---------------------------------------------------------------------------
// covariance-mode component loop (SURVEY.md §8f n4): per component one cross-covariance pass
// (centring / deflation fused in), the inner iteration on (P x M)-sized data in a single kernel,
// one projection pass; no per-trip pass over X and no per-trip collective.
// ---------------------------------------------------------------------------
static int pow2_at_least(int v) {
    int p = 1;
    while (p < v) p <<= 1;
    return p;
}

static bool cov_supported(tpls_handle h, int L) {
    if (!h->cov_alloc || h->m > 8) return false;
    for (int l = 0; l < L; ++l)
        if (h->x[l].masked && h->m > 4) return false;
    return true;
}

static void r1_config(tpls_handle h, int L, size_t* r1_smem, bool* r1_use_smem) {
    *r1_smem = 0;
    *r1_use_smem = true;
    for (int l = 0; l < L; ++l) *r1_smem = std::max(*r1_smem, h->x[l].r1_ws * sizeof(double));
    if (*r1_smem > 200 * 1024) {
        *r1_use_smem = false;
        *r1_smem = 0;
    }
}

// observed entries per row of a masked tensor after centring (constant during the fit): one counting row pass over
// the input with the column means as weights; an entry of a column whose mean is NaN does not count.  Its
// projection, into the scratch vector, is not used.
static int count_rows(tpls_handle h, Tensor& t) {
    RowPassArgs r{};
    r.g = t.gr_cnt;
    r.x_in = t.src;
    r.col_w = t.mean_d;
    r.t_out = h->svec;
    r.tpart = t.tpart;
    r.cpart = t.cpart;
    r.rowcnt = t.rowcnt;
    r.epi = 0;
    r.div = 1.0;
    TRY(row_pass(h, t.dtype, 2, r));
    t.rowcnt_ready = true;
    return 0;
}

// Y'Y of the current (deflated) Y, summed over the ranks: the stop test then needs no pass over the samples and no
// collective of its own (||u_old - u_new||^2 = dq^T Y'Y dq, u = Y q)
static int gram_y(tpls_handle h) {
    int gx = 1;
    {
        ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
        CK(launch_gram_rows(h->y_work, h->n, h->pitch_y, h->m, h->grampart, &gx, h->stream));
        h->stats.kernel_launches++;
    }
    SetList sl;
    sl.add(h->grampart, gx, h->m * h->m, h->m * h->m, 0);
    return fold_sum(h, sl, h->off_gram_y, (size_t)h->m * h->m, nullptr);
}

static int fit_covariance(tpls_handle h, int L, int R, double tol, int max_iter, int flags, double* ss_y) {
    cudaStream_t st = h->stream;
    const long long n = h->n;
    double* A = h->arena;
    const int M = h->m;

    size_t r1_smem = 0;
    bool r1_use_smem = true;
    r1_config(h, L, &r1_smem, &r1_use_smem);
    for (int l = 0; l < L; ++l) {
        Tensor& t = h->x[l];
        t.cov_mr = t.masked ? pow2_at_least(2 * M) : pow2_at_least(M);
        if (t.masked) TRY(count_rows(h, t));
    }

    for (int a = 0; a < R; ++a) {
        double* Ta = h->T + (size_t)a * n;
        double* Ua = h->U + (size_t)a * n;
        // ---- cross-covariance pass: centring (a == 0) or the deflation by component a-1 fused in ----
        SetList cs, ss;
        for (int l = 0; l < L; ++l) {
            Tensor& t = h->x[l];
            CovPassArgs c{};
            c.g = t.gc;
            c.x_in = a == 0 ? t.src : t.work;
            c.x_out = t.work;
            c.row_a = a == 0 ? nullptr : h->T + (size_t)(a - 1) * n;
            c.col_w = a == 0 ? t.mean_d : t.wkron + (size_t)(a - 1) * t.pitch;
            c.row_sw = h->row_w;
            c.y = h->y_work;
            c.pitch_y = h->pitch_y;
            c.m = M;
            c.rowcnt = t.rowcnt;
            c.cpart = t.covpart;
            c.c_stride = (size_t)t.cov_mr * t.pitch;
            c.sspart = t.sspart_cov;
            {
                const double bytes = 2.0 * (double)n * t.pitch * t.elem;
                ProfScope ps(h, TPLS_K_DEFLATE_CONTRACT, bytes);
                CK(launch_covpass(t.dtype, t.masked, t.cov_mr, c, st));
                h->stats.kernel_launches++;
                h->stats.streamed_bytes += bytes;
            }
            cs.add(t.covpart, t.gc.grid_x, (int)c.c_stride, (int)c.c_stride, t.off_c - h->off_cov);
            ss.add(t.sspart_cov, t.gc.grid_x * t.gc.n_slabs, 1, 1, t.off_ss + a - h->off_ss);
        }
        // ---- Y'Y of the current Y for the stop test; C of every tensor and Y'Y cross the ranks together ----
        int gx = 1;
        {
            ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
            CK(launch_gram_rows(h->y_work, n, h->pitch_y, M, h->grampart, &gx, st));
            h->stats.kernel_launches++;
        }
        cs.add(h->grampart, gx, M * M, M * M, h->off_gram_y - h->off_cov);
        TRY(fold_sum(h, cs, h->off_cov, h->cov_len, nullptr));
        TRY(fold_sum(h, ss, h->off_ss, h->ss_len, nullptr, true));
        // ---- the whole inner iteration of this component, on the device ----
        {
            CovLoopArgs la{};
            la.n_tasks = L;
            la.m = M;
            la.gram_y = A + h->off_gram_y;
            la.tol = tol;
            la.max_iter = max_iter;
            la.normalize_on_break = (flags & TPLS_FIT_NORMALIZE_ON_BREAK) ? 1 : 0;
            la.q_out = h->Q + (size_t)a * M;
            la.qvec = h->qvec;
            la.pitch_y = h->pitch_y;
            la.trips_out = h->trips_dev + a;
            la.conv_out = h->conv_dev + a;
            for (int l = 0; l < L; ++l) {
                Tensor& t = h->x[l];
                fill_rank1_task(h, t, a, la.t[l], r1_use_smem);
                la.t[l].z = t.zscratch;
                la.C[l] = A + t.off_c;
                la.masked[l] = t.masked ? t.cov_mr / 2 : 0;
            }
            ProfScope ps(h, TPLS_K_RANK1, 0.0);
            CK(launch_cov_loop(la, r1_smem, r1_use_smem, st));
            h->stats.kernel_launches++;
        }
        // ---- scores of the converged component: t = X x_2 w2 ..., u = Y q ----
        for (int l = 0; l < L; ++l) {
            Tensor& t = h->x[l];
            RowPassArgs r{};
            r.g = t.gr;
            r.x_in = t.work;
            r.col_w = t.wkron + (size_t)a * t.pitch;
            r.t_out = Ta;
            r.tpart = t.tpart;
            r.cpart = t.cpart;
            r.rowcnt = t.rowcnt;
            r.epi = l == 0 ? 0 : (l == L - 1 ? 2 : 1);
            r.div = (double)L;
            TRY(row_pass(h, t.dtype, t.masked ? 1 : 0, r));
        }
        {
            RowPassArgs r{};
            r.g = h->gy_row;
            r.x_in = h->y_work;
            r.col_w = h->qvec;
            r.t_out = Ua;
            r.epi = 0;
            r.div = 1.0;
            TRY(row_pass(h, TPLS_F64, 0, r, TPLS_K_YSIDE));
        }
        TRY(component_tail(h, R, a, ss_y, false));
    }
    // ---- residual norm after the last component ----
    SetList ss;
    for (int l = 0; l < L; ++l) {
        Tensor& t = h->x[l];
        ColPassArgs c{};
        c.g = t.g;
        c.x_in = t.work;
        c.x_out = t.work;
        c.row_a = h->T + (size_t)(R - 1) * n;
        c.col_w = t.wkron + (size_t)(R - 1) * t.pitch;
        c.sspart = t.sspart;
        c.row_sw = h->row_w;
        TRY(col_pass(h, t.dtype, t.masked, PF_DEFLATE | PF_SUMSQ, c));
        ss.add(t.sspart, t.g.grid_x * t.g.n_slabs, 1, 1, t.off_ss + R - h->off_ss);
    }
    TRY(fold_sum(h, ss, h->off_ss, h->ss_len, nullptr, true));
    return 0;
}

// ---------------------------------------------------------------------------
// streaming component loop (tpls.py:76-120, cmtf.py:88-140)
//
// The inner iteration of a component is a FIXED sequence of launches, the trip body, whose arguments do not
// depend on the trip index (the trip counter and the stop flag live in the control block on the device):
//
//     fold / exchange Z -> rank-1 step -> projection of every tensor (the last one also forms the partials of
//     q = Y't in its epilogue) -> fold / exchange q + normalise + stop test -> contraction of every tensor with
//     u = Y q formed on the fly from the staged rows of Y (skipped once the stop flag is up)
//
// i.e. 3 + 2L launches per trip and no pass over Y.  The body is either captured once per component as the body of
// a CUDA-graph WHILE node (tpls_fit then is ONE graph launch and the host plays no part in the loop), or enqueued
// by the host one trip ahead of the last stop flag it has seen (profiling, NCCL collectives).
// With more than kMaxFusedResp responses the Y side keeps its own passes and the explicit ||u_old - u_new||^2.
// ---------------------------------------------------------------------------
struct StreamPlan {
    int L, R, max_iter, flags;
    double tol;
    bool fused;        // Y side fused into the X passes (pitch_y <= kMaxFusedResp)
    size_t r1_smem;
    bool r1_use_smem;
    double* ss_y;
};

static int contraction(tpls_handle h, const StreamPlan& P, int a, bool in_loop) {
    (void)in_loop;
    const long long n = h->n;
    for (int l = 0; l < P.L; ++l) {
        Tensor& t = h->x[l];
        ColPassArgs c{};
        c.g = t.g;
        c.x_in = t.work;
        c.zpart = t.zpart;
        c.ctrl = h->ctrl;
        if (P.fused) {
            c.y = h->y_work;
            c.q = h->qvec;
            c.pitch_y = h->pitch_y;
        } else {
            c.row_u = h->U + (size_t)a * n;
        }
        TRY(col_pass(h, t.dtype, t.masked, PF_CONTRACT, c));
    }
    return 0;
}

static int trip_body(tpls_handle h, const StreamPlan& P, int a, unsigned long long cond, bool has_cond) {
    cudaStream_t st = h->stream;
    const long long n = h->n;
    const int L = P.L;
    double* A = h->arena;
    double* Ta = h->T + (size_t)a * n;
    double* Ua = h->U + (size_t)a * n;
    LoopEnd le{};
    le.tol = P.tol;
    le.max_iter = P.max_iter;
    le.has_cond = has_cond ? 1 : 0;
    le.cond = cond;
    // ---- Z of every tensor: second reduction stage (+ the sum over the ranks) in one launch ----
    {
        SetList sl;
        for (int l = 0; l < L; ++l) {
            Tensor& t = h->x[l];
            sl.add(t.zpart, t.g.grid_x, t.pitch, t.pitch, t.off_z - h->off_zcat);
        }
        TRY(fold_sum(h, sl, h->off_zcat, h->zcat_len, h->ctrl));
    }
    // ---- K3: rank-1 weight vectors, one CTA per tensor ----
    {
        Rank1Args ra{};
        ra.n_tasks = L;
        ra.tol = P.tol;
        ra.normalize_on_break = (P.flags & TPLS_FIT_NORMALIZE_ON_BREAK) ? 1 : 0;
        ra.ctrl = h->ctrl;
        for (int l = 0; l < L; ++l) fill_rank1_task(h, h->x[l], a, ra.t[l], P.r1_use_smem);
        ProfScope ps(h, TPLS_K_RANK1, 0.0);
        CK(launch_rank1(ra, P.r1_smem, st));
        h->stats.kernel_launches++;
    }
    // ---- K2: t = X x_2 w2 x_3 w3 ..., averaged over the coupled tensors (cmtf.py:120) ----
    int q_parts = 0;
    for (int l = 0; l < L; ++l) {
        Tensor& t = h->x[l];
        RowPassArgs r{};
        r.g = t.gr;
        r.x_in = t.work;
        r.col_w = t.wkron + (size_t)a * t.pitch;
        r.t_out = Ta;
        r.tpart = t.tpart;
        r.cpart = t.cpart;
        r.rowcnt = t.rowcnt;
        r.epi = l == 0 ? 0 : (l == L - 1 ? 2 : 1);
        r.div = (double)L;
        r.ctrl = h->ctrl;
        if (P.fused && l == L - 1) {  // K4 fused: partials of q = Y't over the final (averaged) scores
            r.y = h->y_work;
            r.pitch_y = h->pitch_y;
            r.qpart = h->qpart;
            q_parts = d2_grid(t.gr);
        }
        TRY(row_pass(h, t.dtype, t.masked ? 1 : 0, r));
    }
    if (P.fused) {
        // ---- q = Y't / ||.|| and the stop test dq^T (Y'Y) dq (tpls.py:100-107) on the kernel that finishes the
        //      reduction of q: the exchange kernel across ranks, a single CTA on one GPU ----
        if (h->world > 1 && xchg_fits(h, h->pitch_y)) {
            XchgArgs xa{};
            xa.do_qstop = 1;
            xa.q_m = h->m;
            xa.q_pitch = h->pitch_y;
            xa.qcol = h->Q + (size_t)a * h->m;
            xa.qvec = h->qvec;
            xa.gram = A + h->off_gram_y;
            xa.q_prev = h->q_prev;
            xa.ctrl = h->ctrl;
            xa.loop_end = le;
            SetList sl;
            sl.add(h->qpart, q_parts, kMaxFusedResp, h->pitch_y, 0);
            TRY(fold_sum_tail(h, sl, h->off_q, h->pitch_y, h->ctrl, false, &xa));
        } else {
            const double* part = h->qpart;
            int n_parts = q_parts, stride = kMaxFusedResp;
            if (h->world > 1) {
                SetList sl;
                sl.add(h->qpart, q_parts, kMaxFusedResp, h->pitch_y, 0);
                TRY(fold_sum(h, sl, h->off_q, h->pitch_y, h->ctrl));
                part = A + h->off_q;
                n_parts = 1;
                stride = h->pitch_y;
            }
            ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
            CK(launch_reduce_q_stop(part, n_parts, stride, A + h->off_q, h->m, h->pitch_y, h->Q + (size_t)a * h->m, h->qvec,
                                    A + h->off_gram_y, h->q_prev, h->ctrl, le, st));
            h->stats.kernel_launches++;
        }
    } else {
        // ---- many responses: q = Y't and u = Y q keep their own passes over Y, explicit ||u_old - u_new||^2 ----
        {
            ColPassArgs c{};
            c.g = h->gy;
            c.x_in = h->y_work;
            c.row_u = Ta;
            c.zpart = h->zpart_y;
            c.ctrl = h->ctrl;
            TRY(col_pass(h, TPLS_F64, false, PF_CONTRACT, c, TPLS_K_YSIDE));
            SetList sl;
            sl.add(h->zpart_y, h->gy.grid_x, h->pitch_y, h->pitch_y, 0);
            TRY(fold_sum(h, sl, h->off_q, h->pitch_y, h->ctrl));
            ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
            CK(launch_normalize_q(A + h->off_q, h->m, h->pitch_y, h->Q + (size_t)a * h->m, h->qvec, h->ctrl, 0, st));
            h->stats.kernel_launches++;
        }
        RowPassArgs r{};
        r.g = h->gy_row;
        r.x_in = h->y_work;
        r.col_w = h->qvec;
        r.t_out = Ua;
        r.epi = 0;
        r.div = 1.0;
        r.d2part = h->d2part;
        r.ctrl = h->ctrl;
        TRY(row_pass(h, TPLS_F64, 0, r, TPLS_K_YSIDE));
        const int nd2 = d2_grid(h->gy_row);
        if (h->world > 1 && xchg_fits(h, 1)) {
            XchgArgs xa{};
            xa.do_stop = 1;
            xa.ctrl = h->ctrl;
            xa.loop_end = le;
            SetList sl;
            sl.add(h->d2part, nd2, 1, 1, 0);
            TRY(fold_sum_tail(h, sl, h->off_d2, 1, h->ctrl, false, &xa));
        } else {
            const double* parts = h->d2part;
            int np = nd2;
            if (h->world > 1) {
                SetList sl;
                sl.add(h->d2part, nd2, 1, 1, 0);
                TRY(fold_sum(h, sl, h->off_d2, 1, h->ctrl));
                parts = A + h->off_d2;
                np = 1;
            }
            ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
            CK(launch_stop(h->ctrl, parts, np, le, st));
            h->stats.kernel_launches++;
        }
    }
    // ---- K1: Z = X x_1 u for the next trip (returns at once when the stop flag is up) ----
    const double before = h->stats.streamed_bytes;
    TRY(contraction(h, P, a, true));
    h->body[a].tail_streamed = h->stats.streamed_bytes - before;
    return 0;
}

// Can the inner trips of a component run in the resident loop kernel (rank1.cuh)?  One GPU, the Y side fused, rows
// narrow enough for its thread layout, and a working set of at most TPLS_RESIDENT_MB (default 256: measured on one
// B200, tools/resident_sweep.py -- 20 MB 39 vs 51 us per trip, 82 MB 51 vs 71, 164 MB 97 vs 110, 328 MB 168 vs 173; the
// streaming kernels win beyond that) of which at most ~256 rows per CTA stay outside shared memory.  TPLS_RESIDENT=0 turns
// it off, =1 forces it whatever the size.  Profiled fits
// keep the streaming kernels (their per-class timing is what the profile is for) unless forced.
static int resident_ctas(tpls_handle h, const StreamPlan& P) {
    const int force = tune_env("TPLS_RESIDENT", -1);
    if (force == 0 || h->world > 1 || !P.fused || P.L > h->sm_count) return 0;
    if (h->profile && force != 1) return 0;
    double bytes = (double)h->n * h->pitch_y * 8.0;
    for (int l = 0; l < P.L; ++l) {
        const Tensor& t = h->x[l];
        if (t.pitch / (16 / t.elem) > kRank1Threads * kResidentKc) return 0;
        bytes += (double)h->n * t.pitch * t.elem;
    }
    if (force != 1 && bytes > 1048576.0 * tune_env("TPLS_RESIDENT_MB", 256)) return 0;
    if (P.r1_use_smem && P.r1_smem > 200 * 1024) return 0;
    const long long want = (h->n + 15) / 16;  // at least 16 samples per CTA
    const int n_ctas = (int)std::max<long long>(P.L, std::min<long long>(h->sm_count, want));
    if (force != 1) {
        // Rows of a CTA's block that do not fit in shared memory are fetched from L2 / HBM by a warp per row, a few rows
        // at a time: fine for a few hundred of them, slow for thousands of narrow rows (the streaming kernels move those
        // at the HBM rate).  An estimate of the launcher's split is enough here.
        const long long per = (h->n + n_ctas - 1) / n_ctas;
        double row_bytes = (double)h->pitch_y * 8.0;
        for (int l = 0; l < P.L; ++l) row_bytes += (double)h->x[l].pitch * h->x[l].elem;
        const double room = 190.0 * 1024.0 - (P.r1_use_smem ? std::max(0.0, (double)P.r1_smem - 20.0 * 1024.0) : 0.0);
        const long long cached = std::min<long long>(per, (long long)(std::max(0.0, room) / row_bytes));
        if (per - cached > tune_env("TPLS_RESIDENT_UNCACHED_ROWS", 256)) return 0;
    }
    return n_ctas;
}

static bool resident_tail_on() { return tune_env("TPLS_RESIDENT_TAIL", 1) != 0; }

static int run_resident(tpls_handle h, const StreamPlan& P, int a, int n_ctas) {
    ResidentArgs ra{};
    ra.n_tensors = P.L;
    ra.n_rows = h->n;
    ra.y = h->y_work;
    ra.pitch_y = h->pitch_y;
    ra.m = h->m;
    ra.t_out = h->T + (size_t)a * h->n;
    ra.qpart = h->qpart;
    ra.qcol = h->Q + (size_t)a * h->m;
    ra.qvec = h->qvec;
    ra.q_prev = h->q_prev;
    ra.gram = h->arena + h->off_gram_y;
    ra.grampart = h->grampart;
    ra.u_out = h->U + (size_t)a * h->n;
    // the regression / Y-deflation tail of the component in the same launch (TPLS_RESIDENT_TAIL=0: the host launches it)
    ra.tail = resident_tail_on() ? 1 : 0;
    ra.comp = a;
    ra.n_comp = P.R;
    ra.T = h->T;
    ra.row_w = h->row_w;
    ra.y_rw = h->y_work;
    ra.dotpart = h->dotpart;
    ra.gram_t = h->gram;
    ra.coef = h->coef;
    ra.trips_out = h->trips_dev;
    ra.conv_out = h->conv_dev;
    ra.sspart_y = h->sspart_y;
    ra.ctrl = h->ctrl;
    ra.tol = P.tol;
    ra.max_iter = P.max_iter;
    ra.normalize_on_break = (P.flags & TPLS_FIT_NORMALIZE_ON_BREAK) ? 1 : 0;
    ra.r1_in_smem = P.r1_use_smem ? 1 : 0;
    ra.bar = h->res_bar;
    ra.stamps = h->res_stamps;
    double bytes = 0.0;
    for (int l = 0; l < P.L; ++l) {
        Tensor& t = h->x[l];
        ResidentTensor& X = ra.x[l];
        X.x = t.work;
        X.dtype = t.dtype;
        X.p = t.p;
        X.pitch = t.pitch;
        X.masked = t.masked ? 1 : 0;
        X.rowcnt = t.rowcnt;
        X.zpart = t.zpart;
        X.parts0 = t.g.grid_x;
        X.z = h->arena + t.off_z;
        X.wkron = t.wkron + (size_t)a * t.pitch;
        fill_rank1_task(h, t, a, ra.r1[l], P.r1_use_smem);
        bytes += (double)h->n * t.pitch * t.elem;
    }
    tpls_ctx::BodyCount& bc = h->body[a];
    bc = tpls_ctx::BodyCount{};
    {
        ProfScope ps(h, TPLS_K_OTHER, 0.0);
        CK(launch_resident_loop(ra, n_ctas, P.r1_use_smem ? P.r1_smem : 0, h->stream));
    }
    h->stats.kernel_launches++;
    h->stats.resident_loops++;
    // per trip: one projection and one contraction over every tensor; the last trip has no contraction
    h->stats.streamed_bytes += 2.0 * bytes;
    bc.streamed = 2.0 * bytes;
    bc.tail_streamed = bytes;
    bc.enqueued = 1;
    bc.resident = true;
    return 0;
}

// runs the trip body until the stop flag is up: a WHILE node while capturing, host-driven otherwise
static int run_loop(tpls_handle h, const StreamPlan& P, int a) {
    if (const int n_ctas = resident_ctas(h, P)) return run_resident(h, P, a, n_ctas);
    tpls_ctx::BodyCount& bc = h->body[a];
    bc = tpls_ctx::BodyCount{};
    const tpls_stats before = h->stats;
    auto account = [&]() {
        bc.launches = h->stats.kernel_launches - before.kernel_launches;
        bc.collectives = h->stats.collectives - before.collectives;
        bc.streamed = h->stats.streamed_bytes - before.streamed_bytes;
    };
    if (h->capturing) {
        cudaStreamCaptureStatus status;
        cudaGraph_t g = nullptr;
        const cudaGraphNode_t* deps = nullptr;
        size_t n_deps = 0;
        const cudaGraphEdgeData* edges = nullptr;  // programmatic (PDL) edges carry data a plain query would lose
        CK(cudaStreamGetCaptureInfo_v3(h->stream, &status, nullptr, &g, &deps, &edges, &n_deps));
        if (status != cudaStreamCaptureStatusActive) return fail(h, "internal error: capture is not active");
        cudaGraphConditionalHandle cond;
        CK(cudaGraphConditionalHandleCreate(&cond, g, 1, cudaGraphCondAssignDefault));
        cudaGraphNodeParams np{};
        np.type = cudaGraphNodeTypeConditional;
        np.conditional.handle = cond;
        np.conditional.type = cudaGraphCondTypeWhile;
        np.conditional.size = 1;
        cudaGraphNode_t node;
        // full dependencies on whatever precedes the loop (the edge kind is a property of the downstream launch)
        CK(cudaGraphAddNode(&node, g, deps, n_deps, &np));
        cudaGraph_t body = np.conditional.phGraph_out[0];
        cudaStream_t outer = h->stream;
        CK(cudaStreamBeginCaptureToGraph(h->body_stream, body, nullptr, nullptr, 0, cudaStreamCaptureModeRelaxed));
        h->stream = h->body_stream;
        int rc = trip_body(h, P, a, (unsigned long long)cond, true);
        h->stream = outer;
        cudaGraph_t ended = nullptr;
        cudaError_t e = cudaStreamEndCapture(h->body_stream, &ended);
        if (rc) return rc;
        if (e != cudaSuccess) return fail(h, "capturing the trip body -> %s", cudaGetErrorString(e));
        CK(cudaStreamUpdateCaptureDependencies(outer, &node, 1, cudaStreamSetCaptureDependencies));
        pdl_hold_next();
        account();
        bc.enqueued = 1;
        return 0;
    }
    const int LOOK = 1;
    for (int trip = 0; trip < P.max_iter; ++trip) {
        char nm[48];
        snprintf(nm, sizeof nm, "component %d trip %d (enqueue)", a, trip);
        NvtxRange nvtx_trip(nm);
        if (trip >= 1 + LOOK) {
            const int back = trip - 1 - LOOK;
            CK(cudaEventSynchronize(h->ev_trip[back & 3]));
            if (h->h_done[back] != 0) break;
        }
        TRY(trip_body(h, P, a, 0ull, false));
        if (trip == 0) account();
        bc.enqueued++;
        CK(cudaMemcpyAsync(&h->h_done[trip], &h->ctrl->stop, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaEventRecord(h->ev_trip[trip & 3], h->stream));
    }
    // the loop body was counted once; the stats of the whole fit are rebuilt from the trip counts at the end
    h->stats.kernel_launches = before.kernel_launches + bc.launches;
    h->stats.collectives = before.collectives + bc.collectives;
    h->stats.streamed_bytes = before.streamed_bytes + bc.streamed;
    return 0;
}

static int fit_streaming(tpls_handle h, const StreamPlan& P) {
    cudaStream_t st = h->stream;
    const long long n = h->n;
    const int L = P.L, R = P.R;
    double* A = h->arena;
    for (int l = 0; l < L; ++l)
        if (h->x[l].masked) TRY(count_rows(h, h->x[l]));
    if (!P.fused) {
        ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
        CK(launch_gather_col(h->y_work, n, h->pitch_y, 0, h->U, st));  // u0 = first column of Y (tpls.py:78)
        h->stats.kernel_launches++;
    }
    for (int a = 0; a <= R; ++a) {
        // ---- centring (a == 0) or the deflation by component a-1 (tpls.py:109), fused with the first contraction
        //      of component a (u0 = Y e0) and with the residual norm; after the last component: the norm alone ----
        SetList ss;
        for (int l = 0; l < L; ++l) {
            Tensor& t = h->x[l];
            ColPassArgs c{};
            c.g = t.g;
            c.x_in = a == 0 ? t.src : t.work;
            c.x_out = t.work;
            c.row_a = a == 0 ? nullptr : h->T + (size_t)(a - 1) * n;
            c.col_w = a == 0 ? t.mean_d : t.wkron + (size_t)(a - 1) * t.pitch;
            c.sspart = t.sspart;
            c.row_sw = h->row_w;
            if (a < R) {
                c.zpart = t.zpart;
                if (P.fused) {
                    c.y = h->y_work;
                    c.q = h->e0vec;
                    c.pitch_y = h->pitch_y;
                } else {
                    c.row_u = h->U + (size_t)a * n;
                }
                TRY(col_pass(h, t.dtype, t.masked, PF_DEFLATE | PF_WRITE | PF_CONTRACT | PF_SUMSQ, c));
            } else {
                TRY(col_pass(h, t.dtype, t.masked, PF_DEFLATE | PF_SUMSQ, c));
            }
            ss.add(t.sspart, t.g.grid_x * t.g.n_slabs, 1, 1, t.off_ss + a - h->off_ss);
        }
        if (a > 0) ss.add(h->sspart_y, h->sspart_y_n, 1, 1, (size_t)(P.ss_y + a - A) - h->off_ss);
        TRY(fold_sum(h, ss, h->off_ss, h->ss_len, nullptr, true));
        if (a == R) break;

        char nm[32];
        snprintf(nm, sizeof nm, "component %d", a);
        NvtxRange nvtx_comp(nm);
        double* Ua = h->U + (size_t)a * n;
        // the resident loop forms Y'Y and u = Y q itself and leaves the control block as the streaming loop would
        const bool resident = resident_ctas(h, P) > 0;
        if (!resident) {
            ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
            CK(launch_reset_ctrl(h->ctrl, st));
            h->stats.kernel_launches++;
        }
        if (P.fused && !resident) TRY(gram_y(h));
        TRY(run_loop(h, P, a));
        if (P.fused && !resident) {
            // u = Y q of the last trip (tpls.py:102): inside the loop it only ever exists row by row
            RowPassArgs r{};
            r.g = h->gy_row;
            r.x_in = h->y_work;
            r.col_w = h->qvec;
            r.t_out = Ua;
            r.epi = 0;
            r.div = 1.0;
            TRY(row_pass(h, TPLS_F64, 0, r, TPLS_K_YSIDE));
        }
        if (resident && resident_tail_on()) {
            h->sspart_y_n = resident_ctas(h, P);  // the resident loop ran the tail: one partial of ||Y||^2 per CTA
        } else {
            TRY(component_tail(h, R, a, P.ss_y, true));
            h->sspart_y_n = h->gy.grid_x * h->gy.n_slabs;
        }
        if (!P.fused && a + 1 < R) {
            ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
            CK(launch_gather_col(h->y_work, n, h->pitch_y, 0, h->U + (size_t)(a + 1) * n, st));
            h->stats.kernel_launches++;
        }
    }
    return 0;
}

static unsigned long long fnv(unsigned long long hsh, const void* p, size_t n) {
    const unsigned char* b = static_cast<const unsigned char*>(p);
    for (size_t i = 0; i < n; ++i) hsh = (hsh ^ b[i]) * 1099511628211ull;
    return hsh;
}

// everything the captured launches depend on: buffers, shapes, options, what the statistics pass decided
static unsigned long long graph_key_of(tpls_handle h, int L, int R, double tol, int max_iter, int flags, bool cov_mode) {
    unsigned long long k = 1469598103934665603ull;
#define KEY(v) k = fnv(k, &(v), sizeof(v))
    KEY(L); KEY(R); KEY(tol); KEY(max_iter); KEY(flags); KEY(cov_mode);
    KEY(h->n); KEY(h->m); KEY(h->n_total); KEY(h->world); KEY(h->rank); KEY(h->xchg_ready); KEY(h->xchg_buf);
    KEY(h->y_src); KEY(h->y_work); KEY(h->row_w); KEY(h->slab); KEY(h->slab_need);
    const bool pdl = pdl_enabled();
    KEY(pdl);
    const int res_switch = tune_env("TPLS_RESIDENT", -1), res_mb = tune_env("TPLS_RESIDENT_MB", 256);  // resident_ctas()
    const int res_tail = tune_env("TPLS_RESIDENT_TAIL", 1), res_unc = tune_env("TPLS_RESIDENT_UNCACHED_ROWS", 256);
    KEY(res_switch); KEY(res_mb); KEY(res_tail); KEY(res_unc);
    for (int l = 0; l < L; ++l) {
        Tensor& t = h->x[l];
        KEY(t.src); KEY(t.work); KEY(t.dtype); KEY(t.ndim); KEY(t.masked);
        for (int d = 0; d < t.ndim; ++d) KEY(t.shape[d]);
    }
#undef KEY
    return k ? k : 1;
}

int tpls_fit(tpls_handle h, int n_tensors, int n_components, double tol, int max_iter, int flags) {
    if (!h) return fail(nullptr, "NULL handle");
    const int L = n_tensors, R = n_components;
    if (L < 1 || L > TPLS_MAX_TENSORS) return fail(h, "tpls_fit: n_tensors must be 1..%d", TPLS_MAX_TENSORS);
    if (R < 1 || R > 32) return fail(h, "tpls_fit: n_components must be 1..32");
    if (max_iter < 1 || max_iter > 4096) return fail(h, "tpls_fit: max_iter must be 1..4096");
    if (!h->y_src) return fail(h, "tpls_fit: Y not set");
    for (int l = 0; l < L; ++l) {
        if (!h->x[l].set) return fail(h, "tpls_fit: X[%d] not set", l);
        if (h->x[l].n != h->n)
            return fail(h, "tpls_fit: X[%d] has %lld samples, Y has %lld", l, h->x[l].n, h->n);
    }
    CK(cudaSetDevice(h->device));
    NvtxRange nvtx_fit("tpls_fit");
    cudaStream_t st = h->stream;
    const double h2d = h->h2d_bytes;
    h->stats = tpls_stats{};
    h->stats.h2d_bytes = h2d;
    h->h2d_bytes = 0;
    h->profile = (flags & TPLS_FIT_PROFILE) != 0;
    h->cov_alloc = (flags & TPLS_FIT_COVARIANCE) != 0 && h->m <= 8;
    TRY(alloc_fit(h, L, R));
    if (h->xchg_ready) {  // a time-out of an earlier fit must not fail this one; the wait diagnostics start from zero
        CK(cudaMemsetAsync(static_cast<char*>(h->xchg_buf) + 520, 0, sizeof(int), st));
        CK(cudaMemsetAsync(static_cast<char*>(h->xchg_buf) + 536, 0, 3 * sizeof(unsigned long long), st));
    }
    CK(cudaEventRecord(h->ev_start, st));
    const long long n = h->n;
    double* A = h->arena;

    // ---- column statistics (np.nanmean, tpls.py:66-67): sums, weighted counts, the sample count and an
    //      UNWEIGHTED census of the NaNs, folded and summed over the ranks in one launch ----
    nvtxRangePushA("tpls_fit: column statistics");
    {
        SetList sl;
        for (int l = 0; l < L; ++l) {
            Tensor& t = h->x[l];
            ColPassArgs c{};
            c.g = t.g;
            c.x_in = t.src;
            c.zpart = t.zpart;
            c.cntpart = t.cntpart;
            c.sspart = t.sspart;
            c.row_sw = h->row_w;
            TRY(col_pass(h, t.dtype, true, PF_COLSTAT, c));
            sl.add(t.zpart, t.g.grid_x, t.pitch, t.pitch, t.off_colsum);
            sl.add(t.cntpart, t.g.grid_x, t.pitch, t.pitch, t.off_colcnt);
        }
        ColPassArgs c{};
        c.g = h->gy;
        c.x_in = h->y_src;
        c.zpart = h->zpart_y;
        c.cntpart = h->cntpart_y;
        c.row_sw = h->row_w;
        TRY(col_pass(h, TPLS_F64, true, PF_COLSTAT, c, TPLS_K_YSIDE));
        sl.add(h->zpart_y, h->gy.grid_x, h->pitch_y, h->pitch_y, h->off_ysum);
        sl.add(h->cntpart_y, h->gy.grid_x, h->pitch_y, h->pitch_y, h->off_ycnt);
        if (h->row_w == nullptr) {
            ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
            CK(launch_fill(h->nloc, 1, (double)n, st));
            h->stats.kernel_launches++;
            sl.add(h->nloc, 1, 1, 1, h->off_n);
        } else {
            // sample count of the fold = sum of the 0/1 weights
            DotPairs d{};
            d.n = n;
            d.npairs = 1;
            d.a[0] = h->row_w;
            d.b[0] = h->row_w;
            int gx = 1;
            CK(launch_multi_dot(d, h->dotpart, &gx, st));
            h->stats.kernel_launches++;
            sl.add(h->dotpart, gx, 1, 1, h->off_n);
        }
        for (int l = 0; l < L; ++l) {
            Tensor& t = h->x[l];
            sl.add(t.sspart, t.g.grid_x * t.g.n_slabs, 1, 1, h->off_nmiss + l);
        }
        TRY(fold_sum(h, sl, 0, h->off_stats_end, nullptr));
    }
    for (int l = 0; l < L; ++l) {
        Tensor& t = h->x[l];
        ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
        CK(launch_finalize_mean(t.dtype, A + t.off_colsum, A + t.off_colcnt, A + h->off_n, t.p, t.pitch, t.mean_d,
                                t.mean_native, t.miss_flag, A + h->off_nmiss + l, st));
        h->stats.kernel_launches++;
    }
    {
        ProfScope ps_small(h, TPLS_K_OTHER, 0.0);
        CK(launch_finalize_mean(TPLS_F64, A + h->off_ysum, A + h->off_ycnt, A + h->off_n, h->m, h->pitch_y, h->ymean_d,
                                nullptr, h->ymiss_flag, nullptr, st));
        h->stats.kernel_launches++;
        CK(launch_fill(h->e0vec, 1, 1.0, st));  // e0 = (1, 0, ...): u0 = Y e0 (tpls.py:78); the slab is zeroed
        h->stats.kernel_launches++;
    }
    {
        int flagsh[TPLS_MAX_TENSORS] = {0};
        for (int l = 0; l < L; ++l)
            CK(cudaMemcpyAsync(&flagsh[l], h->x[l].miss_flag, sizeof(int), cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&h->n_total, A + h->off_n, sizeof(double), cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        for (int l = 0; l < L; ++l) {
            Tensor& t = h->x[l];
            t.masked = flagsh[l] != 0;
            t.gr = make_row_geom(n, t.p, t.pitch, t.elem, h->sm_count, false);
            t.gr_cnt = make_row_geom(n, t.p, t.pitch, t.elem, h->sm_count, true);
        }
    }
    nvtxRangePop();

    const bool cov_mode = (flags & TPLS_FIT_COVARIANCE) != 0 && cov_supported(h, L);
    h->stats.covariance_mode = cov_mode ? 1 : 0;
    StreamPlan P{};
    P.L = L;
    P.R = R;
    P.tol = tol;
    P.max_iter = max_iter;
    P.flags = flags;
    P.fused = h->pitch_y <= kMaxFusedResp;
    P.ss_y = A + h->off_ss + (size_t)L * (R + 1);
    r1_config(h, L, &P.r1_smem, &P.r1_use_smem);

    // Everything from here to the residual norms is ONE sequence of launches with no host decision in it: captured
    // into a CUDA graph (and kept for the next fit with the same key) unless the fit is profiled, some collective
    // has to go through NCCL, or TPLS_NO_GRAPH is set.
    bool use_graph = !h->profile && !h->graph_broken && getenv("TPLS_NO_GRAPH") == nullptr;
    if (h->world > 1) {
        const size_t biggest = std::max(h->zcat_len, cov_mode ? h->cov_len : (size_t)0);
        if (!xchg_fits(h, biggest)) use_graph = false;
    }
    h->fit_mode = use_graph ? 1 : 0;
    for (auto& b : h->body) b = tpls_ctx::BodyCount{};
    const tpls_stats pre = h->stats;

    auto enqueue_main = [&]() -> int {
        cudaStream_t s2 = h->stream;
        // ---- centre Y (tpls.py:71) ----
        ColPassArgs c{};
        c.g = h->gy;
        c.x_in = h->y_src;
        c.x_out = h->y_work;
        c.col_w = h->ymean_d;
        c.sspart = h->sspart_y;
        c.row_sw = h->row_w;
        TRY(col_pass(h, TPLS_F64, false, PF_DEFLATE | PF_WRITE | PF_SUMSQ, c, TPLS_K_YSIDE));
        {
            SetList sl;
            sl.add(h->sspart_y, h->gy.grid_x * h->gy.n_slabs, 1, 1, (size_t)(P.ss_y - A) - h->off_ss);
            TRY(fold_sum(h, sl, h->off_ss, h->ss_len, nullptr, true));
        }
        if (h->row_w != nullptr) {
            // held-out rows of the centred Y are zeroed: they then drop out of u, Z, q and the stop test
            CK(launch_scale_rows(h->y_work, n, h->pitch_y, h->row_w, s2));
            h->stats.kernel_launches++;
        }
        return cov_mode ? fit_covariance(h, L, R, tol, max_iter, flags, P.ss_y) : fit_streaming(h, P);
    };

    if (use_graph) {
        const unsigned long long key = graph_key_of(h, L, R, tol, max_iter, flags, cov_mode);
        if (h->graph_exec == nullptr || key != h->graph_key) {
            drop_graph(h);
            if (!h->cap_stream) CK(cudaStreamCreateWithFlags(&h->cap_stream, cudaStreamNonBlocking));
            if (!h->body_stream) CK(cudaStreamCreateWithFlags(&h->body_stream, cudaStreamNonBlocking));
            NvtxRange nvtx_cap("tpls_fit: capture + instantiate");
            CK(cudaStreamBeginCapture(h->cap_stream, cudaStreamCaptureModeRelaxed));
            h->stream = h->cap_stream;
            h->capturing = true;
            int rc = enqueue_main();
            h->capturing = false;
            h->stream = st;
            cudaGraph_t g = nullptr;
            cudaError_t e = cudaStreamEndCapture(h->cap_stream, &g);
            if (rc == 0 && e != cudaSuccess) rc = fail(h, "tpls_fit: capturing the fit -> %s", cudaGetErrorString(e));
            if (rc == 0) {
                h->graph = g;
                g = nullptr;
                e = cudaGraphInstantiate(&h->graph_exec, h->graph, 0);
                if (e != cudaSuccess) rc = fail(h, "tpls_fit: cudaGraphInstantiate -> %s", cudaGetErrorString(e));
            }
            if (rc != 0) {
                if (g) cudaGraphDestroy(g);
                drop_graph(h);
                cudaGetLastError();
                // Nothing has run yet.  A single-GPU fit falls back to host-enqueued trips (and stays there); on
                // several GPUs every rank must drive its loop the same way (a host-driven rank enqueues a fixed number
                // of bodies past the stop, a graph does not), so there the failure is reported.
                if (h->world > 1) return rc;
                h->graph_broken = true;
                h->stats = pre;
                for (auto& b : h->body) b = tpls_ctx::BodyCount{};
                h->fit_mode = 0;
                use_graph = false;
                TRY(enqueue_main());
                goto loops_done;
            }
            h->graph_key = key;
            // static launches of the captured fit (the loop bodies were captured once each)
            h->g_static = h->stats;
            h->g_static.kernel_launches -= pre.kernel_launches;
            h->g_static.collectives -= pre.collectives;
            h->g_static.streamed_bytes -= pre.streamed_bytes;
            for (int a = 0; a < R; ++a) h->g_body[a] = h->body[a];
        } else {
            for (int a = 0; a < R; ++a) h->body[a] = h->g_body[a];
            h->stats.kernel_launches = pre.kernel_launches + h->g_static.kernel_launches;
            h->stats.collectives = pre.collectives + h->g_static.collectives;
            h->stats.streamed_bytes = pre.streamed_bytes + h->g_static.streamed_bytes;
            h->stats.resident_loops = h->g_static.resident_loops;
        }
        CK(cudaGraphLaunch(h->graph_exec, st));
        h->stats.graph_launches = 1;
    } else {
        TRY(enqueue_main());
    }
loops_done:

    // ---- R2X / R2Y from the residual norms (SURVEY.md §0.4) ----
    // through NCCL on purpose: it cannot complete before every peer has finished all earlier exchanges,
    // so no rank can leave the fit (and possibly free its exchange buffer) while a peer still reads it
    TRY(allreduce_nccl(h, A + h->off_ss, h->ss_len));
    std::vector<double> ss(h->ss_len);
    h->trips.assign(R, 0);
    h->converged.assign(R, 0);
    CK(cudaMemcpyAsync(ss.data(), A + h->off_ss, sizeof(double) * h->ss_len, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h->trips.data(), h->trips_dev, sizeof(int) * R, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h->converged.data(), h->conv_dev, sizeof(int) * R, cudaMemcpyDeviceToHost, st));
    CK(cudaEventRecord(h->ev_stop, st));
    CK(cudaStreamSynchronize(st));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->ev_start, h->ev_stop));
    h->stats.fit_ms = ms;
    if (h->xchg_ready) {
        int xerr = 0;
        unsigned long long diag[3] = {0, 0, 0};
        CK(cudaMemcpy(&xerr, static_cast<char*>(h->xchg_buf) + 520, sizeof(int), cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(diag, static_cast<char*>(h->xchg_buf) + 536, sizeof diag, cudaMemcpyDeviceToHost));
        if (xerr) return fail(h, "tpls_fit: a peer-memory exchange timed out (a rank died or fell out of step)");
        h->stats.xchg_wait_ms = 1e-6 * (double)diag[0];
        h->stats.xchg_ms = 1e-6 * (double)diag[1];
        h->stats.xchg_count = (int64_t)diag[2];
    }
    for (int l = 0; l < L; ++l) {
        h->r2x[l].assign(R, 0.0);
        const double* s = ss.data() + (h->x[l].off_ss - h->off_ss);
        for (int a = 0; a < R; ++a) h->r2x[l][a] = 1.0 - s[a + 1] / s[0];
    }
    h->r2y.assign(R, 0.0);
    {
        const double* s = ss.data() + (size_t)L * (R + 1);
        for (int a = 0; a < R; ++a) h->r2y[a] = 1.0 - s[a + 1] / s[0];
    }
    long long total = 0;
    for (int a = 0; a < R; ++a) total += h->trips[a];
    h->stats.total_trips = total;
    if (h->res_stamps != nullptr && h->stats.resident_loops > 0) {
        long long hs[16];
        CK(cudaMemcpy(hs, h->res_stamps, sizeof hs, cudaMemcpyDeviceToHost));
        CK(cudaMemset(h->res_stamps, 0, sizeof hs));
        const double tr = (double)std::max<long long>(1, hs[9]);
        fprintf(stderr,
                "resident loop, us per trip (CTA 0, %lld trips): fold %.2f  rank-1 %.2f  projection %.2f  q/stop %.2f  "
                "contraction %.2f | barriers %.2f %.2f %.2f %.2f\n",
                hs[9], hs[0] / tr * 1e-3, hs[1] / tr * 1e-3, hs[2] / tr * 1e-3, hs[3] / tr * 1e-3, hs[4] / tr * 1e-3,
                hs[5] / tr * 1e-3, hs[6] / tr * 1e-3, hs[7] / tr * 1e-3, hs[8] / tr * 1e-3);
        long long fs[32];
        if (resident_fine_stamps(fs))
            fprintf(stderr,
                    "   cycles per trip: projection [t0 first round %.0f, later %.0f | t1+ first %.0f, later %.0f | epilogues %.0f | "
                    "fold+store %.0f]  contraction [u %.0f  rows %.0f  write %.0f]\n",
                    fs[0] / tr, fs[1] / tr, fs[2] / tr, fs[3] / tr, fs[4] / tr, fs[5] / tr, fs[8] / tr, fs[9] / tr, fs[10] / tr);
    }
    // launches / collectives / streamed bytes of the loops: one body was counted per component
    if (!cov_mode) {
        int per_trip = 0;
        for (int a = 0; a < R; ++a) {
            const tpls_ctx::BodyCount& b = h->body[a];
            const long long runs = b.resident ? 1 : (use_graph ? h->trips[a] : b.enqueued);
            h->stats.kernel_launches += b.launches * (runs - 1);
            h->stats.collectives += b.collectives * (runs - 1);
            h->stats.streamed_bytes += b.streamed * (h->trips[a] - 1) - b.tail_streamed;
            per_trip = std::max<long long>(per_trip, b.launches);
        }
        h->stats.launches_per_trip = per_trip;
    }
    double alg = 0.0;
    for (int l = 0; l < L; ++l) alg += (double)h->x[l].elem * n * h->x[l].p * (2.0 * total + R + 2);
    h->stats.alg_bytes = alg;
    h->fitted = true;
    return 0;
}

// ---------------------------------------------------------------------------
// getters
// ---------------------------------------------------------------------------

#define NEED_FIT()                                     \
    if (!h) return fail(nullptr, "NULL handle");       \
    if (!h->fitted) return fail(h, "not fitted")

int tpls_get_x_factor(tpls_handle h, int index, int mode, double* out) {
    NEED_FIT();
    if (index < 0 || index >= h->L) return fail(h, "tensor index %d out of range", index);
    Tensor& t = h->x[index];
    if (mode < 0 || mode >= t.ndim) return fail(h, "mode %d out of range", mode);
    if (mode == 0) return copy_out_transposed(h, h->T, h->n, h->R, out);
    return copy_out_transposed(h, t.W[mode], t.shape[mode], h->R, out);
}

int tpls_get_y_factor(tpls_handle h, int which, double* out) {
    NEED_FIT();
    if (which == 0) return copy_out_transposed(h, h->U, h->n, h->R, out);
    if (which == 1) return copy_out_transposed(h, h->Q, h->m, h->R, out);
    return fail(h, "which must be 0 (U) or 1 (Q)");
}

int tpls_get_coef(tpls_handle h, double* out) {
    NEED_FIT();
    CK(cudaMemcpyAsync(out, h->coef, sizeof(double) * h->R * h->R, cudaMemcpyDefault, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int tpls_get_r2x(tpls_handle h, int index, double* out) {
    NEED_FIT();
    if (index < 0 || index >= h->L) return fail(h, "tensor index %d out of range", index);
    memcpy(out, h->r2x[index].data(), sizeof(double) * h->R);
    return 0;
}

int tpls_get_r2y(tpls_handle h, double* out) {
    NEED_FIT();
    memcpy(out, h->r2y.data(), sizeof(double) * h->R);
    return 0;
}

int tpls_get_x_mean(tpls_handle h, int index, void* out) {
    NEED_FIT();
    if (index < 0 || index >= h->L) return fail(h, "tensor index %d out of range", index);
    Tensor& t = h->x[index];
    CK(cudaMemcpyAsync(out, t.mean_native, (size_t)t.elem * t.p, cudaMemcpyDefault, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int tpls_get_y_mean(tpls_handle h, double* out) {
    NEED_FIT();
    CK(cudaMemcpyAsync(out, h->ymean_d, sizeof(double) * h->m, cudaMemcpyDefault, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return 0;
}

int tpls_get_has_missing(tpls_handle h, int index, int* out) {
    NEED_FIT();
    if (index < 0 || index >= h->L) return fail(h, "tensor index %d out of range", index);
    *out = h->x[index].masked ? 1 : 0;
    return 0;
}

int tpls_get_trips(tpls_handle h, int* out) {
    NEED_FIT();
    memcpy(out, h->trips.data(), sizeof(int) * h->R);
    return 0;
}

int tpls_get_converged(tpls_handle h, int* out) {
    NEED_FIT();
    memcpy(out, h->converged.data(), sizeof(int) * h->R);
    return 0;
}

int tpls_get_profile(tpls_handle h, tpls_profile* out) {
    if (h && !h->prof.empty()) {
        CK(cudaSetDevice(h->device));
        CK(cudaStreamSynchronize(h->stream));
        prof_collect(h);
    }
    if (!h) return fail(nullptr, "NULL handle");
    *out = h->prof_sum;
    return 0;
}

int tpls_get_stats(tpls_handle h, tpls_stats* out) {
    if (!h) return fail(nullptr, "NULL handle");
    *out = h->stats;
    return 0;
}

// ---------------------------------------------------------------------------
// transform
// ---------------------------------------------------------------------------
int tpls_release_data(tpls_handle h) {
    if (!h) return fail(nullptr, "NULL handle");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    for (auto& t : h->x) {
        if (t.owned) pool_put(h, t.owned);
        if (t.owned2) pool_put(h, t.owned2);
        t.owned = t.owned2 = nullptr;
        t.src = nullptr;
        t.work = nullptr;
        t.set = false;
    }
    if (h->y_src) pool_put(h, h->y_src);
    if (h->y_work) pool_put(h, h->y_work);
    if (h->row_w) pool_put(h, h->row_w);
    h->y_src = h->y_work = h->row_w = nullptr;
    return 0;
}

int tpls_set_row_weights(tpls_handle h, const double* w, int64_t n) {
    if (!h) return fail(nullptr, "NULL handle");
    CK(cudaSetDevice(h->device));
    if (h->row_w) pool_put(h, h->row_w);
    h->row_w = nullptr;
    if (w == nullptr) return 0;
    if (n != h->n) return fail(h, "tpls_set_row_weights: %lld weights for %lld samples (call tpls_set_y first)", (long long)n, h->n);
    TRY(pool_get(h, (void**)&h->row_w, sizeof(double) * n));
    CK(cudaMemcpyAsync(h->row_w, w, sizeof(double) * n, cudaMemcpyDefault, h->stream));
    h->fitted = false;
    return 0;
}

int tpls_trim(tpls_handle h) {
    if (!h) return fail(nullptr, "NULL handle");
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    pool_trim(h);
    return 0;
}

}  // extern "C"
