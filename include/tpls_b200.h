/* tpls_b200 -- C ABI of the B200-native tensor-PLS (tPLS / coupled ctPLS) fit path.
 *
 * The reference (meyer-lab/cmtf-pls) is pure Python and has no FFI of its own;
 * its boundary for this path is the estimator API
 *     tPLS.fit / predict / transform     cmtf_pls/tpls.py:73-186
 *     ctPLS.fit / predict / transform    cmtf_pls/cmtf.py:85-231
 * and the fitted attributes listed in SURVEY.md §8 row a15.  Each entry point
 * below names the reference lines it replaces.  The Python classes in
 * cmtf_pls_b200/{tpls,cmtf}.py bind these with ctypes and keep the reference's
 * names, argument meaning and error behaviour (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; the message is
 *     available from tpls_last_error().  No exceptions cross the ABI.
 *   - data pointers may be HOST or DEVICE pointers (resolved with
 *     cudaPointerGetAttributes); results are copied into caller-owned buffers.
 *   - a handle is bound to one device and one stream; calls on one handle must
 *     not overlap.  Different handles are independent.
 *   - sample-mode sharding: every rank holds the same rows of every coupled
 *     tensor and of Y; only small replicated quantities cross devices (NCCL).
 */
#ifndef TPLS_B200_H
#define TPLS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tpls_ctx* tpls_handle;

enum { TPLS_F32 = 0, TPLS_F64 = 1 };

/* tpls_set_x flags */
enum {
    TPLS_X_MAY_OVERWRITE = 1 /* a DEVICE tensor may be centred/deflated in place (saves one copy of X) */
};

/* tpls_fit flags */
enum {
    TPLS_FIT_NORMALIZE_ON_BREAK = 1, /* the other reading of tensorly's last ALS sweep, oracle/_cp.py */
    TPLS_FIT_PROFILE = 2,            /* time every pass with CUDA events on the handle's stream (tpls_get_profile) */
    TPLS_FIT_COVARIANCE = 4          /* cross-covariance mode (SURVEY.md §8f n4): per component ONE pass forms C = X'Y
                                        (all responses at once), the inner NIPALS iteration then runs on (P x M)-sized
                                        data in a single kernel -- no pass over X and no collective per inner trip.
                                        Same results to rounding; needs <= 8 responses (<= 4 with NaNs), else the
                                        streaming loop is used.  tpls_stats.covariance_mode tells which one ran. */
};

/* kernel classes of tpls_get_profile */
enum {
    TPLS_K_COLSTAT = 0,          /* column sums / counts (np.nanmean, tpls.py:66) */
    TPLS_K_CONTRACT = 1,         /* Z = X x_1 u (tpls.py:83) */
    TPLS_K_PROJECT = 2,          /* t = X x_2 w2 x_3 w3 ... (tpls.py:97-99) */
    TPLS_K_DEFLATE_CONTRACT = 3, /* centring or rank-1 deflation fused with the next contraction */
    TPLS_K_RESIDUAL = 4,         /* read-only residual norm after the last component */
    TPLS_K_RANK1 = 5,            /* single-CTA rank-1 step (tpls.py:84-88) */
    TPLS_K_YSIDE = 6,            /* passes over Y (q, u, Y deflation) */
    TPLS_K_OTHER = 7,            /* second reduction stages and the scalar tail of a trip */
    TPLS_K_NCCL = 8,             /* ncclAllReduce calls */
    TPLS_K_XCHG = 9              /* peer-memory exchange kernels (second reduction stage + sum over the ranks) */
};
#define TPLS_N_KERNEL_CLASSES 10

#define TPLS_MAX_TENSORS 8
#define TPLS_MAX_MODES 8

int tpls_version(void);
/* last error of `h`, or of the last failed call without a handle when h == NULL */
const char* tpls_last_error(tpls_handle h);

/* Context bound to CUDA device `device`.  `cuda_stream` is a cudaStream_t to
 * enqueue on, or NULL for a private non-blocking stream. */
int tpls_create(tpls_handle* out, int device, void* cuda_stream);
int tpls_destroy(tpls_handle h);
/* Rebinds the handle to another stream (NULL: back to the private one).  Work already enqueued is waited for
 * first, so one handle per device can follow the caller's current stream from call to call. */
int tpls_set_stream(tpls_handle h, void* cuda_stream);

/* Multi-GPU (one process per GPU).  Rank 0 obtains a 128-byte id, the caller
 * broadcasts it by any means, every rank calls tpls_comm_init. */
int tpls_comm_unique_id(void* id128);
int tpls_comm_init(tpls_handle h, const void* id128, int rank, int world);

/* Optional, after tpls_comm_init: replace the small per-trip all-reduces (Z, q, the stop norm; a few KB each)
 * by a one-shot exchange over NVLink peer memory (csrc/xchg.cuh).  Every rank obtains the 64-byte CUDA IPC
 * handle of its exchange buffer, the caller all-gathers the handles in rank order, every rank opens them.
 * Without these two calls NCCL is used throughout. */
int tpls_comm_xchg_handle(tpls_handle h, void* handle64);
int tpls_comm_xchg_open(tpls_handle h, const void* handles /* world x 64 bytes */);

/* Training data.  X number `index` of `n_tensors` coupled tensors, C-ordered,
 * shape[0] = this rank's sample count; Y is (n, m) float64 C-ordered.
 * Replaces the array arguments of tPLS.fit (tpls.py:73) / ctPLS.fit (cmtf.py:85).
 * Caller memory is never modified unless TPLS_X_MAY_OVERWRITE is given. */
int tpls_set_x(tpls_handle h, int index, const void* x, int dtype, int ndim, const int64_t* shape, int flags);
int tpls_set_y(tpls_handle h, const double* y, int64_t n, int64_t m);

/* Optional 0/1 sample weights for the NEXT fit (n = this rank's sample count; NULL clears them).  Rows with
 * weight 0 are held out: they contribute to no sample-mode reduction (means, Z, q, the stop test, the
 * regression, R2), but they are still centred, projected and deflated with their own projections -- so their
 * rows of the score matrix are exactly transform() of the held-out data under the fold's model
 * (tpls.py:145-165).  This is how a K-fold Q2Y sweep runs without copying X (validate.py:24-37 refits on
 * sliced copies).  Call after tpls_set_y; cleared by tpls_release_data. */
int tpls_set_row_weights(tpls_handle h, const double* w, int64_t n);

/* The NIPALS fit: preprocess (tpls.py:44-71) + the component loop (tpls.py:76-120,
 * cmtf.py:88-140).  n_tensors = how many tpls_set_x slots are in use. */
int tpls_fit(tpls_handle h, int n_tensors, int n_components, double tol, int max_iter, int flags);

/* Fitted state (row a15).  All outputs are C-ordered float64 unless noted. */
int tpls_get_x_factor(tpls_handle h, int index, int mode, double* out); /* mode 0: scores (n, R); k: (shape[k], R) */
int tpls_get_y_factor(tpls_handle h, int which, double* out);           /* 0: U (n, R)   1: Q (m, R) */
int tpls_get_coef(tpls_handle h, double* out);                           /* (R, R), upper triangular */
int tpls_get_r2x(tpls_handle h, int index, double* out);                 /* (R,) */
int tpls_get_r2y(tpls_handle h, double* out);                            /* (R,) */
int tpls_get_x_mean(tpls_handle h, int index, void* out);                /* shape[1:], in X's dtype */
int tpls_get_y_mean(tpls_handle h, double* out);                         /* (m,) */
int tpls_get_has_missing(tpls_handle h, int index, int* out);
int tpls_get_trips(tpls_handle h, int* out);                             /* (R,) inner iterations taken */
int tpls_get_converged(tpls_handle h, int* out);                         /* (R,) 1 = the component met the stop test of
                                                                            tpls.py:103 (possibly on the last allowed trip) */

typedef struct tpls_stats {
    double fit_ms;              /* device time of the last tpls_fit (CUDA events on the handle's stream) */
    double alg_bytes;           /* sum_l s*N_local*P_l*(2*sum(trips) + R + 2)  (SURVEY.md §8d) */
    double streamed_bytes;      /* bytes of X actually read + written by the passes of the last fit */
    int64_t kernel_launches;    /* kernels of this library launched by the last fit */
    int64_t total_trips;
    int64_t collectives;        /* NCCL all-reduces issued by the last fit */
    double h2d_bytes;           /* bytes staged host->device by tpls_set_x / tpls_set_y since the last fit */
    int64_t covariance_mode;    /* 1 when the last fit ran the cross-covariance loop */
    int64_t last_transform_path; /* last tpls_transform: 1 = read-only path (complete data), 2 = sequential path */
    int64_t graph_launches;     /* 1 when the last fit ran as ONE CUDA graph (a WHILE node per component: the host takes
                                   no part in the inner loops), 0 when the host enqueued the trips */
    int64_t launches_per_trip;  /* kernels in one inner trip of the last streaming fit (3 + 2 * n_tensors when the Y side
                                   is fused into the X passes) */
    /* peer-memory exchanges of the last fit on THIS rank (0 without them): how many, the time from the start of an
     * exchange kernel until every rank's contribution had arrived, and the part of it spent waiting for the peers --
     * the rank that waits least is the slowest one */
    int64_t xchg_count;
    double xchg_ms;
    double xchg_wait_ms;
    int64_t resident_loops;     /* components whose inner trips ran in ONE persistent launch (one CTA per SM, rows cached in
                                   shared memory, grid barriers between the phases of a trip): working sets of up to 256 MB
                                   (TPLS_RESIDENT_MB), one GPU, <= 8 responses */
} tpls_stats;
int tpls_get_stats(tpls_handle h, tpls_stats* out);

typedef struct tpls_profile {
    double ms[TPLS_N_KERNEL_CLASSES];        /* summed launch durations of the profiled fits since the last call */
    int64_t launches[TPLS_N_KERNEL_CLASSES];
    double bytes[TPLS_N_KERNEL_CLASSES];     /* algorithmic bytes of X moved by those launches */
} tpls_profile;
int tpls_get_profile(tpls_handle h, tpls_profile* out);

/* Frees the device copies of X and Y held by the handle (the fitted state stays readable). */
int tpls_release_data(tpls_handle h);
/* tpls_release_data keeps the X-sized buffers cached for the next fit on this handle (allocating tens
 * of GB costs hundreds of ms); tpls_trim returns the cached buffers to the CUDA driver. */
int tpls_trim(tpls_handle h);

/* New data through a fitted model: scores (n_new, R) of transform (tpls.py:145-165,
 * cmtf.py:179-210) -- centre with the training mean, then per component project
 * (averaging over the coupled tensors) and deflate with the stored loadings.
 * Stateless with respect to tpls_fit: the model is passed in, so it also serves an
 * estimator that was pickled or fitted elsewhere.  xs[l]: (n_new, ps[l]) in dtypes[l];
 * means[l]: ps[l] values in dtypes[l]; wkrons[l]: (R, ps[l]) float64, row a = kron of the
 * component-a loading vectors.
 * proj_offset (R) and proj_gram (R x R), optional: c_a = mean_l <mean_l, wkron_l[a]> and
 * G_ba = mean_l <wkron_l[b], wkron_l[a]>.  With them, data WITHOUT NaNs is never copied or
 * deflated: R read-only projection passes over the rows where they lie, then the deflation
 * recurrence t_a = r_a - c_a - sum_{b<a} t_b G_ba on the scores.  Rows with NaNs (or NULL
 * constants) take the sequential path with the masked projection (missingvals.py:23-38). */
int tpls_transform(tpls_handle h, int n_tensors, int n_components, const void* const* xs, const int* dtypes,
                   int64_t n_new, const int64_t* ps, const void* const* means, const double* const* wkrons,
                   const double* proj_offset, const double* proj_gram, double* scores_out);

/* Dense reconstruction from a fitted model (X_reconstructed, tpls.py:188-189 = util.py:18-20 + the mean; the
 * imputation path of tests/test_missingvals.py:83-91):  out[i, c] = mean[c] + sum_a scores[i, a] * wkron[a, c].
 * scores: (n, R) float64 C-ordered; wkron: (R, p) float64; mean: p values in `mean_dtype` (or NULL);
 * out: (n, p) float64 C-ordered.  Host or device pointers; a host `out` is filled block by block. */
int tpls_reconstruct(tpls_handle h, int n_components, const double* scores, int64_t n, int64_t p, const double* wkron,
                     const void* mean, int mean_dtype, double* out);

/* ---- batched fits: many small problems in ONE launch, one CTA per problem ----
 *
 * B independent tPLS / ctPLS fits (cross-validation folds, choosing the number of components, repeated seeds,
 * one model per subgroup), each with exactly the semantics of tpls_fit (+ tpls_set_row_weights): the same
 * statistics, centring, inner loop, stop test, regression and deflations, rounded at the same points.  The whole
 * fit of a problem runs inside one CTA of a persistent kernel (csrc/batch.cu): no grid barrier, no host round trip
 * and no launch per fit.  The working set of a problem lives in shared memory when it fits (~195 KB), else in the
 * CTA's slot of a global workspace.
 *
 * Problem b reads tensor l at xs[l] + b * x_batch_stride[l] elements (0 = every problem shares the tensor),
 * shaped shapes[l][0 .. ndims[l]) = (n, d1, ...) in C order; Y at y + b * y_batch_stride, (n, m) float64; row_w
 * (batch, n) 0/1 weights or NULL.  Inputs may be host or device memory; device inputs are read where they are and
 * never written, host inputs are staged once.  Outputs are caller-owned, host or device, leading axis = problem.
 *
 * Returns 0, non-zero on an invalid argument, or TPLS_E_BATCH_UNSUPPORTED -- with nothing written -- when a
 * problem is outside the kernel's limits: more than 8 responses, more than 32 components, a rank-1 workspace
 * above 200 KB, or a working set per problem above TPLS_BATCH_MB megabytes (default 16).  The caller then fits the
 * problems one by one with tpls_fit.  TPLS_BATCH=0 forces that code; TPLS_BATCH_SMEM=0 keeps the working sets in
 * global memory (both for A/B runs and tests). */
#define TPLS_E_BATCH_UNSUPPORTED 2

typedef struct tpls_batch_out {
    double* T; double* U;             /* (B, n, R) */
    double* Q;                        /* (B, m, R) */
    double* W[TPLS_MAX_TENSORS];      /* (B, sum_k shape[k] for k >= 1, R): the loading matrices of modes 1.. back to back */
    double* coef;                     /* (B, R, R) */
    double* r2x;                      /* (B, n_tensors, R) */
    double* r2y;                      /* (B, R) */
    void* x_mean[TPLS_MAX_TENSORS];   /* (B, P_l) in X's dtype */
    double* y_mean;                   /* (B, m) */
    int* trips; int* converged;       /* (B, R) */
    int* has_missing;                 /* (B, n_tensors) */
    double fit_ms;                    /* out: device time of the call (staging and result copies included) */
} tpls_batch_out;

int tpls_fit_batch(tpls_handle h, int n_tensors, int64_t batch,
                   const void* const* xs, const int* dtypes, const int* ndims, const int64_t* const* shapes,
                   const int64_t* x_batch_stride,
                   const double* y, int64_t m, int64_t y_batch_stride,
                   const double* row_w,
                   int n_components, double tol, int max_iter, int flags, tpls_batch_out* out);

/* ---- single operators (used by the parity tests and by bench.py's per-kernel roofline) ----
 * All pointers here are DEVICE pointers; x is (n, p) C-ordered with p*elem a multiple of 16. */
/* z[p] = sum_i x[i,:] * u[i]                      tpls.py:83  (masked: missingvals.py:7-20, n_total = n) */
int tpls_op_contract(tpls_handle h, const void* x, int dtype, int64_t n, int64_t p, const double* u, int masked,
                     double* z_out, float* ms_out, int repeats);
/* t[i] = sum_c x[i,c] * w[c]                      tpls.py:97-99 (masked: missingvals.py:23-38) */
int tpls_op_project(tpls_handle h, const void* x, int dtype, int64_t n, int64_t p, const double* w, int masked,
                    double* t_out, float* ms_out, int repeats);
/* x -= t (x) w in place, z[p] = sum_i x_new[i,:]*u[i], ss = ||x_new||^2   tpls.py:109 fused with :83 and util.py:7-15 */
int tpls_op_deflate_contract(tpls_handle h, void* x, int dtype, int64_t n, int64_t p, const double* t,
                             const double* w, const double* u, int masked, double* z_out, double* ss_out,
                             float* ms_out, int repeats);
/* unit weight vectors of z (dims[0..nmodes)), concatenated into w_out; kron into wkron_out[p]  tpls.py:84-90 */
int tpls_op_rank1(tpls_handle h, const double* z, int nmodes, const int* dims, double tol, int flags, double* w_out,
                  double* wkron_out, int* sweeps_out, float* ms_out, int repeats);

#ifdef __cplusplus
}
#endif
#endif /* TPLS_B200_H */
