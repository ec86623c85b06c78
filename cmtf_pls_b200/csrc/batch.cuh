// Batched fits (tpls_fit_batch): many small tPLS / ctPLS problems, one CTA per problem, the WHOLE fit of a problem
// -- column statistics, centring, every component's inner loop, regression, deflation -- inside that CTA.  No grid
// barrier, no host round trip, no launch per fit: a launch of G CTAs runs G fits at once (DESIGN.md section 4d).
#pragma once

#include "rank1.cuh"

namespace tpls {

constexpr int kBatchMaxResp = 8;    // responses of a batched fit
constexpr int kBatchMaxComp = 32;   // components of a batched fit

struct BatchTensor {
    const void* x;          // input [problem][n][p] (C order), never written
    long long x_bstride;    // elements between problems; 0 = every problem shares this tensor
    int dtype;              // 0 = float32, 1 = float64
    int p;
    int nmodes;             // modes of Z (= ndim(X) - 1)
    int dims[kMaxZModes];
    int w_rows;             // sum of dims: rows of this tensor's loading block in W
    int r1_nmax, r1_zs, r1_mt, r1_tab;  // rank-1 workspace geometry (rank1_workspace_doubles)
    // byte offsets into a problem's working set
    size_t off_x;           // centred / deflated working copy [n][p] in the storage type
    size_t off_mean, off_cnt, off_z, off_wk, off_fac, off_rowcnt;  // doubles: [p] x 4, [w_rows], [n]
    // outputs, leading axis = problem
    double* W;              // [problem][w_rows][R]
    void* mean_out;         // [problem][p] in the storage type
};

struct BatchArgs {
    BatchTensor x[kMaxTensors];
    int n_tensors;
    int batch;
    int n, m, R;
    const double* y;        // [problem][n][m]
    long long y_bstride;
    const double* row_w;    // [problem][n] 0/1 weights, or nullptr
    double tol;
    int max_iter;
    int normalize_on_break;
    size_t ws_bytes;        // bytes of one problem's working set
    size_t off_y, off_t, off_u, off_r1;  // byte offsets: Y [n][m], T [R][n], u [n], rank-1 workspace
    char* gws;              // global slots [gridDim.x][ws_bytes]; nullptr: the working set is in dynamic shared memory
    // outputs
    double *T, *U, *Q, *coef, *r2x, *r2y, *y_mean;
    int *trips, *conv, *has_missing;
};

cudaError_t launch_batch_fit(const BatchArgs& a, int grid, size_t smem_bytes, cudaStream_t s);
// co-resident CTAs of batch_fit_kernel on this device with smem_bytes of dynamic shared memory (0 on failure)
int batch_fit_max_ctas(size_t smem_bytes);
// dynamic shared memory a CTA can have beside the kernel's static shared memory
size_t batch_fit_smem_limit();

}  // namespace tpls
