// Dataset-side helpers for the sequential sweeps (device resident CSC; reference dataset.py:94-134
// hands out column slices, here the column slices are additionally range-partitioned over the
// CTAs of a thread-block cluster and tagged with intra-CTA read-after-write hazards).
#include "common.cuh"
#include "sparsepoly_b200.h"

namespace {

// out[j] = sum_i x_ij^2  (sparse_factorization_machines.py:409  row_norms(X.T, squared=True) -> sklearn's
// csr_row_norms: ONE sequential sum per feature, samples ascending).  Setup-only, so each thread walks one
// column in exactly that order: the step sizes of cd_linear (cd_linear.py:22) are then bit-identical to
// the reference's, which matters because pcd amplifies ulp-level differences at n >= 10^4.
__global__ void col_norm_sq_kernel(int d, const int32_t *__restrict__ indptr,
                                   const double *__restrict__ data, double *out) {
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < d; j += gridDim.x * blockDim.x) {
        double acc = 0.0;
        for (int e = indptr[j]; e < indptr[j + 1]; e++) acc += data[e] * data[e];
        out[j] = acc;
    }
}

// col_part[j*(C+1)+c] = first CSC offset of column j whose row index >= c*chunk  (c=0..C)
__global__ void partition_kernel(int d, int C, int chunk, const int32_t *__restrict__ indptr,
                                 const int32_t *__restrict__ indices, int32_t *col_part) {
    const long long total = (long long)d * (C + 1);
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < total;
         g += (long long)gridDim.x * blockDim.x) {
        const int j = (int)(g / (C + 1)), c = (int)(g % (C + 1));
        int lo = indptr[j], hi = indptr[j + 1];
        if (c == C) { col_part[g] = hi; continue; }
        const long long bound = (long long)c * chunk;
        while (lo < hi) {                       // lower_bound(rows, bound)
            const int mid = (lo + hi) >> 1;
            if (indices[mid] < bound) lo = mid + 1; else hi = mid;
        }
        col_part[g] = lo;
    }
}

__global__ void order_ptr_kernel(int d, int C, const int32_t *__restrict__ idx_feat,
                                 const int32_t *__restrict__ col_part, int32_t *pos_ptr) {
    const long long total = (long long)d * (C + 1);
    for (long long g = blockIdx.x * (long long)blockDim.x + threadIdx.x; g < total;
         g += (long long)gridDim.x * blockDim.x) {
        const int t = (int)(g / (C + 1)), c = (int)(g % (C + 1));
        pos_ptr[g] = col_part[(long long)idx_feat[t] * (C + 1) + c];
    }
}

// flag_idx[e] = row | bit31 if the same sample also has a nonzero in the column visited at
// position t-1, | bit30 if it has one in the column visited at position t-2: records of those
// samples are (possibly) still being rewritten when position t's asynchronous prefetch is
// issued, so the sweep kernel re-reads them after the barrier.  pos_conf[t] = 1 when ANY sample
// of column t carries bit31 (columns t-1 and t are not sample-disjoint).
__device__ __forceinline__ bool col_has_row(const int32_t *__restrict__ indices, int lo, int hi, int row) {
    const int end = hi;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (indices[mid] < row) lo = mid + 1; else hi = mid;
    }
    return (lo < end) && (indices[lo] == row);
}

__global__ void order_flag_kernel(int d, const int32_t *__restrict__ idx_feat,
                                  const int32_t *__restrict__ indptr,
                                  const int32_t *__restrict__ indices, int32_t *flag_idx,
                                  int32_t *pos_conf) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const int n_warps = (gridDim.x * blockDim.x) >> 5;
    for (int t = warp; t < d; t += n_warps) {
        const int j = idx_feat[t];
        int p1lo = 0, p1hi = 0, p2lo = 0, p2hi = 0;
        if (t > 0) { const int jp = idx_feat[t - 1]; p1lo = indptr[jp]; p1hi = indptr[jp + 1]; }
        if (t > 1) { const int jp = idx_feat[t - 2]; p2lo = indptr[jp]; p2hi = indptr[jp + 1]; }
        bool any1 = false;
        for (int e = indptr[j] + lane; e < indptr[j + 1]; e += 32) {
            const int row = indices[e];
            const bool h1 = col_has_row(indices, p1lo, p1hi, row);
            const bool h2 = col_has_row(indices, p2lo, p2hi, row);
            any1 = any1 || h1;
            flag_idx[e] = (int32_t)((uint32_t)row | (h1 ? SP_FLAG_BIT : 0u) | (h2 ? SP_FLAG2_BIT : 0u));
        }
        any1 = __any_sync(0xffffffffu, any1);
        if (lane == 0) pos_conf[t] = any1 ? 1 : 0;
    }
}

__global__ void transpose_kernel(const double *__restrict__ in, double *__restrict__ out, int rows,
                                 int cols) {
    __shared__ double tile[32][33];
    const size_t mat = (size_t)rows * cols;             // matrix blockIdx.y of a batch
    in += blockIdx.y * mat;
    out += blockIdx.y * mat;
    // tiles are numbered along ONE grid dimension (grid.y is limited to 65 535: a [d,k] matrix with d > 2 M rows
    // -- sparse CTR feature spaces -- would not fit there)
    const int tiles_x = (cols + 31) / 32;
    const int bx = (int)(blockIdx.x % tiles_x) * 32, by = (int)(blockIdx.x / tiles_x) * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int rr = by + r, cc = bx + threadIdx.x;
        if (rr < rows && cc < cols) tile[r][threadIdx.x] = in[(size_t)rr * cols + cc];
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        const int cc = bx + r, rr = by + threadIdx.x;
        if (rr < rows && cc < cols) out[(size_t)cc * rows + rr] = tile[threadIdx.x][r];
    }
}

int blocks_for(long long work, int threads) {
    long long b = (work + threads - 1) / threads;
    if (b > 148 * 16) b = 148 * 16;
    if (b < 1) b = 1;
    return (int)b;
}

}  // namespace

extern "C" int sp_col_norm_sq(const sp_dataset *ds, double *out, sp_stream stream) {
    if (!ds || !ds->csc_indptr || !out) { sp_set_error("sp_col_norm_sq: invalid argument"); return SP_ERR_INVALID; }
    if (ds->n_features == 0) return SP_OK;
    col_norm_sq_kernel<<<blocks_for((long long)ds->n_features, 128), 128, 0, (cudaStream_t)stream>>>(
        ds->n_features, ds->csc_indptr, ds->csc_data, out);
    SP_LAUNCH_CHECK("col_norm_sq_kernel");
    return SP_OK;
}

extern "C" int sp_plan_partition(const sp_dataset *ds, int n_cta, int32_t *col_part, sp_stream stream) {
    if (!ds || !ds->csc_indptr || !col_part || n_cta < 1 || n_cta > 16) {
        sp_set_error("sp_plan_partition: invalid argument (n_cta must be 1..16)");
        return SP_ERR_INVALID;
    }
    if (ds->n_features == 0) return SP_OK;
    const int chunk = (ds->n_samples + n_cta - 1) / n_cta;
    partition_kernel<<<blocks_for((long long)ds->n_features * (n_cta + 1), 256), 256, 0,
                       (cudaStream_t)stream>>>(ds->n_features, n_cta, chunk > 0 ? chunk : 1,
                                               ds->csc_indptr, ds->csc_indices, col_part);
    SP_LAUNCH_CHECK("partition_kernel");
    return SP_OK;
}

extern "C" int sp_plan_order(const sp_dataset *ds, int n_cta, const int32_t *col_part,
                             const int32_t *idx_feat, int32_t *pos_ptr, int32_t *flag_idx,
                             int32_t *pos_conf, sp_stream stream) {
    if (!ds || !col_part || !idx_feat || !pos_ptr || !flag_idx || !pos_conf || n_cta < 1 || n_cta > 16) {
        sp_set_error("sp_plan_order: invalid argument");
        return SP_ERR_INVALID;
    }
    if (ds->n_features == 0) return SP_OK;
    if (ds->n_samples >= (1 << 30)) {
        sp_set_error("sp_plan_order: n_samples >= 2^30 is not supported (two flag bits in the row index)");
        return SP_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    order_ptr_kernel<<<blocks_for((long long)ds->n_features * (n_cta + 1), 256), 256, 0, st>>>(
        ds->n_features, n_cta, idx_feat, col_part, pos_ptr);
    SP_LAUNCH_CHECK("order_ptr_kernel");
    order_flag_kernel<<<blocks_for((long long)ds->n_features * 32, 256), 256, 0, st>>>(
        ds->n_features, idx_feat, ds->csc_indptr, ds->csc_indices, flag_idx, pos_conf);
    SP_LAUNCH_CHECK("order_flag_kernel");
    return SP_OK;
}

extern "C" int sp_transpose_f64_batch(const double *in, double *out, int batch, int rows, int cols, sp_stream stream) {
    if (!in || !out || batch < 0 || batch > 65535 || rows < 0 || cols < 0) {
        sp_set_error("sp_transpose_f64: invalid argument");
        return SP_ERR_INVALID;
    }
    if (batch == 0 || rows == 0 || cols == 0) return SP_OK;
    const long long tiles = (long long)((cols + 31) / 32) * ((rows + 31) / 32);
    if (tiles > 2147483647LL) { sp_set_error("sp_transpose_f64: matrix too large (%d x %d)", rows, cols); return SP_ERR_INVALID; }
    dim3 grid((unsigned)tiles, (unsigned)batch), block(32, 8);
    transpose_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(in, out, rows, cols);
    SP_LAUNCH_CHECK("transpose_kernel");
    return SP_OK;
}

extern "C" int sp_transpose_f64(const double *in, double *out, int rows, int cols, sp_stream stream) {
    return sp_transpose_f64_batch(in, out, 1, rows, cols, stream);
}
