// Device input (DESIGN.md 2): checks a design matrix that already lives on the GPU and converts it to the library's
// layout (int32 indptr / indices, fp64 values) in one pass, so a CUDA X never goes through the host.
//
// sp_csr_prepare: one warp per row, coalesced over the row's nonzeros in chunks of 32 lanes; the column of the
// previous nonzero is carried across chunks for the "strictly increasing" test.  Every fault is recorded as the first
// (lowest) offending row with atomicMin, so the report does not depend on the schedule.  A dense (strided) matrix
// takes the same pass with every entry stored.
// sp_csr_sum_runs: the second half of canonicalisation, after a stable sort of the (row, column) keys: each run of
// equal keys is summed left to right (scipy's csr_sum_duplicates order) and written compacted.
#include <math.h>

#include "common.cuh"
#include "sparsepoly_b200.h"

namespace {

constexpr int kRowsPerBlock = 8;     // warps per 256-thread block, one row each

__global__ void report_init_kernel(int64_t *report) {
    const int t = threadIdx.x;
    if (t < SP_CSR_REPORT_LEN)
        report[t] = (t == SP_CSR_REPORT_INDPTR0 || t == SP_CSR_REPORT_INDPTRN || t == SP_CSR_REPORT_N_UNSORTED)
                        ? 0 : INT64_MAX;
}

template <typename V> __device__ __forceinline__ double widen(V v) { return (double)v; }

// flags a lane accumulates over its entries of one row
enum { F_RANGE = 1, F_NAN = 2, F_INF = 4, F_UNSORTED = 8 };

__device__ __forceinline__ void report_row(int flags, int64_t row, int64_t *report) {
    // one lane per row reports, after the warp has OR-ed its lanes' flags
    if (flags & F_RANGE) atomicMin((unsigned long long *)&report[SP_CSR_REPORT_RANGE], (unsigned long long)row);
    if (flags & F_NAN) atomicMin((unsigned long long *)&report[SP_CSR_REPORT_NAN], (unsigned long long)row);
    if (flags & F_INF) atomicMin((unsigned long long *)&report[SP_CSR_REPORT_INF], (unsigned long long)row);
    if (flags & F_UNSORTED) {
        atomicAdd((unsigned long long *)&report[SP_CSR_REPORT_N_UNSORTED], 1ull);
        atomicMin((unsigned long long *)&report[SP_CSR_REPORT_UNSORTED], (unsigned long long)row);
    }
}

__device__ __forceinline__ int value_flags(double x) {
    return isnan(x) ? F_NAN : (isinf(x) ? F_INF : 0);
}

__device__ __forceinline__ int warp_or(int v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v |= __shfl_xor_sync(0xffffffffu, v, m);
    return v;
}

template <typename IP, typename IX, typename V>
__global__ void __launch_bounds__(32 * kRowsPerBlock)
csr_prepare_kernel(int64_t n_rows, int64_t n_cols, int64_t nnz, const IP *__restrict__ indptr,
                   const IX *__restrict__ indices, const V *__restrict__ values, int n_dummy,
                   int32_t *__restrict__ out_indptr, int32_t *__restrict__ out_indices, double *__restrict__ out_data,
                   int64_t *report) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kRowsPerBlock + (threadIdx.x >> 5);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        report[SP_CSR_REPORT_INDPTR0] = (int64_t)indptr[0];
        report[SP_CSR_REPORT_INDPTRN] = (int64_t)indptr[n_rows];
        if (out_indptr) out_indptr[0] = (int32_t)indptr[0];
    }
    if (row >= n_rows) return;
    const int64_t a = (int64_t)indptr[row], b = (int64_t)indptr[row + 1];
    if (b < a && lane == 0)
        atomicMin((unsigned long long *)&report[SP_CSR_REPORT_DECREASING], (unsigned long long)row);
    // a corrupt indptr is reported above and never read out of bounds
    const int64_t s = a < 0 ? 0 : (a > nnz ? nnz : a);
    const int64_t e = b < s ? s : (b > nnz ? nnz : b);
    const int64_t shift = (row + 1) * (int64_t)n_dummy;      // dummies of rows 0..row
    if (out_indptr && lane == 0) out_indptr[row + 1] = (int32_t)(b + shift);
    if (out_indices && lane < n_dummy) {
        out_indices[s + row * n_dummy + lane] = lane;
        out_data[s + row * n_dummy + lane] = 1.0;
    }
    int flags = 0;
    int64_t prev = -1;                                       // column of the nonzero before this chunk
    for (int64_t p0 = s; p0 < e; p0 += 32) {
        const int64_t p = p0 + lane;
        const bool live = p < e;
        const int64_t c = live ? (int64_t)indices[p] : INT64_MAX;
        const double x = live ? widen(values[p]) : 0.0;
        int64_t left = __shfl_up_sync(0xffffffffu, c, 1);
        if (lane == 0) left = prev;
        if (live) {
            if (c < 0 || c >= n_cols) flags |= F_RANGE;
            flags |= value_flags(x);
            if (c <= left) flags |= F_UNSORTED;
            if (out_indices) {
                out_indices[p + shift] = (int32_t)(c + n_dummy);
                out_data[p + shift] = x;
            }
        }
        prev = __shfl_sync(0xffffffffu, c, 31);          // (only a full chunk has a successor)
    }
    flags = warp_or(flags);
    if (lane == 0 && flags) report_row(flags, row, report);
}

// dense X[i, j] = values[i * stride_row + j * stride_col]: every entry is stored (host_csr's dense layout)
template <typename V>
__global__ void __launch_bounds__(32 * kRowsPerBlock)
dense_prepare_kernel(int64_t n_rows, int64_t n_cols, const V *__restrict__ values, int64_t stride_row,
                     int64_t stride_col, int n_dummy, int32_t *__restrict__ out_indptr,
                     int32_t *__restrict__ out_indices, double *__restrict__ out_data, int64_t *report) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kRowsPerBlock + (threadIdx.x >> 5);
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        report[SP_CSR_REPORT_INDPTRN] = n_rows * n_cols;
        if (out_indptr) out_indptr[0] = 0;
    }
    if (row >= n_rows) return;
    const int64_t width = n_cols + n_dummy;
    const int64_t base = row * width;
    if (out_indptr && lane == 0) out_indptr[row + 1] = (int32_t)(base + width);
    if (out_indices && lane < n_dummy) {
        out_indices[base + lane] = lane;
        out_data[base + lane] = 1.0;
    }
    int flags = 0;
    const V *x_row = values + row * stride_row;
    for (int64_t j = lane; j < n_cols; j += 32) {
        const double x = widen(x_row[j * stride_col]);
        flags |= value_flags(x);
        if (out_indices) {
            out_indices[base + n_dummy + j] = (int32_t)(j + n_dummy);
            out_data[base + n_dummy + j] = x;
        }
    }
    flags = warp_or(flags);
    if (lane == 0 && flags) report_row(flags, row, report);
}

__global__ void sum_runs_kernel(int64_t nnz, const int64_t *__restrict__ keys, const int64_t *__restrict__ perm,
                                const double *__restrict__ data, const int64_t *__restrict__ run_index,
                                int64_t n_cols, int32_t *__restrict__ out_indices, double *__restrict__ out_data) {
    const int64_t p = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nnz) return;
    const int64_t key = keys[p];
    if (p > 0 && keys[p - 1] == key) return;                 // not the head of its run
    double sum = data[perm[p]];                               // scipy: x = first; x += next ... (no 0 + first)
    for (int64_t q = p + 1; q < nnz && keys[q] == key; q++) sum += data[perm[q]];
    const int64_t r = run_index[p];
    out_indices[r] = (int32_t)(key % n_cols);
    out_data[r] = sum;
}

template <typename IP, typename IX, typename V>
void launch_csr(int64_t n_rows, int64_t n_cols, int64_t nnz, const void *indptr, const void *indices,
                const void *values, int n_dummy, int32_t *oi, int32_t *ox, double *od, int64_t *report,
                cudaStream_t st) {
    const unsigned grid = (unsigned)((n_rows + kRowsPerBlock - 1) / kRowsPerBlock);
    csr_prepare_kernel<IP, IX, V><<<grid > 0 ? grid : 1, 32 * kRowsPerBlock, 0, st>>>(
        n_rows, n_cols, nnz, (const IP *)indptr, (const IX *)indices, (const V *)values, n_dummy, oi, ox, od, report);
}

template <typename IP, typename IX>
void launch_csr_v(int values_f64, int64_t n_rows, int64_t n_cols, int64_t nnz, const void *indptr,
                  const void *indices, const void *values, int n_dummy, int32_t *oi, int32_t *ox, double *od,
                  int64_t *report, cudaStream_t st) {
    if (values_f64)
        launch_csr<IP, IX, double>(n_rows, n_cols, nnz, indptr, indices, values, n_dummy, oi, ox, od, report, st);
    else
        launch_csr<IP, IX, float>(n_rows, n_cols, nnz, indptr, indices, values, n_dummy, oi, ox, od, report, st);
}

}  // namespace

extern "C" int sp_csr_prepare(int64_t n_rows, int64_t n_cols, int64_t nnz, const void *indptr, int indptr_i64,
                              const void *indices, int indices_i64, const void *values, int values_f64,
                              int64_t stride_row, int64_t stride_col, int n_dummy, int32_t *out_indptr,
                              int32_t *out_indices, double *out_data, int64_t *report, sp_stream stream) {
    const bool dense = indptr == nullptr;
    const int64_t stored = dense ? n_rows * n_cols : nnz;
    // (values / indices of an empty matrix may be NULL: torch gives an empty tensor no storage)
    if (!report || n_rows < 0 || n_cols < 0 || nnz < 0 || n_dummy < 0 || n_dummy > 32 ||
        (stored > 0 && !values) || (!dense && nnz > 0 && !indices)) {
        sp_set_error("sp_csr_prepare: invalid arguments");
        return SP_ERR_INVALID;
    }
    if ((out_indptr == nullptr) != (out_indices == nullptr) || (out_indices == nullptr) != (out_data == nullptr)) {
        sp_set_error("sp_csr_prepare: out_indptr, out_indices and out_data are given together or not at all");
        return SP_ERR_INVALID;
    }
    if (out_indices && stored + n_rows * (int64_t)n_dummy > INT32_MAX) {
        sp_set_error("sp_csr_prepare: %lld stored entries do not fit int32 indptr",
                     (long long)(stored + n_rows * (int64_t)n_dummy));
        return SP_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    report_init_kernel<<<1, 32, 0, st>>>(report);
    if (dense) {
        if (n_rows > 0) {
            const unsigned grid = (unsigned)((n_rows + kRowsPerBlock - 1) / kRowsPerBlock);
            if (values_f64)
                dense_prepare_kernel<double><<<grid, 32 * kRowsPerBlock, 0, st>>>(
                    n_rows, n_cols, (const double *)values, stride_row, stride_col, n_dummy, out_indptr, out_indices,
                    out_data, report);
            else
                dense_prepare_kernel<float><<<grid, 32 * kRowsPerBlock, 0, st>>>(
                    n_rows, n_cols, (const float *)values, stride_row, stride_col, n_dummy, out_indptr, out_indices,
                    out_data, report);
        } else if (out_indptr) {
            SP_CUDA(cudaMemsetAsync(out_indptr, 0, sizeof(int32_t), st));
        }
    } else if (indptr_i64 && indices_i64) {
        launch_csr_v<int64_t, int64_t>(values_f64, n_rows, n_cols, nnz, indptr, indices, values, n_dummy, out_indptr,
                                       out_indices, out_data, report, st);
    } else if (indptr_i64) {
        launch_csr_v<int64_t, int32_t>(values_f64, n_rows, n_cols, nnz, indptr, indices, values, n_dummy, out_indptr,
                                       out_indices, out_data, report, st);
    } else if (indices_i64) {
        launch_csr_v<int32_t, int64_t>(values_f64, n_rows, n_cols, nnz, indptr, indices, values, n_dummy, out_indptr,
                                       out_indices, out_data, report, st);
    } else {
        launch_csr_v<int32_t, int32_t>(values_f64, n_rows, n_cols, nnz, indptr, indices, values, n_dummy, out_indptr,
                                       out_indices, out_data, report, st);
    }
    SP_LAUNCH_CHECK("sp_csr_prepare");
    return SP_OK;
}

extern "C" int sp_csr_sum_runs(int64_t nnz, const int64_t *keys, const int64_t *perm, const double *data,
                               const int64_t *run_index, int64_t n_cols, int32_t *out_indices, double *out_data,
                               sp_stream stream) {
    if (nnz < 0 || n_cols < 1 || (nnz > 0 && (!keys || !perm || !data || !run_index || !out_indices || !out_data))) {
        sp_set_error("sp_csr_sum_runs: invalid arguments");
        return SP_ERR_INVALID;
    }
    if (nnz == 0) return SP_OK;
    const int threads = 256;
    sum_runs_kernel<<<(unsigned)((nnz + threads - 1) / threads), threads, 0, (cudaStream_t)stream>>>(
        nnz, keys, perm, data, run_index, n_cols, out_indices, out_data);
    SP_LAUNCH_CHECK("sp_csr_sum_runs");
    return SP_OK;
}
