// Row-wise (CSR) dynamic-programming kernels: ANOVA degree-m / all-subsets kernel values per
// (sample, component).  Replaces, on device:
//   * kernels.poly_predict / anova_kernel / _all_subsets_fast   (reference kernels.py:71-153)
//   * pcd._precompute_A_all_degree / pcd_all._precompute_A_all  (optimizer/pcd.py:15-30,
//     optimizer/pcd_all.py:8-18)  -- one component, written into the per-sample record array
//   * pbcd._precompute_A_all_degree / pbcd_all._precompute_A_all (optimizer/pbcd.py:18-33,
//     optimizer/pbcd_all.py:9-20) -- all components, written into A[n, m-1, k]
// The reference walks columns (CSC) and scatters into A; per sample that visits its features in
// ascending order, which is exactly the CSR row order used here, so every A[i,t] sees the same
// sequence of fp64 operations (bit-identical DP), while the loads are coalesced row streams.
#include "common.cuh"
#include "sparsepoly_b200.h"

namespace {

constexpr int ROWS_THREADS = 256;

// ---------------------------------------------------------------------------------------------
// all-components kernels: one group of G lanes per sample, lanes over components.
//   MODE 0 (rows_predict_kernel): out[i*out_stride] (+)= sum_j x w_j + sum_s lam_s * K_s(i)      (predict)
//   MODE 2 (rows_all_kernel): Aout[i, s] = K_s(i) (the Gram matrix of kernels.anova_kernel / all_subsets_kernel)
template <int DEG, int G>
__global__ void __launch_bounds__(ROWS_THREADS)
rows_all_kernel(int n, int k, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                const double *__restrict__ data, const double *__restrict__ P_dk, double *Aout) {
    constexpr int MODE = 2;
    constexpr bool PX = false;
    const double *__restrict__ lams = nullptr;
    const double *__restrict__ w = nullptr;
    double *out = nullptr;
    const int out_stride = 1, accumulate = 0;
#include "rows_all_body.inc"
}

// prediction of a table of models: block row y computes the model tab.m[y] {P_dk, lams, w, out}.  The table is a
// kernel parameter (no copy, no wait for one), so a single prediction is one launch as before.
struct PredictTable { sp_predict_model m[SP_PREDICT_MAX_MODELS]; };

template <int DEG, int G>
__global__ void __launch_bounds__(ROWS_THREADS)
rows_predict_kernel(int n, int k, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                    const double *__restrict__ data, const __grid_constant__ PredictTable tab, int out_stride,
                    int accumulate) {
    constexpr int MODE = 0;
    constexpr bool PX = false;
    const sp_predict_model &e = tab.m[blockIdx.y];
    const double *__restrict__ P_dk = e.P_dk;
    const double *__restrict__ lams = e.lams;
    const double *__restrict__ w = e.w;
    double *out = e.out, *Aout = nullptr;
#include "rows_all_body.inc"
}

// pbcd cache precompute (pbcd._precompute_A_all_degree / pbcd_all._precompute_A_all): block row y writes the cache
// of the entry table[y] {P_dk, A}: A[i, t-1, s] = A^t_s(i), t=1..DEG-1 (ANOVA) / A[i, s] = A_s(i) (all-subsets), with
// A += (A*p)*x (pcd.py:30, pbcd.py:33).  At three CTAs per SM ptxas spills in none of the instantiations (72..80
// registers); with the budget of rows_all_kernel it spills in 5 of the 15.
template <int DEG, int G>
__global__ void __launch_bounds__(ROWS_THREADS, 3)
rows_pbcd_cache_kernel(int n, int k, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                       const double *__restrict__ data, const SpBlockEntry *__restrict__ table) {
    constexpr int MODE = 1;
    constexpr bool PX = true;
    const SpBlockEntry e = table[blockIdx.y];
    const double *__restrict__ P_dk = e.P;
    const double *__restrict__ lams = nullptr;
    const double *__restrict__ w = nullptr;
    double *out = nullptr, *Aout = e.out;
    const int out_stride = 1, accumulate = 0;
#include "rows_all_body.inc"
}

// ---------------------------------------------------------------------------------------------
// pcd cache precompute (one component per entry): block row y computes the entry table[y] {p_s, rec}.  8 lanes per
// sample; lanes own nonzeros (coalesced idx/val load + parallel gather of p_s[j]); the recurrence itself is run
// redundantly by all lanes.  Writes rec[i*stride + 2 + (t-1)] = A^t(i), t=1..DEG-1 (ANOVA) or rec[i*stride+2] = A(i).
template <int DEG>
__global__ void __launch_bounds__(ROWS_THREADS)
rows_one_kernel(int n, const int32_t *__restrict__ indptr, const int32_t *__restrict__ indices,
                const double *__restrict__ data, const SpRowsEntry *__restrict__ table, int rec_stride) {
    const SpRowsEntry ent = table[blockIdx.y];
    const double *__restrict__ p_s = ent.p;
    double *rec = ent.rec;
    constexpr int G = 8;
    constexpr int ND = DEG > 0 ? DEG : 1;
    const int lane = threadIdx.x & (G - 1);
    const unsigned gmask = 0xffu << ((threadIdx.x & 31) & ~(G - 1));
    const int groups_per_block = ROWS_THREADS / G;
    const int group = blockIdx.x * groups_per_block + threadIdx.x / G;
    const int n_groups = gridDim.x * groups_per_block;
    for (int i = group; i < n; i += n_groups) {
        const int st = indptr[i], en = indptr[i + 1];
        double A[ND + 1];
        A[0] = 1.0;
#pragma unroll
        for (int t = 1; t <= ND; t++) A[t] = (DEG > 0) ? 0.0 : 1.0;
        for (int base = st; base < en; base += G) {
            const int e = base + lane;
            double pl = 0.0, xl = 0.0;
            if (e < en) { xl = data[e]; pl = p_s[indices[e]]; }
            const int cnt = min(G, en - base);
#pragma unroll
            for (int q = 0; q < G; q++) {
                const double p = __shfl_sync(gmask, pl, q, G);
                const double x = __shfl_sync(gmask, xl, q, G);
                if (q < cnt) {
                    if (DEG > 0) {
#pragma unroll
                        for (int t = 0; t < ND; t++) A[ND - t] += (A[ND - t - 1] * p) * x;  // pcd.py:30
                    } else {
                        A[1] *= 1.0 + p * x;                                               // pcd_all.py:18
                    }
                }
            }
        }
        if (lane == 0) {
            double *r = rec + (size_t)i * rec_stride + 2;
            if (DEG > 0) {
#pragma unroll
                for (int t = 1; t < ND; t++) r[t - 1] = A[t];
            } else {
                r[0] = A[1];
            }
        }
    }
}

int grid_for(int n, int per_block) {
    long long blocks = ((long long)n + per_block - 1) / per_block;
    const long long cap = 148LL * 8 * 4;   // a few waves of 8 resident CTAs per SM
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

template <int DEG>
int launch_kernel_matrix(int n, int k, const sp_dataset *ds, const double *P_dk, double *K, cudaStream_t st) {
    sp_prof_begin(SP_PROF_ROWS, st);
    if (k <= 8) {
        rows_all_kernel<DEG, 8><<<grid_for(n, ROWS_THREADS / 8), ROWS_THREADS, 0, st>>>(
            n, k, ds->csr_indptr, ds->csr_indices, ds->csr_data, P_dk, K);
    } else if (k <= 16) {
        rows_all_kernel<DEG, 16><<<grid_for(n, ROWS_THREADS / 16), ROWS_THREADS, 0, st>>>(
            n, k, ds->csr_indptr, ds->csr_indices, ds->csr_data, P_dk, K);
    } else {
        rows_all_kernel<DEG, 32><<<grid_for(n, ROWS_THREADS / 32), ROWS_THREADS, 0, st>>>(
            n, k, ds->csr_indptr, ds->csr_indices, ds->csr_data, P_dk, K);
    }
    sp_prof_end(st);
    SP_LAUNCH_CHECK("rows_all_kernel");
    return SP_OK;
}

// the predictions of n_tab models in one launch, with the group width launch_kernel_matrix picks for k
template <int DEG>
int launch_predict(int n, int k, const sp_dataset *ds, const PredictTable &tab, int n_tab, int out_stride,
                   int accumulate, cudaStream_t st) {
    sp_prof_begin(SP_PROF_ROWS, st);
    if (k <= 8) {
        rows_predict_kernel<DEG, 8><<<dim3(grid_for(n, ROWS_THREADS / 8), n_tab), ROWS_THREADS, 0, st>>>(
            n, k, ds->csr_indptr, ds->csr_indices, ds->csr_data, tab, out_stride, accumulate);
    } else if (k <= 16) {
        rows_predict_kernel<DEG, 16><<<dim3(grid_for(n, ROWS_THREADS / 16), n_tab), ROWS_THREADS, 0, st>>>(
            n, k, ds->csr_indptr, ds->csr_indices, ds->csr_data, tab, out_stride, accumulate);
    } else {
        rows_predict_kernel<DEG, 32><<<dim3(grid_for(n, ROWS_THREADS / 32), n_tab), ROWS_THREADS, 0, st>>>(
            n, k, ds->csr_indptr, ds->csr_indices, ds->csr_data, tab, out_stride, accumulate);
    }
    sp_prof_end(st);
    SP_LAUNCH_CHECK("rows_predict_kernel");
    return SP_OK;
}

// the pbcd cache of n_tab entries {P_dk, A} in one launch, with the group width launch_all picks for k
template <int DEG>
void launch_pbcd_cache(int n, int k, const sp_dataset *ds, const SpBlockEntry *table, int n_tab, cudaStream_t st) {
    if (k <= 8) {
        rows_pbcd_cache_kernel<DEG, 8><<<dim3(grid_for(n, ROWS_THREADS / 8), n_tab), ROWS_THREADS, 0, st>>>(
            n, k, ds->csr_indptr, ds->csr_indices, ds->csr_data, table);
    } else if (k <= 16) {
        rows_pbcd_cache_kernel<DEG, 16><<<dim3(grid_for(n, ROWS_THREADS / 16), n_tab), ROWS_THREADS, 0, st>>>(
            n, k, ds->csr_indptr, ds->csr_indices, ds->csr_data, table);
    } else {
        rows_pbcd_cache_kernel<DEG, 32><<<dim3(grid_for(n, ROWS_THREADS / 32), n_tab), ROWS_THREADS, 0, st>>>(
            n, k, ds->csr_indptr, ds->csr_indices, ds->csr_data, table);
    }
}

}  // namespace

extern "C" int sp_predict_multi(const sp_dataset *ds, const sp_predict_model *models, int n_models, int k,
                                int degree, int out_stride, int accumulate, sp_stream stream) {
    if (!ds || !ds->csr_indptr || !models || n_models < 0 || n_models > SP_PREDICT_MAX_MODELS || k <= 0 ||
        out_stride <= 0) {
        sp_set_error("sp_predict: invalid argument");
        return SP_ERR_INVALID;
    }
    PredictTable tab;
    for (int b = 0; b < n_models; b++) {
        if (!models[b].P_dk || !models[b].lams || !models[b].out) {
            sp_set_error("sp_predict: invalid argument (model %d)", b);
            return SP_ERR_INVALID;
        }
        tab.m[b] = models[b];
    }
    const int n = ds->n_samples;
    if (n == 0 || n_models == 0) return SP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    switch (degree) {
    case -1: return launch_predict<-1>(n, k, ds, tab, n_models, out_stride, accumulate, st);
    case 1: return launch_predict<1>(n, k, ds, tab, n_models, out_stride, accumulate, st);
    case 2: return launch_predict<2>(n, k, ds, tab, n_models, out_stride, accumulate, st);
    case 3: return launch_predict<3>(n, k, ds, tab, n_models, out_stride, accumulate, st);
    case 4: return launch_predict<4>(n, k, ds, tab, n_models, out_stride, accumulate, st);
    case 5: return launch_predict<5>(n, k, ds, tab, n_models, out_stride, accumulate, st);
    default:
        sp_set_error("degree %d is not supported (1..%d or -1 for all-subsets)", degree, SP_MAXDEG);
        return SP_ERR_UNSUPPORTED;
    }
}

extern "C" int sp_predict(const sp_dataset *ds, const double *P_dk, int k, const double *lams,
                          int degree, const double *w, double *out, int out_stride, int accumulate,
                          sp_stream stream) {
    const sp_predict_model m = {P_dk, lams, w, out};
    return sp_predict_multi(ds, &m, 1, k, degree, out_stride, accumulate, stream);
}

extern "C" int sp_kernel_matrix(const sp_dataset *ds, const double *P_dk, int k, int degree, double *K,
                                sp_stream stream) {
    if (!ds || !ds->csr_indptr || !P_dk || !K || k <= 0) {
        sp_set_error("sp_kernel_matrix: invalid argument");
        return SP_ERR_INVALID;
    }
    const int n = ds->n_samples;
    if (n == 0) return SP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    switch (degree) {
    case -1: return launch_kernel_matrix<-1>(n, k, ds, P_dk, K, st);
    case 1: return launch_kernel_matrix<1>(n, k, ds, P_dk, K, st);
    case 2: return launch_kernel_matrix<2>(n, k, ds, P_dk, K, st);
    case 3: return launch_kernel_matrix<3>(n, k, ds, P_dk, K, st);
    case 4: return launch_kernel_matrix<4>(n, k, ds, P_dk, K, st);
    case 5: return launch_kernel_matrix<5>(n, k, ds, P_dk, K, st);
    default:
        sp_set_error("degree %d is not supported (1..%d or -1 for all-subsets)", degree, SP_MAXDEG);
        return SP_ERR_UNSUPPORTED;
    }
}

// pbcd cache precompute of n_tab models in one launch: entry y is {P_dk, A} of one model, A [n, m-1, k] (ANOVA)
// or [n, k] (all-subsets)
int sp_rows_precompute_all_multi(const sp_dataset *ds, const SpBlockEntry *table, int n_tab, int k, int degree,
                                 cudaStream_t st) {
    const int n = ds->n_samples;
    if (n == 0 || n_tab == 0) return SP_OK;
    sp_prof_begin(SP_PROF_ROWS, st);
    switch (degree) {
    case -1: launch_pbcd_cache<-1>(n, k, ds, table, n_tab, st); break;
    case 2: launch_pbcd_cache<2>(n, k, ds, table, n_tab, st); break;
    case 3: launch_pbcd_cache<3>(n, k, ds, table, n_tab, st); break;
    case 4: launch_pbcd_cache<4>(n, k, ds, table, n_tab, st); break;
    case 5: launch_pbcd_cache<5>(n, k, ds, table, n_tab, st); break;
    default:
        sp_set_error("pbcd degree %d is not supported (2..%d or -1)", degree, SP_MAXDEG);
        return SP_ERR_UNSUPPORTED;
    }
    sp_prof_end(st);
    SP_LAUNCH_CHECK("rows_pbcd_cache_kernel");
    return SP_OK;
}

// pcd cache precompute of n_tab (model, component) entries in one launch, into each entry's record array
int sp_rows_precompute_multi(const sp_dataset *ds, const SpRowsEntry *table, int n_tab, int degree, int rec_stride,
                             cudaStream_t st) {
    const int n = ds->n_samples;
    if (n == 0 || n_tab == 0) return SP_OK;
    const dim3 grid((unsigned)grid_for(n, ROWS_THREADS / 8), (unsigned)n_tab);
#define SP_ONE(D)                                                                                    \
    rows_one_kernel<D><<<grid, ROWS_THREADS, 0, st>>>(n, ds->csr_indptr, ds->csr_indices,            \
                                                      ds->csr_data, table, rec_stride)
    sp_prof_begin(SP_PROF_ROWS, st);
    switch (degree) {
    case -1: SP_ONE(-1); break;
    case 2: SP_ONE(2); break;
    case 3: SP_ONE(3); break;
    case 4: SP_ONE(4); break;
    case 5: SP_ONE(5); break;
    default:
        sp_set_error("pcd degree %d is not supported (2..%d or -1)", degree, SP_MAXDEG);
        return SP_ERR_UNSUPPORTED;
    }
#undef SP_ONE
    sp_prof_end(st);
    SP_LAUNCH_CHECK("rows_one_kernel");
    return SP_OK;
}
