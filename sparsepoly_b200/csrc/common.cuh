// Shared device helpers for the sparsepoly B200 backend (sm_100a only).
// All arithmetic is IEEE fp64 and the whole library is compiled with -fmad=false so that
// a*b+c is never contracted (numba, which JIT-compiles the reference, does not contract).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#define SP_MAXDEG 5           // highest ANOVA degree with a compiled sweep kernel
#define SP_FLAG_BIT 0x80000000u    // sample also occurs at position t-1
#define SP_FLAG2_BIT 0x40000000u   // sample also occurs at position t-2
#define SP_ROW_MASK 0x3fffffff

enum { SP_LOSS_SQUARED = 0, SP_LOSS_LOGISTIC = 1, SP_LOSS_SQHINGE = 2 };
enum { SP_REG_L1 = 0, SP_REG_L21 = 1, SP_REG_SQL12 = 2, SP_REG_SQL21 = 3, SP_REG_OMEGATI = 4,
       SP_REG_OMEGACS = 5 };

enum { SP_OK = 0, SP_ERR_INVALID = 1, SP_ERR_UNSUPPORTED = 2, SP_ERR_CUDA = 3 };

// kernel classes for sp_profile_* (see errors.cu)
enum { SP_PROF_ROWS = 0, SP_PROF_REGCACHE = 1, SP_PROF_SWEEP_PCD = 2, SP_PROF_SWEEP_PBCD = 3,
       SP_PROF_PSGD_GRAD = 4, SP_PROF_PSGD_STEP = 5, SP_PROF_PROX = 6, SP_PROF_PLAN = 7,
       SP_PROF_CLASSES = 8 };
void sp_prof_begin(int cls, cudaStream_t st);
void sp_prof_end(cudaStream_t st);

// table entries of the pcd / pbcd launches (a single fit is a table of one model): one component row of one model
// with its sample records (rows.cu), or a vector with the regularizer scratch and cache mode computed from it
// (regcache.cu)
struct SpRowsEntry { const double *p; double *rec; };
struct SpRegEntry { const double *p; double *regstate; int mode; };
// pbcd: one model's feature-major P_dk [d,k] and what is computed from it (the row-DP cache A in rows.cu, the row
// norms in pbcd.cu)
struct SpBlockEntry { const double *P; double *out; };

// pinned host staging of the argument tables (pcd.cu): acquire waits until the copy that last read the buffer has
// completed; upload copies its first `bytes` to the device and records that copy
int sp_stage_acquire(size_t bytes, unsigned char **out);
int sp_stage_upload(void *dst, size_t bytes, cudaStream_t st);

void sp_set_error(const char *fmt, ...);
int sp_check_cuda(cudaError_t e, const char *what);

#define SP_CUDA(expr)                                            \
    do {                                                         \
        int _rc = sp_check_cuda((expr), #expr);                  \
        if (_rc != SP_OK) return _rc;                            \
    } while (0)
#define SP_LAUNCH_CHECK(name)                                    \
    do {                                                         \
        int _rc = sp_check_cuda(cudaGetLastError(), name);       \
        if (_rc != SP_OK) return _rc;                            \
    } while (0)

// ---------------------------------------------------------------- losses (reference loss.py:13-71)
template <int LOSS> __device__ __forceinline__ double sp_mu() {
    return LOSS == SP_LOSS_SQUARED ? 1.0 : (LOSS == SP_LOSS_LOGISTIC ? 0.25 : 2.0);
}

template <int LOSS> __device__ __forceinline__ double sp_dloss(double p, double y) {
    if (LOSS == SP_LOSS_SQUARED) {
        return p - y;                                   // loss.py:22-23
    } else if (LOSS == SP_LOSS_LOGISTIC) {              // loss.py:43-51
        double z = p * y;
        if (z > 18.0) return -y * exp(-z);
        if (z < -18.0) return -y;
        return -y / (exp(z) + 1.0);
    } else {                                            // loss.py:67-71
        double z = 1.0 - p * y;
        if (z > 0.0) return (-2.0 * y) * z;
        return 0.0;
    }
}

template <int LOSS> __device__ __forceinline__ double sp_loss(double p, double y) {
    if (LOSS == SP_LOSS_SQUARED) {                      // loss.py:19-20
        double r = p - y;
        return 0.5 * (r * r);
    } else if (LOSS == SP_LOSS_LOGISTIC) {              // loss.py:34-41
        double z = p * y;
        if (z > 18.0) return exp(-z);
        if (z < -18.0) return -z;
        return log(1.0 + exp(-z));
    } else {                                            // loss.py:61-65
        double z = 1.0 - p * y;
        if (z > 0.0) return z * z;
        return 0.0;
    }
}

__device__ __forceinline__ double sp_dloss_rt(int loss, double p, double y) {
    return loss == SP_LOSS_SQUARED ? sp_dloss<SP_LOSS_SQUARED>(p, y)
         : loss == SP_LOSS_LOGISTIC ? sp_dloss<SP_LOSS_LOGISTIC>(p, y)
                                    : sp_dloss<SP_LOSS_SQHINGE>(p, y);
}
__device__ __forceinline__ double sp_loss_rt(int loss, double p, double y) {
    return loss == SP_LOSS_SQUARED ? sp_loss<SP_LOSS_SQUARED>(p, y)
         : loss == SP_LOSS_LOGISTIC ? sp_loss<SP_LOSS_LOGISTIC>(p, y)
                                    : sp_loss<SP_LOSS_SQHINGE>(p, y);
}
__host__ __device__ __forceinline__ double sp_mu_rt(int loss) {
    return loss == SP_LOSS_SQUARED ? 1.0 : (loss == SP_LOSS_LOGISTIC ? 0.25 : 2.0);
}

__device__ __forceinline__ double sp_np_sign(double x) {      // np.sign
    return (double)((x > 0.0) - (x < 0.0));
}
// sign(x) * max(|x| - t, 0)  (regularizer/utils.py:7-9, l1.py:32-33)
__device__ __forceinline__ double sp_soft_threshold(double x, double t) {
    double m = fabs(x) - t;
    if (!(m > 0.0)) m = 0.0;
    return sp_np_sign(x) * m;
}

// ---------------------------------------------------------------- warp helpers
__device__ __forceinline__ double sp_shfl_xor(double v, int m) {
    return __shfl_xor_sync(0xffffffffu, v, m);
}
__device__ __forceinline__ double sp_shfl(double v, int src) {
    return __shfl_sync(0xffffffffu, v, src);
}
// butterfly all-reduce: every lane ends with the same sum (fixed order -> deterministic)
__device__ __forceinline__ double sp_warp_allsum(double v) {
#pragma unroll
    for (int m = 16; m > 0; m >>= 1) v += sp_shfl_xor(v, m);
    return v;
}
