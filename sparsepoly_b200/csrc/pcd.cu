// Sequential coordinate sweeps on ONE thread-block cluster (sm_100a):
//   * cd_linear._cd_linear_epoch                     (reference optimizer/cd_linear.py:8-33)
//   * pcd.pcd_epoch  (_update + synchronize loop)    (reference optimizer/pcd.py:33-137)
//   * pcd_all.pcd_epoch                              (reference optimizer/pcd_all.py:21-102)
//
// Design (DESIGN.md 3.2).  Coordinate order is a true dependency chain, so a sweep is bound by the
// latency of one coordinate step, not by bandwidth.  One cluster of C CTAs walks the d coordinates
// of one component in order:
//   * samples are range-partitioned over the CTAs, so a sample's record {y_pred, y, A^1..A^{m-1}}
//     is only ever touched by one SM; the only inter-SM traffic is the all-to-all exchange of the
//     per-warp partial sums (g, h) through distributed shared memory (st.async + mbarrier
//     complete_tx, 4-deep mailboxes);
//   * warps are specialised: W gather warps (stage, gradient terms, push, write-back) and one
//     scalar-chain warp per CTA that sums the partials and runs the ~20-flop chain (step, prox_cd,
//     regularizer cache) redundantly in every CTA, handing (upd, p_new) back through shared memory;
//   * column slices and records of the coming positions are staged through shared memory with
//     cp.async (no scoreboard coupling with the step's own loads); the per-position table lives in
//     registers, 32 positions per warp, broadcast by shuffles;
//   * the partial sums of position t+1 are computed and pushed BEFORE the scalar chain of position
//     t whenever the plan marks the two columns sample-disjoint (pos_conf == 0), which hides the
//     DSMEM hop behind the scalar chain; otherwise they are recomputed after the write-back;
//   * records the previous two positions may still be rewriting are tagged by the plan (bits
//     31/30 of flag_idx) and re-read from global memory after the barrier.
#include <string.h>

#include <vector>

#include "common.cuh"
#include "cluster.cuh"
#include "pcd_common.cuh"
#include "sparsepoly_b200.h"

int sp_rows_precompute_one(const sp_dataset *ds, const double *p_s, int degree, double *rec,
                           int rec_stride, cudaStream_t st);
int sp_launch_reg_cache(int mode, int degree, int d, const double *v, double *regstate, cudaStream_t st);
int sp_rows_precompute_multi(const sp_dataset *ds, const SpRowsEntry *table, int n_tab, int degree, int rec_stride,
                             cudaStream_t st);
int sp_launch_reg_cache_multi(const SpRegEntry *table, int n_tab, int degree, int d, cudaStream_t st);
int sp_wsweep(const sp_dataset *ds, const sp_wplan *wp, const int32_t *idx_feat, int degree, double *prow,
              const double *cns, const double *lam_ptr, double ab, double gamma, double eta, int reg,
              int loss, double *rec, int rec_stride, double *regstate, double *viol, cudaStream_t st);

namespace {

constexpr int SWEEP_MAX_THREADS = 256;
constexpr int SWEEP_MAX_CTAS = 16;
constexpr int MBOX_DEPTH = 4;

struct SweepArgs {
    int d, C;
    const int32_t *pos_ptr;    // [d*(C+1)]
    const int32_t *flag_idx;   // [nnz]
    const double *data;        // [nnz] CSC values
    const int32_t *idx_feat;   // [d]
    const int32_t *pos_conf;   // [d]
    double *prow;              // P[s, :] (or w)
    const double *cns;         // col_norm_sq (linear only)
    const double *lam_ptr;     // &lams[s] (FM / all-subsets)
    double ab;                 // alpha (linear) or beta
    double gamma, eta;
    int reg;
    double *rec;
    int stride;
    double *regstate;          // in/out regularizer scalars
    double *viol;              // in/out running sum of |updates|
};

__device__ __forceinline__ void cp_async4(void *smem, const void *g) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(smem)), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async8(void *smem, const void *g) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(smem)), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async16(void *smem, const void *g) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(g) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// 32 positions of the per-position table, one per lane
struct MetaChunk {
    int s, e, jf;        // slice [s,e) of this CTA, feature id | conflict << 31
    double pold, cn;     // P[s_comp, j] (or w_j), col_norm_sq[j]
};

__device__ __forceinline__ void meta_load_ptr(MetaChunk &m, const SweepArgs &a, int base, int c, int lane) {
    const int q = base + lane;
    m.s = 0; m.e = 0; m.jf = 0;
    if (q < a.d) {
        m.s = a.pos_ptr[(size_t)q * (a.C + 1) + c];
        m.e = a.pos_ptr[(size_t)q * (a.C + 1) + c + 1];
        m.jf = a.idx_feat[q] | (a.pos_conf[q] ? (int)SP_FLAG_BIT : 0);
    }
}
template <int KIND>
__device__ __forceinline__ void meta_load_val(MetaChunk &m, const SweepArgs &a, int base, int lane) {
    m.pold = 0.0; m.cn = 0.0;
    if (base + lane < a.d) {
        const int j = m.jf & 0x7fffffff;
        m.pold = a.prow[j];
        if (KIND == KIND_LINEAR) m.cn = a.cns[j];
    }
}


template <int KIND, int DEG, int LOSS, int NZ>
__global__ void __launch_bounds__(SWEEP_MAX_THREADS + 32) sweep_kernel(const SweepArgs a) {
#include "sweep_body.inc"
}

// Many models per launch (sp_pcd_epoch_multi / sp_cd_linear_epoch_multi): clusters along x, cluster b
// runs the sweep of table[b] exactly as sweep_kernel runs its argument.
template <int KIND, int DEG, int LOSS, int NZ>
__global__ void __launch_bounds__(SWEEP_MAX_THREADS + 32) sweep_multi_kernel(const SweepArgs *__restrict__ table,
                                                                             int width) {
    const SweepArgs &a = table[blockIdx.x / width];   // read in place: no register copy of the entry
#include "sweep_body.inc"
}

// table == nullptr: one cluster runs `a`.  Otherwise n_tab clusters run the device table (its host copy
// starts with `a`, and every entry has the width a.C).
template <int KIND, int DEG, int LOSS, int NZ>
int launch_sweep(const SweepArgs &a, const SweepArgs *table, int n_tab, int threads, cudaStream_t st) {
    constexpr int NA = (KIND == KIND_FM) ? DEG - 1 : (KIND == KIND_ALL ? 1 : 0);
    constexpr int NCH = (2 + NA + 1) / 2;
    const int W = threads / 32;
    const size_t smem = (size_t)2 * NZ * NCH * threads * 16 + (size_t)3 * NZ * threads * 8 +
                        (size_t)MBOX_DEPTH * a.C * W * 16 + (size_t)3 * NZ * threads * 4;
    auto set_attrs = [&](auto kern) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return sp_check_cuda(e, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize)");
        if (a.C > 8) {
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e != cudaSuccess) return sp_check_cuda(e, "cudaFuncSetAttribute(NonPortableClusterSizeAllowed)");
        }
        return (int)SP_OK;
    };
    int rc = table ? set_attrs(sweep_multi_kernel<KIND, DEG, LOSS, NZ>) : set_attrs(sweep_kernel<KIND, DEG, LOSS, NZ>);
    if (rc) return rc;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)a.C * (unsigned)(table ? n_tab : 1), 1, 1);
    cfg.blockDim = dim3((unsigned)threads + 32, 1, 1);      // gather warps + the scalar-chain warp
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)a.C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    sp_prof_begin(SP_PROF_SWEEP_PCD, st);
    cudaError_t le = table ? cudaLaunchKernelEx(&cfg, sweep_multi_kernel<KIND, DEG, LOSS, NZ>, table, a.C)
                           : cudaLaunchKernelEx(&cfg, sweep_kernel<KIND, DEG, LOSS, NZ>, a);
    sp_prof_end(st);
    return sp_check_cuda(le, table ? "sweep_multi_kernel launch" : "sweep_kernel launch");
}

template <int KIND, int DEG>
int dispatch_loss(int loss, const SweepArgs &a, const SweepArgs *table, int n_tab, int threads, int nz,
                  cudaStream_t st) {
#define SP_DISPATCH_NZ(L)                                                                    \
    return nz >= 2 ? launch_sweep<KIND, DEG, L, 2>(a, table, n_tab, threads, st)             \
                   : launch_sweep<KIND, DEG, L, 1>(a, table, n_tab, threads, st)
    switch (loss) {
    case SP_LOSS_SQUARED: SP_DISPATCH_NZ(SP_LOSS_SQUARED);
    case SP_LOSS_LOGISTIC: SP_DISPATCH_NZ(SP_LOSS_LOGISTIC);
    case SP_LOSS_SQHINGE: SP_DISPATCH_NZ(SP_LOSS_SQHINGE);
    default: sp_set_error("unknown loss id %d", loss); return SP_ERR_INVALID;
    }
#undef SP_DISPATCH_NZ
}

int dispatch_degree(int degree, int loss, const SweepArgs &a, const SweepArgs *table, int n_tab, int threads, int nz,
                    cudaStream_t st) {
    switch (degree) {
    case -1: return dispatch_loss<KIND_ALL, 1>(loss, a, table, n_tab, threads, nz, st);
    case 2: return dispatch_loss<KIND_FM, 2>(loss, a, table, n_tab, threads, nz, st);
    case 3: return dispatch_loss<KIND_FM, 3>(loss, a, table, n_tab, threads, nz, st);
    case 4: return dispatch_loss<KIND_FM, 4>(loss, a, table, n_tab, threads, nz, st);
    case 5: return dispatch_loss<KIND_FM, 5>(loss, a, table, n_tab, threads, nz, st);
    default: sp_set_error("pcd degree %d is not supported by the CUDA backend (2..%d or -1)", degree, SP_MAXDEG);
             return SP_ERR_UNSUPPORTED;
    }
}

int check_plan(const sp_dataset *ds, const sp_plan *plan, const char *who) {
    if (ds && plan && plan->win) {                      // window sweep: only the order is needed
        if (!ds->csc_data || !ds->csc_indptr || !plan->idx_feat) {
            sp_set_error("%s: dataset/plan pointers missing", who);
            return SP_ERR_INVALID;
        }
        return SP_OK;
    }
    if (!ds || !plan || !ds->csc_data || !plan->pos_ptr || !plan->flag_idx || !plan->idx_feat ||
        !plan->pos_conf) {
        sp_set_error("%s: dataset/plan pointers missing", who);
        return SP_ERR_INVALID;
    }
    if (plan->n_cta < 1 || plan->n_cta > SWEEP_MAX_CTAS || (plan->n_cta & (plan->n_cta - 1))) {
        sp_set_error("%s: plan.n_cta must be a power of two in 1..%d", who, SWEEP_MAX_CTAS);
        return SP_ERR_INVALID;
    }
    if (plan->threads < 32 || plan->threads > SWEEP_MAX_THREADS || plan->threads % 32) {
        sp_set_error("%s: plan.threads must be a multiple of 32 in 32..%d", who, SWEEP_MAX_THREADS);
        return SP_ERR_INVALID;
    }
    return SP_OK;
}

// nonzeros per thread staged through shared memory: 2 when the mean slice exceeds the CTA
int pick_nz(const sp_dataset *ds, const sp_plan *plan) {
    const double avg = (double)ds->nnz / (ds->n_features > 0 ? ds->n_features : 1);
    return (avg / plan->n_cta > 0.8 * plan->threads) ? 2 : 1;
}

}  // namespace

int sp_min_rec_stride(int degree) {   // record = {y_pred, y, A^1..A^{m-1}}, multiple of 4 doubles
    const int r = (degree == -1) ? 3 : (degree < 1 ? 2 : degree + 1);
    return (r + 3) & ~3;
}

extern "C" int sp_rec_stride(int degree) { return sp_min_rec_stride(degree); }

extern "C" int sp_cd_linear_epoch(const sp_dataset *ds, const sp_plan *plan, double *w,
                                  const double *col_norm_sq, double alpha, int loss, double *rec,
                                  int rec_stride, double *viol, sp_stream stream) {
    int rc = check_plan(ds, plan, "sp_cd_linear_epoch");
    if (rc) return rc;
    if (!w || !col_norm_sq || !rec || !viol || rec_stride < 2 || (rec_stride & 1)) {
        sp_set_error("sp_cd_linear_epoch: invalid argument");
        return SP_ERR_INVALID;
    }
    if (ds->n_features == 0) return SP_OK;
    if (plan->win)
        return sp_wsweep(ds, plan->win, plan->idx_feat, 1, w, col_norm_sq, nullptr, alpha, 0.0, 1.0, SP_REG_L1,
                         loss, rec, rec_stride, viol, viol, (cudaStream_t)stream);
    SweepArgs a = {};
    a.d = ds->n_features; a.C = plan->n_cta;
    a.pos_ptr = plan->pos_ptr; a.flag_idx = plan->flag_idx; a.data = ds->csc_data;
    a.idx_feat = plan->idx_feat; a.pos_conf = plan->pos_conf;
    a.prow = w; a.cns = col_norm_sq; a.lam_ptr = nullptr; a.ab = alpha; a.gamma = 0.0; a.eta = 1.0;
    a.reg = SP_REG_L1; a.rec = rec; a.stride = rec_stride; a.regstate = viol; a.viol = viol;
    return dispatch_loss<KIND_LINEAR, 1>(loss, a, nullptr, 0, plan->threads, pick_nz(ds, plan), (cudaStream_t)stream);
}

// *flag = 1 when row[0..d) has a nonzero entry (one block)
__device__ __forceinline__ void row_any_nonzero(const double *__restrict__ row, int d, int *flag) {
    __shared__ int s_any;
    if (threadIdx.x == 0) s_any = 0;
    __syncthreads();
    int any = 0;
    for (int j = threadIdx.x; j < d; j += blockDim.x) any |= (row[j] != 0.0);
    if (any) s_any = 1;
    __syncthreads();
    if (threadIdx.x == 0) *flag = s_any;
}

// flags[s] = 1 when row s of P [k,d] has a nonzero entry
__global__ void row_any_nonzero_kernel(const double *__restrict__ P, int d, int *flags) {
    row_any_nonzero(P + (size_t)blockIdx.x * d, d, flags + blockIdx.x);
}

// flags[b*k + s] = 1 when row s of the [k,d] matrix Ps[b] has a nonzero entry (grid k x models)
__global__ void row_any_nonzero_multi_kernel(const double *const *__restrict__ Ps, int d, int k, int *flags) {
    row_any_nonzero(Ps[blockIdx.y] + (size_t)blockIdx.x * d, d, flags + (size_t)blockIdx.y * k + blockIdx.x);
}

extern "C" int sp_pcd_epoch(const sp_dataset *ds, const sp_plan *plan, double *P_kd, int k,
                            const double *lams, int degree, double beta, double gamma, double eta,
                            int reg, int loss, double *rec, int rec_stride, double *regstate,
                            double *viol, const int32_t *idx_comp_host, sp_stream stream) {
    int rc = check_plan(ds, plan, "sp_pcd_epoch");
    if (rc) return rc;
    if (!P_kd || !lams || !rec || !regstate || !viol || !idx_comp_host || k <= 0 || !ds->csr_indptr) {
        sp_set_error("sp_pcd_epoch: invalid argument");
        return SP_ERR_INVALID;
    }
    // solver x regularizer x degree support matrix (reference README.md:25-31; the reference
    // fails with a numba TypingError / ValueError inside the jitclass for the others)
    if (reg != SP_REG_L1 && reg != SP_REG_SQL12 && reg != SP_REG_OMEGATI) {
        sp_set_error("regularizer id %d does not implement the pcd protocol (use l1, squaredl12 or omegati)", reg);
        return SP_ERR_UNSUPPORTED;
    }
    if (reg == SP_REG_SQL12 && degree != 2) {
        sp_set_error(degree == -1 ? "squaredl12 is not available for all-subsets models"
                                  : "SquaredL12 supports only degree=2.");
        return SP_ERR_UNSUPPORTED;
    }
    if (!(degree == -1 || (degree >= 2 && degree <= SP_MAXDEG))) {
        sp_set_error("pcd degree %d is not supported by the CUDA backend (2..%d or -1)", degree, SP_MAXDEG);
        return SP_ERR_UNSUPPORTED;
    }
    if (rec_stride < sp_min_rec_stride(degree) || (rec_stride & 1)) {
        sp_set_error("sp_pcd_epoch: rec_stride %d too small for degree %d", rec_stride, degree);
        return SP_ERR_INVALID;
    }
    const int d = ds->n_features;
    if (d == 0) return SP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const int nz = plan->win ? 1 : pick_nz(ds, plan);
    // Dead components (ANOVA, degree >= 2, beta > 0): when row P[s,:] is entirely zero, A^t_i = 0 for every
    // t >= 1, so dA[m-1] = x (A^{m-1} - p dA[m-2]) = 0 on every nonzero, g = h = 0, the step is
    // (lams*0 + beta*0) / beta = 0 and the prox of 0 is 0 for l1 / squaredl12 / omegati: the reference's sweep
    // over that component (pcd.py:33-68, :92-135) changes nothing and adds 0 to the violation.  It is skipped
    // exactly; with beta == 0 the reference divides 0/0, so there the sweep runs as usual.  One small
    // reduction + ONE stream synchronisation per call (the only one this library makes inside an epoch).
    std::vector<int> alive(k, 1);
    if (degree >= 2 && beta > 0.0) {
        int *flags = nullptr;
        SP_CUDA(cudaMallocAsync((void **)&flags, sizeof(int) * k, st));
        row_any_nonzero_kernel<<<k, 256, 0, st>>>(P_kd, d, flags);
        cudaError_t e1 = cudaGetLastError();
        if (e1 == cudaSuccess) e1 = cudaMemcpyAsync(alive.data(), flags, sizeof(int) * k, cudaMemcpyDeviceToHost, st);
        if (e1 == cudaSuccess) e1 = cudaStreamSynchronize(st);
        cudaFreeAsync(flags, st);
        if (e1 != cudaSuccess) return sp_check_cuda(e1, "sp_pcd_epoch: dead-component scan");
    }
    for (int ss = 0; ss < k; ss++) {
        const int s = idx_comp_host[ss];
        if (s < 0 || s >= k) { sp_set_error("sp_pcd_epoch: bad component index %d", s); return SP_ERR_INVALID; }
        if (!alive[s]) continue;
        double *prow = P_kd + (size_t)s * d;
        rc = sp_rows_precompute_one(ds, prow, degree, rec, rec_stride, st);      // pcd.py:94 / pcd_all.py:65
        if (rc) return rc;
        if (reg != SP_REG_L1) {                                                   // pcd.py:96
            const int mode = (reg == SP_REG_SQL12) ? 0 : (degree == -1 ? 2 : 1);
            rc = sp_launch_reg_cache(mode, degree, d, prow, regstate, st);
            if (rc) return rc;
        }
        if (plan->win) {
            rc = sp_wsweep(ds, plan->win, plan->idx_feat, degree, prow, nullptr, lams + s, beta, gamma, eta, reg,
                           loss, rec, rec_stride, regstate, viol, st);
            if (rc) return rc;
            continue;
        }
        SweepArgs a = {};
        a.d = d; a.C = plan->n_cta;
        a.pos_ptr = plan->pos_ptr; a.flag_idx = plan->flag_idx; a.data = ds->csc_data;
        a.idx_feat = plan->idx_feat; a.pos_conf = plan->pos_conf;
        a.prow = prow; a.cns = nullptr; a.lam_ptr = lams + s; a.ab = beta; a.gamma = gamma; a.eta = eta;
        a.reg = reg; a.rec = rec; a.stride = rec_stride; a.regstate = regstate; a.viol = viol;
        rc = dispatch_degree(degree, loss, a, nullptr, 0, plan->threads, nz, st);
        if (rc) return rc;
    }
    return SP_OK;
}

// ------------------------------------------------------------------------------------------------
// Many models on one design matrix (fit_many, DESIGN.md 3.2).  One call runs one order of every model
// given; each of its launches covers all of them (one cluster, one row-DP block row, one regularizer-cache
// block per model), so the number of launches does not depend on the number of models.  Every cluster runs
// the code a single sp_pcd_epoch / sp_cd_linear_epoch runs on that model's own records, P and scratch.
namespace {

// Pinned host staging of the argument tables (also used by sp_pbcd_epoch_multi).  It is rewritten only after
// the copy that last read it has completed: `copied` is recorded behind every copy out of it.
struct Staging {
    unsigned char *host = nullptr;
    size_t cap = 0;
    cudaEvent_t copied = nullptr;
    int device = -1;
};
thread_local Staging g_stage;

}  // namespace

int sp_stage_acquire(size_t bytes, unsigned char **out) {
    Staging &s = g_stage;
    int dev = 0;
    SP_CUDA(cudaGetDevice(&dev));
    if (s.copied) {
        SP_CUDA(cudaEventSynchronize(s.copied));
        if (s.device != dev) {
            cudaEventDestroy(s.copied);
            s.copied = nullptr;
        }
    }
    if (!s.copied) {
        SP_CUDA(cudaEventCreateWithFlags(&s.copied, cudaEventDisableTiming));
        s.device = dev;
    }
    if (bytes > s.cap) {
        if (s.host) cudaFreeHost(s.host);
        s.host = nullptr;
        s.cap = 0;
        size_t cap = 4096;
        while (cap < bytes) cap *= 2;
        SP_CUDA(cudaMallocHost((void **)&s.host, cap));
        s.cap = cap;
    }
    *out = s.host;
    return SP_OK;
}

int sp_stage_upload(void *dst, size_t bytes, cudaStream_t st) {
    SP_CUDA(cudaMemcpyAsync(dst, g_stage.host, bytes, cudaMemcpyHostToDevice, st));
    SP_CUDA(cudaEventRecord(g_stage.copied, st));
    return SP_OK;
}

namespace {

constexpr int MULTI_MAX_MODELS = 65535;   // gridDim.y of the row-DP and dead-scan launches

int check_models(const sp_dataset *ds, int n_cta, int threads, const sp_pcd_model *models, int n_models,
                 bool linear, const char *who) {
    if (!ds || n_models < 0 || n_models > MULTI_MAX_MODELS || (n_models > 0 && !models)) {
        sp_set_error("%s: invalid argument (n_models must be 0..%d)", who, MULTI_MAX_MODELS);
        return SP_ERR_INVALID;
    }
    for (int b = 0; b < n_models; b++) {
        const sp_pcd_model &m = models[b];
        sp_plan pl = {n_cta, threads, m.pos_ptr, m.flag_idx, m.idx_feat, m.pos_conf, nullptr};
        int rc = check_plan(ds, &pl, who);
        if (rc) return rc;
        if (!m.P || !m.rec || !m.viol || (!linear && (!m.lams || !m.regstate || !m.idx_comp_host))) {
            sp_set_error("%s: invalid argument (model %d)", who, b);
            return SP_ERR_INVALID;
        }
    }
    return SP_OK;
}

SweepArgs model_args(const sp_dataset *ds, int n_cta, const sp_pcd_model &m, int rec_stride) {
    SweepArgs a = {};
    a.d = ds->n_features; a.C = n_cta;
    a.pos_ptr = m.pos_ptr; a.flag_idx = m.flag_idx; a.data = ds->csc_data;
    a.idx_feat = m.idx_feat; a.pos_conf = m.pos_conf;
    a.ab = m.ab; a.gamma = m.gamma; a.eta = m.eta; a.reg = m.reg;
    a.rec = m.rec; a.stride = rec_stride; a.regstate = m.regstate; a.viol = m.viol;
    return a;
}

}  // namespace

extern "C" int sp_cd_linear_epoch_multi(const sp_dataset *ds, int n_cta, int threads, const double *col_norm_sq,
                                        const sp_pcd_model *models, int n_models, int loss, int rec_stride,
                                        sp_stream stream) {
    int rc = check_models(ds, n_cta, threads, models, n_models, true, "sp_cd_linear_epoch_multi");
    if (rc) return rc;
    if (!col_norm_sq || rec_stride < 2 || (rec_stride & 1)) {
        sp_set_error("sp_cd_linear_epoch_multi: invalid argument");
        return SP_ERR_INVALID;
    }
    if (loss < SP_LOSS_SQUARED || loss > SP_LOSS_SQHINGE) { sp_set_error("unknown loss id %d", loss); return SP_ERR_INVALID; }
    if (ds->n_features == 0 || n_models == 0) return SP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t bytes = sizeof(SweepArgs) * n_models;
    unsigned char *h = nullptr;
    rc = sp_stage_acquire(bytes, &h);
    if (rc) return rc;
    SweepArgs *tab = reinterpret_cast<SweepArgs *>(h);
    for (int b = 0; b < n_models; b++) {
        SweepArgs a = model_args(ds, n_cta, models[b], rec_stride);
        a.prow = models[b].P; a.cns = col_norm_sq; a.lam_ptr = nullptr;      // as sp_cd_linear_epoch
        a.gamma = 0.0; a.eta = 1.0; a.reg = SP_REG_L1; a.regstate = models[b].viol;
        tab[b] = a;
    }
    const SweepArgs first = tab[0];
    SweepArgs *dtab = nullptr;
    SP_CUDA(cudaMallocAsync((void **)&dtab, bytes, st));
    rc = sp_stage_upload(dtab, bytes, st);
    if (!rc) {
        sp_plan pl = {n_cta, threads, nullptr, nullptr, nullptr, nullptr, nullptr};
        rc = dispatch_loss<KIND_LINEAR, 1>(loss, first, dtab, n_models, threads, pick_nz(ds, &pl), st);
    }
    cudaFreeAsync(dtab, st);
    return rc;
}

extern "C" int sp_pcd_epoch_multi(const sp_dataset *ds, int n_cta, int threads, const sp_pcd_model *models,
                                  int n_models, int k, int degree, int loss, int rec_stride, sp_stream stream) {
    int rc = check_models(ds, n_cta, threads, models, n_models, false, "sp_pcd_epoch_multi");
    if (rc) return rc;
    if (k <= 0 || !ds->csr_indptr) {
        sp_set_error("sp_pcd_epoch_multi: invalid argument");
        return SP_ERR_INVALID;
    }
    for (int b = 0; b < n_models; b++) {             // the support matrix of sp_pcd_epoch, per model
        const int reg = models[b].reg;
        if (reg != SP_REG_L1 && reg != SP_REG_SQL12 && reg != SP_REG_OMEGATI) {
            sp_set_error("regularizer id %d does not implement the pcd protocol (use l1, squaredl12 or omegati)", reg);
            return SP_ERR_UNSUPPORTED;
        }
        if (reg == SP_REG_SQL12 && degree != 2) {
            sp_set_error(degree == -1 ? "squaredl12 is not available for all-subsets models"
                                      : "SquaredL12 supports only degree=2.");
            return SP_ERR_UNSUPPORTED;
        }
        for (int ss = 0; ss < k; ss++) {
            const int s = models[b].idx_comp_host[ss];
            if (s < 0 || s >= k) {
                sp_set_error("sp_pcd_epoch_multi: bad component index %d", s);
                return SP_ERR_INVALID;
            }
        }
    }
    if (!(degree == -1 || (degree >= 2 && degree <= SP_MAXDEG))) {
        sp_set_error("pcd degree %d is not supported by the CUDA backend (2..%d or -1)", degree, SP_MAXDEG);
        return SP_ERR_UNSUPPORTED;
    }
    if (rec_stride < sp_min_rec_stride(degree) || (rec_stride & 1)) {
        sp_set_error("sp_pcd_epoch_multi: rec_stride %d too small for degree %d", rec_stride, degree);
        return SP_ERR_INVALID;
    }
    if (loss < SP_LOSS_SQUARED || loss > SP_LOSS_SQHINGE) { sp_set_error("unknown loss id %d", loss); return SP_ERR_INVALID; }
    const int d = ds->n_features;
    if (d == 0 || n_models == 0) return SP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    sp_plan pl = {n_cta, threads, nullptr, nullptr, nullptr, nullptr, nullptr};
    const int nz = pick_nz(ds, &pl);

    // Dead components, the rule of sp_pcd_epoch per model (degree >= 2 and the model's beta > 0): one scan of
    // every (model, component) row, one copy back and one stream synchronisation per call.
    std::vector<int> alive((size_t)n_models * k, 1);
    std::vector<int> scanned;
    if (degree >= 2)
        for (int b = 0; b < n_models; b++)
            if (models[b].ab > 0.0) scanned.push_back(b);
    if (!scanned.empty()) {
        const int ns = (int)scanned.size();
        unsigned char *h = nullptr;
        rc = sp_stage_acquire(sizeof(double *) * ns, &h);
        if (rc) return rc;
        const double **hp = reinterpret_cast<const double **>(h);
        for (int i = 0; i < ns; i++) hp[i] = models[scanned[i]].P;
        void *buf = nullptr;
        SP_CUDA(cudaMallocAsync(&buf, sizeof(double *) * ns + sizeof(int) * ns * k, st));
        const double **dP = reinterpret_cast<const double **>(buf);
        int *flags = reinterpret_cast<int *>(dP + ns);
        std::vector<int> f((size_t)ns * k);
        rc = sp_stage_upload(dP, sizeof(double *) * ns, st);
        cudaError_t e1 = cudaSuccess;
        if (!rc) {
            row_any_nonzero_multi_kernel<<<dim3((unsigned)k, (unsigned)ns), 256, 0, st>>>(dP, d, k, flags);
            e1 = cudaGetLastError();
            if (e1 == cudaSuccess) e1 = cudaMemcpyAsync(f.data(), flags, sizeof(int) * ns * k, cudaMemcpyDeviceToHost, st);
            if (e1 == cudaSuccess) e1 = cudaStreamSynchronize(st);
        }
        cudaFreeAsync(buf, st);
        if (rc) return rc;
        if (e1 != cudaSuccess) return sp_check_cuda(e1, "sp_pcd_epoch_multi: dead-component scan");
        for (int i = 0; i < ns; i++)
            for (int s = 0; s < k; s++) alive[(size_t)scanned[i] * k + s] = f[(size_t)i * k + s];
    }

    // Tables, by position ss of the component order and then in model order: the sweep arguments and the
    // row-DP entries (one per live (model, component) pair, same index), the regularizer-cache entries
    // (pairs of models other than l1, as sp_pcd_epoch skips the cache for l1).
    std::vector<SweepArgs> sw;
    std::vector<SpRowsEntry> rw;
    std::vector<SpRegEntry> rg;
    std::vector<int> sw_off(k + 1), rg_off(k + 1);
    for (int ss = 0; ss < k; ss++) {
        sw_off[ss] = (int)sw.size();
        rg_off[ss] = (int)rg.size();
        for (int b = 0; b < n_models; b++) {
            const sp_pcd_model &m = models[b];
            const int s = m.idx_comp_host[ss];
            if (!alive[(size_t)b * k + s]) continue;
            double *prow = m.P + (size_t)s * d;
            SweepArgs a = model_args(ds, n_cta, m, rec_stride);
            a.prow = prow; a.cns = nullptr; a.lam_ptr = m.lams + s;
            sw.push_back(a);
            rw.push_back({prow, m.rec});
            if (m.reg != SP_REG_L1) rg.push_back({prow, m.regstate, m.reg == SP_REG_SQL12 ? 0 : (degree == -1 ? 2 : 1)});
        }
    }
    sw_off[k] = (int)sw.size();
    rg_off[k] = (int)rg.size();
    if (sw.empty()) return SP_OK;
    const size_t b_sw = sizeof(SweepArgs) * sw.size(), b_rw = sizeof(SpRowsEntry) * rw.size();
    const size_t bytes = b_sw + b_rw + sizeof(SpRegEntry) * rg.size();
    unsigned char *h = nullptr;
    rc = sp_stage_acquire(bytes, &h);
    if (rc) return rc;
    memcpy(h, sw.data(), b_sw);
    memcpy(h + b_sw, rw.data(), b_rw);
    memcpy(h + b_sw + b_rw, rg.data(), sizeof(SpRegEntry) * rg.size());
    unsigned char *dbuf = nullptr;
    SP_CUDA(cudaMallocAsync((void **)&dbuf, bytes, st));
    const SweepArgs *dsw = reinterpret_cast<const SweepArgs *>(dbuf);
    const SpRowsEntry *drw = reinterpret_cast<const SpRowsEntry *>(dbuf + b_sw);
    const SpRegEntry *drg = reinterpret_cast<const SpRegEntry *>(dbuf + b_sw + b_rw);
    rc = sp_stage_upload(dbuf, bytes, st);
    for (int ss = 0; ss < k && !rc; ss++) {
        const int n = sw_off[ss + 1] - sw_off[ss], nr = rg_off[ss + 1] - rg_off[ss];
        if (n == 0) continue;
        rc = sp_rows_precompute_multi(ds, drw + sw_off[ss], n, degree, rec_stride, st);    // pcd.py:94
        if (!rc && nr > 0) rc = sp_launch_reg_cache_multi(drg + rg_off[ss], nr, degree, d, st);   // pcd.py:96
        if (!rc) rc = dispatch_degree(degree, loss, sw[sw_off[ss]], dsw + sw_off[ss], n, threads, nz, st);
    }
    cudaFreeAsync(dbuf, st);
    return rc;
}
