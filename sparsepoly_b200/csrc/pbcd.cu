// Proximal BLOCK coordinate descent sweeps on one thread-block cluster (sm_100a):
//   * pbcd.pbcd_epoch      (reference optimizer/pbcd.py:36-148)
//   * pbcd_all.pbcd_epoch  (reference optimizer/pbcd_all.py:23-132)
// One block step = all k components of feature j.  Lanes run over components (coalesced rows of
// A[i, t, :] and P[j, :]), warps run over the nonzeros of the column slice their CTA owns
// (samples are range-partitioned over the cluster's CTAs exactly as in pcd.cu), the per-CTA
// partial (g_s, h_s) vectors are exchanged all-to-all through distributed shared memory, and the
// row prox + regularizer cache chain is evaluated redundantly by every warp.  The reference's
// dA[n, m, k] stash (pbcd.py:60-67) is recomputed instead of stored (SURVEY.md 8d).
#include <string.h>

#include <vector>

#include "common.cuh"
#include "cluster.cuh"
#include "sparsepoly_b200.h"
#include "pbcd_common.cuh"

int sp_rows_precompute_all(const sp_dataset *ds, const double *P_dk, int k, int degree, double *A,
                           cudaStream_t st);
int sp_launch_reg_cache(int mode, int degree, int d, const double *v, double *regstate, cudaStream_t st);
int sp_rows_precompute_all_multi(const sp_dataset *ds, const SpBlockEntry *table, int n_tab, int k, int degree,
                                 cudaStream_t st);
int sp_launch_reg_cache_multi(const SpRegEntry *table, int n_tab, int degree, int d, cudaStream_t st);
int sp_pbcd_wsweep(const sp_dataset *ds, const sp_wplan *wp, const int32_t *idx_feat, double *P_dk, int k,
                   const double *lams, int degree, double beta, double gamma, double eta, int reg, int loss,
                   double *yrec, double *A, double *norms, double *regstate, double *viol, cudaStream_t st);

namespace {

constexpr int PB_MAX_THREADS = 256;
constexpr int PB_MAX_CTAS = 16;
constexpr int PB_MULTI_MAX_MODELS = 65535;   // gridDim.y of the row-DP and row-norm launches

struct BlockArgs {
    int d, C, k;
    const int32_t *pos_ptr, *flag_idx, *idx_feat;
    const double *data;
    double *P;            // [d,k]
    const double *lams;   // [k]
    double beta, gamma, eta;
    int reg, loss;
    double *yrec;         // [n,2]
    double *A;            // [n,(m-1),k] or [n,k]
    double *norms;        // [d]
    double *regstate;     // cache[0..]
    double *viol;
};

// row norms: norms[j] = ||P[j,:]||_2   (squaredl21.py:37, omegacs.py:65)
__device__ __forceinline__ void row_norms_body(int d, int k, const double *__restrict__ P, double *norms) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int n_warps = (gridDim.x * blockDim.x) >> 5;
    for (int j = warp; j < d; j += n_warps) {
        double acc = 0.0;
        for (int s = lane; s < k; s += 32) { const double v = P[(size_t)j * k + s]; acc += v * v; }
        acc = sp_warp_allsum(acc);
        if (lane == 0) norms[j] = sqrt(acc);
    }
}

__global__ void row_norms_kernel(int d, int k, const double *__restrict__ P, double *norms) {
    row_norms_body(d, k, P, norms);
}

// many models (sp_pbcd_epoch_multi): block row y computes the norms of table[y] as row_norms_kernel does
__global__ void row_norms_multi_kernel(int d, int k, const SpBlockEntry *__restrict__ table) {
    const SpBlockEntry e = table[blockIdx.y];
    row_norms_body(d, k, e.P, e.out);
}

int row_norms_blocks(int d) {
    int blocks = (d + 7) / 8;
    if (blocks > 148 * 8) blocks = 148 * 8;
    return blocks;
}

template <int KIND, int DEG, int KCH>
__global__ void __launch_bounds__(PB_MAX_THREADS) pbcd_sweep_kernel(const BlockArgs a) {
#include "pbcd_sweep_body.inc"
}

// Many models per launch (sp_pbcd_epoch_multi): clusters along x, cluster b runs the block sweep of table[b]
// exactly as pbcd_sweep_kernel runs its argument.  The entry is read from a shared-memory copy, and the register
// budget is one CTA per SM: read in place from global memory, or with the single kernel's budget, ptxas spills
// in 7 of the 15 instantiations (up to 196 bytes); this way none spills (166..238 registers).
template <int KIND, int DEG, int KCH>
__global__ void __launch_bounds__(PB_MAX_THREADS, 1) pbcd_sweep_multi_kernel(const BlockArgs *__restrict__ table,
                                                                             int width) {
    __shared__ BlockArgs entry;
    if (threadIdx.x == 0) entry = table[blockIdx.x / width];
    __syncthreads();
    const BlockArgs &a = entry;
#include "pbcd_sweep_body.inc"
}

// table == nullptr: one cluster runs `a`.  Otherwise n_tab clusters run the device table (its host copy
// starts with `a`; every entry has the width a.C and the same k).
template <int KIND, int DEG, int KCH>
int launch_block(const BlockArgs &a, const BlockArgs *table, int n_tab, int threads, cudaStream_t st) {
    const size_t smem = ((size_t)PB_MAX_THREADS / 32 + 2 * (size_t)a.C) * a.k * sizeof(double2);
    auto set_attrs = [&](auto kern) {
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return sp_check_cuda(e, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize)");
        if (a.C > 8) {
            e = cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e != cudaSuccess) return sp_check_cuda(e, "cudaFuncSetAttribute(NonPortableClusterSizeAllowed)");
        }
        return (int)SP_OK;
    };
    int rc = table ? set_attrs(pbcd_sweep_multi_kernel<KIND, DEG, KCH>) : set_attrs(pbcd_sweep_kernel<KIND, DEG, KCH>);
    if (rc) return rc;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)a.C * (unsigned)(table ? n_tab : 1), 1, 1);
    cfg.blockDim = dim3((unsigned)threads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)a.C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    sp_prof_begin(SP_PROF_SWEEP_PBCD, st);
    cudaError_t le = table ? cudaLaunchKernelEx(&cfg, pbcd_sweep_multi_kernel<KIND, DEG, KCH>, table, a.C)
                           : cudaLaunchKernelEx(&cfg, pbcd_sweep_kernel<KIND, DEG, KCH>, a);
    sp_prof_end(st);
    return sp_check_cuda(le, table ? "pbcd_sweep_multi_kernel launch" : "pbcd_sweep_kernel launch");
}

template <int KIND, int DEG>
int dispatch_kch(const BlockArgs &a, const BlockArgs *table, int n_tab, int threads, cudaStream_t st) {
    if (a.k <= 32) return launch_block<KIND, DEG, 1>(a, table, n_tab, threads, st);
    if (a.k <= 64) return launch_block<KIND, DEG, 2>(a, table, n_tab, threads, st);
    if (a.k <= 128) return launch_block<KIND, DEG, 4>(a, table, n_tab, threads, st);
    sp_set_error("pbcd: n_components=%d > 128 is not supported by the CUDA backend", a.k);
    return SP_ERR_UNSUPPORTED;
}

int dispatch_degree(int degree, const BlockArgs &a, const BlockArgs *table, int n_tab, int threads, cudaStream_t st) {
    switch (degree) {
    case -1: return dispatch_kch<PK_ALL, 1>(a, table, n_tab, threads, st);
    case 2: return dispatch_kch<PK_FM, 2>(a, table, n_tab, threads, st);
    case 3: return dispatch_kch<PK_FM, 3>(a, table, n_tab, threads, st);
    case 4: return dispatch_kch<PK_FM, 4>(a, table, n_tab, threads, st);
    case 5: return dispatch_kch<PK_FM, 5>(a, table, n_tab, threads, st);
    }
    return SP_ERR_UNSUPPORTED;
}

// the checks sp_pbcd_epoch makes on its arguments, shared with sp_pbcd_epoch_multi
int check_geometry(int n_cta, int threads, const char *who) {
    if (n_cta < 1 || n_cta > PB_MAX_CTAS || (n_cta & (n_cta - 1)) || threads < 32 || threads > PB_MAX_THREADS ||
        threads % 32) {
        sp_set_error("%s: bad plan (n_cta power of two <= %d, threads multiple of 32 <= %d)", who, PB_MAX_CTAS,
                     PB_MAX_THREADS);
        return SP_ERR_INVALID;
    }
    return SP_OK;
}

int check_reg_degree(int reg, int degree) {
    if (reg != SP_REG_L1 && reg != SP_REG_L21 && reg != SP_REG_SQL21 && reg != SP_REG_OMEGACS) {
        sp_set_error("regularizer id %d does not implement the pbcd protocol (use l1, l21, squaredl21 or omegacs)", reg);
        return SP_ERR_UNSUPPORTED;
    }
    if (reg == SP_REG_SQL21 && degree != 2) {
        sp_set_error(degree == -1 ? "squaredl21 is not available for all-subsets models"
                                  : "SquaredL21 supports only degree=2.");
        return SP_ERR_UNSUPPORTED;
    }
    if (!(degree == -1 || (degree >= 2 && degree <= SP_MAXDEG))) {
        sp_set_error("pbcd degree %d is not supported by the CUDA backend (2..%d or -1)", degree, SP_MAXDEG);
        return SP_ERR_UNSUPPORTED;
    }
    return SP_OK;
}

// regularizer-cache mode of reg_cache_body for the row norms (squaredl21: sum, omegacs: ESP or product)
int reg_cache_mode(int reg, int degree) { return (reg == SP_REG_SQL21) ? 0 : (degree == -1 ? 2 : 1); }

}  // namespace

extern "C" int sp_pbcd_epoch(const sp_dataset *ds, const sp_plan *plan, double *P_dk, int k,
                             const double *lams, int degree, double beta, double gamma, double eta,
                             int reg, int loss, double *yrec, double *A, double *reg_norms,
                             double *regstate, double *viol, sp_stream stream) {
    if (!ds || !plan || !ds->csc_data || !ds->csr_indptr || !plan->idx_feat || !P_dk || !lams || !yrec || !A ||
        !reg_norms || !regstate || !viol || k <= 0 || (!plan->win && (!plan->pos_ptr || !plan->flag_idx))) {
        sp_set_error("sp_pbcd_epoch: invalid argument");
        return SP_ERR_INVALID;
    }
    if (!plan->win) {
        int rc = check_geometry(plan->n_cta, plan->threads, "sp_pbcd_epoch");
        if (rc) return rc;
    }
    int rc = check_reg_degree(reg, degree);
    if (rc) return rc;
    if (loss < 0 || loss > 2) { sp_set_error("unknown loss id %d", loss); return SP_ERR_INVALID; }
    const int d = ds->n_features;
    if (d == 0) return SP_OK;
    cudaStream_t st = (cudaStream_t)stream;
    rc = sp_rows_precompute_all(ds, P_dk, k, degree, A, st);                   // pbcd.py:107
    if (rc) return rc;
    if (reg == SP_REG_SQL21 || reg == SP_REG_OMEGACS) {                         // pbcd.py:109
        sp_prof_begin(SP_PROF_REGCACHE, st);
        row_norms_kernel<<<row_norms_blocks(d), 256, 0, st>>>(d, k, P_dk, reg_norms);
        sp_prof_end(st);
        SP_LAUNCH_CHECK("row_norms_kernel");
        rc = sp_launch_reg_cache(reg_cache_mode(reg, degree), degree, d, reg_norms, regstate, st);
        if (rc) return rc;
    }
    if (plan->win)
        return sp_pbcd_wsweep(ds, plan->win, plan->idx_feat, P_dk, k, lams, degree, beta, gamma, eta, reg, loss, yrec,
                              A, reg_norms, regstate, viol, st);
    BlockArgs a = {};
    a.d = d; a.C = plan->n_cta; a.k = k;
    a.pos_ptr = plan->pos_ptr; a.flag_idx = plan->flag_idx; a.idx_feat = plan->idx_feat;
    a.data = ds->csc_data; a.P = P_dk; a.lams = lams;
    a.beta = beta; a.gamma = gamma; a.eta = eta; a.reg = reg; a.loss = loss;
    a.yrec = yrec; a.A = A; a.norms = reg_norms; a.regstate = regstate; a.viol = viol;
    return dispatch_degree(degree, a, nullptr, 0, plan->threads, st);
}

// ------------------------------------------------------------------------------------------------
// Many models on one design matrix (fit_many, DESIGN.md 3.3).  One call runs one order of every model given in
// at most four launches, each covering all of them: the row DP (one block row per model), the row norms and the
// regularizer caches (squaredl21 / omegacs models only) and the block sweep (one cluster per model).  Every
// cluster runs the code sp_pbcd_epoch runs with a cluster plan, on that model's own P, records and scratch.
extern "C" int sp_pbcd_epoch_multi(const sp_dataset *ds, int n_cta, int threads, const sp_pbcd_model *models,
                                   int n_models, int k, int degree, int loss, sp_stream stream) {
    if (!ds || !ds->csc_data || !ds->csr_indptr || k <= 0 || n_models < 0 || n_models > PB_MULTI_MAX_MODELS ||
        (n_models > 0 && !models)) {
        sp_set_error("sp_pbcd_epoch_multi: invalid argument (n_models must be 0..%d)", PB_MULTI_MAX_MODELS);
        return SP_ERR_INVALID;
    }
    int rc = check_geometry(n_cta, threads, "sp_pbcd_epoch_multi");
    if (rc) return rc;
    for (int b = 0; b < n_models; b++) {             // what sp_pbcd_epoch checks, per model
        const sp_pbcd_model &m = models[b];
        if (!m.pos_ptr || !m.flag_idx || !m.idx_feat || !m.P || !m.lams || !m.yrec || !m.A || !m.reg_norms ||
            !m.regstate || !m.viol) {
            sp_set_error("sp_pbcd_epoch_multi: invalid argument (model %d)", b);
            return SP_ERR_INVALID;
        }
        rc = check_reg_degree(m.reg, degree);
        if (rc) return rc;
    }
    rc = check_reg_degree(SP_REG_L1, degree);
    if (rc) return rc;
    if (k > 128) {
        sp_set_error("pbcd: n_components=%d > 128 is not supported by the CUDA backend", k);
        return SP_ERR_UNSUPPORTED;
    }
    if (loss < SP_LOSS_SQUARED || loss > SP_LOSS_SQHINGE) { sp_set_error("unknown loss id %d", loss); return SP_ERR_INVALID; }
    const int d = ds->n_features;
    if (d == 0 || n_models == 0) return SP_OK;
    cudaStream_t st = (cudaStream_t)stream;

    // Tables in model order: the sweep arguments and row-DP entries (every model), the row-norm and
    // regularizer-cache entries (squaredl21 / omegacs models, as sp_pbcd_epoch skips both for l1 / l21).
    std::vector<BlockArgs> sw(n_models);
    std::vector<SpBlockEntry> rw(n_models), nw;
    std::vector<SpRegEntry> rg;
    for (int b = 0; b < n_models; b++) {
        const sp_pbcd_model &m = models[b];
        BlockArgs &a = sw[b];
        a = {};
        a.d = d; a.C = n_cta; a.k = k;
        a.pos_ptr = m.pos_ptr; a.flag_idx = m.flag_idx; a.idx_feat = m.idx_feat;
        a.data = ds->csc_data; a.P = m.P; a.lams = m.lams;
        a.beta = m.beta; a.gamma = m.gamma; a.eta = m.eta; a.reg = m.reg; a.loss = loss;
        a.yrec = m.yrec; a.A = m.A; a.norms = m.reg_norms; a.regstate = m.regstate; a.viol = m.viol;
        rw[b] = {m.P, m.A};
        if (m.reg == SP_REG_SQL21 || m.reg == SP_REG_OMEGACS) {
            nw.push_back({m.P, m.reg_norms});
            rg.push_back({m.reg_norms, m.regstate, reg_cache_mode(m.reg, degree)});
        }
    }
    const int nn = (int)nw.size();
    const size_t b_sw = sizeof(BlockArgs) * sw.size(), b_rw = sizeof(SpBlockEntry) * rw.size();
    const size_t b_nw = sizeof(SpBlockEntry) * nw.size(), b_rg = sizeof(SpRegEntry) * rg.size();
    const size_t bytes = b_sw + b_rw + b_nw + b_rg;
    unsigned char *h = nullptr;
    rc = sp_stage_acquire(bytes, &h);
    if (rc) return rc;
    memcpy(h, sw.data(), b_sw);
    memcpy(h + b_sw, rw.data(), b_rw);
    if (nn > 0) {
        memcpy(h + b_sw + b_rw, nw.data(), b_nw);
        memcpy(h + b_sw + b_rw + b_nw, rg.data(), b_rg);
    }
    unsigned char *dbuf = nullptr;
    SP_CUDA(cudaMallocAsync((void **)&dbuf, bytes, st));
    const BlockArgs *dsw = reinterpret_cast<const BlockArgs *>(dbuf);
    const SpBlockEntry *drw = reinterpret_cast<const SpBlockEntry *>(dbuf + b_sw);
    const SpBlockEntry *dnw = reinterpret_cast<const SpBlockEntry *>(dbuf + b_sw + b_rw);
    const SpRegEntry *drg = reinterpret_cast<const SpRegEntry *>(dbuf + b_sw + b_rw + b_nw);
    rc = sp_stage_upload(dbuf, bytes, st);
    if (!rc) rc = sp_rows_precompute_all_multi(ds, drw, n_models, k, degree, st);          // pbcd.py:107
    if (!rc && nn > 0) {                                                                   // pbcd.py:109
        sp_prof_begin(SP_PROF_REGCACHE, st);
        row_norms_multi_kernel<<<dim3((unsigned)row_norms_blocks(d), (unsigned)nn), 256, 0, st>>>(d, k, dnw);
        sp_prof_end(st);
        rc = sp_check_cuda(cudaGetLastError(), "row_norms_multi_kernel");
        if (!rc) rc = sp_launch_reg_cache_multi(drg, nn, degree, d, st);
    }
    if (!rc) rc = dispatch_degree(degree, sw[0], dsw, n_models, threads, st);
    cudaFreeAsync(dbuf, st);
    return rc;
}
