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

// row norms of the models of a table: block row y writes norms[j] = ||P[j,:]||_2 of the entry table[y] {P, norms}
// (squaredl21.py:37, omegacs.py:65)
__global__ void row_norms_kernel(int d, int k, const SpBlockEntry *__restrict__ table) {
    const SpBlockEntry e = table[blockIdx.y];
    const double *__restrict__ P = e.P;
    double *norms = e.out;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    const int n_warps = (gridDim.x * blockDim.x) >> 5;
    for (int j = warp; j < d; j += n_warps) {
        double acc = 0.0;
        for (int s = lane; s < k; s += 32) { const double v = P[(size_t)j * k + s]; acc += v * v; }
        acc = sp_warp_allsum(acc);
        if (lane == 0) norms[j] = sqrt(acc);
    }
}

int row_norms_blocks(int d) {
    int blocks = (d + 7) / 8;
    if (blocks > 148 * 8) blocks = 148 * 8;
    return blocks;
}

// Clusters along x: cluster b runs the block sweep of table[b] (a single fit is a table of one entry).  The entry is
// read from a shared-memory copy, and the register budget is one CTA per SM: read in place from global memory, or
// with __launch_bounds__(PB_MAX_THREADS) alone, ptxas spills in 7 of the 15 instantiations (up to 196 bytes); this
// way none spills (166..238 registers).
template <int KIND, int DEG, int KCH>
__global__ void __launch_bounds__(PB_MAX_THREADS, 1) pbcd_sweep_kernel(const BlockArgs *__restrict__ table, int width) {
    __shared__ BlockArgs entry;
    if (threadIdx.x == 0) entry = table[blockIdx.x / width];
    __syncthreads();
    const BlockArgs &a = entry;
    constexpr int ND = (KIND == PK_FM) ? DEG : 1;          // dA chain length
    constexpr int NA = (KIND == PK_FM) ? DEG - 1 : 1;      // A rows stored per sample
    constexpr int NC = (KIND == PK_FM) ? DEG + 1 : 1;
    constexpr int UB = (KCH * NA <= 2) ? 4 : ((KCH * NA <= 8) ? 2 : 1);   // nonzeros in flight per warp

    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long mbar[2];

    const int T = blockDim.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, W = T >> 5;
    const int C = a.C, PS = C + 1, d = a.d, k = a.k;
    const int c = (C > 1) ? (int)cluster_ctarank() : 0;
    // dynamic smem: red[W][k] double2, then mbox[2][C][k] double2
    double2 *red = reinterpret_cast<double2 *>(smem_raw);
    double2 *mbox = red + (size_t)PB_MAX_THREADS / 32 * k;

    const double mu = sp_mu_rt(a.loss);
    const double beta = a.beta, gamma = a.gamma, eta = a.eta;
    const int reg = a.reg, loss = a.loss;
    const size_t strideA = (size_t)NA * k;

    double lam[KCH];
#pragma unroll
    for (int q = 0; q < KCH; q++) { const int s = lane + 32 * q; lam[q] = s < k ? a.lams[s] : 0.0; }

    double viol = *a.viol;
    double cache[NC];
#pragma unroll
    for (int t = 0; t < NC; t++) cache[t] = a.regstate[t];

    if (C > 1) {
        if (tid == 0) {
            mbar_init(smem_u32(&mbar[0]), 1);
            mbar_init(smem_u32(&mbar[1]), 1);
            fence_mbar_init();
        }
        __syncthreads();
        cluster_sync_all();
    }

    const bool use_norms = (reg == SP_REG_SQL21 || reg == SP_REG_OMEGACS);
    int s1 = 0, e1 = 0, j1 = 0, s2 = 0, e2 = 0, j2 = 0;
    double pnext[KCH], norm_next = 0.0;
#pragma unroll
    for (int q = 0; q < KCH; q++) pnext[q] = 0.0;
    if (0 < d) {
        s1 = a.pos_ptr[c]; e1 = a.pos_ptr[c + 1]; j1 = a.idx_feat[0];
#pragma unroll
        for (int q = 0; q < KCH; q++) { const int s = lane + 32 * q; if (s < k) pnext[q] = a.P[(size_t)j1 * k + s]; }
        if (use_norms) norm_next = a.norms[j1];
    }
    if (1 < d) { s2 = a.pos_ptr[PS + c]; e2 = a.pos_ptr[PS + c + 1]; j2 = a.idx_feat[1]; }

    for (int t = 0; t < d; t++) {
        const int s0 = s1, e0 = e1, j0 = j1;
        double pold[KCH], g[KCH], h[KCH];
#pragma unroll
        for (int q = 0; q < KCH; q++) { pold[q] = pnext[q]; g[q] = 0.0; h[q] = 0.0; }
        const double norm_old = norm_next;
        s1 = s2; e1 = e2; j1 = j2;
        if (t + 1 < d) {       // P row / norm of the next position (never touched by this step)
#pragma unroll
            for (int q = 0; q < KCH; q++) { const int s = lane + 32 * q; if (s < k) pnext[q] = a.P[(size_t)j1 * k + s]; }
            if (use_norms) norm_next = a.norms[j1];
        }
        if (t + 2 < d) {
            s2 = a.pos_ptr[(size_t)(t + 2) * PS + c];
            e2 = a.pos_ptr[(size_t)(t + 2) * PS + c + 1];
            j2 = a.idx_feat[t + 2];
        }
        if (C > 1 && tid == 0) mbar_arrive_expect_tx(smem_u32(&mbar[t & 1]), 16u * (uint32_t)C * (uint32_t)k);
        // this warp's nonzeros of the slice: e = s0 + warp + W*q, q < nq
        const int cnt = e0 - s0;
        const int nq = cnt > warp ? (cnt - warp + W - 1) / W : 0;

        // ------------------------------------------------ partial gradient / curvature sums
        for (int qb = 0; qb < nq; qb += 32) {
            const int ql = qb + lane;
            int idx_l = 0;
            double x_l = 0.0;
            if (ql < nq) {
                const int e = s0 + warp + W * ql;
                idx_l = a.flag_idx[e] & SP_ROW_MASK;
                x_l = a.data[e];
            }
            const int nloc = min(32, nq - qb);
            for (int q0 = 0; q0 < nloc; q0 += UB) {
                int iv[UB];
                double xv[UB], Av[UB][KCH][NA];
                double2 yy[UB];
#pragma unroll
                for (int u = 0; u < UB; u++) {
                    iv[u] = __shfl_sync(0xffffffffu, idx_l, (q0 + u) & 31);
                    xv[u] = sp_shfl(x_l, (q0 + u) & 31);
                }
#pragma unroll
                for (int u = 0; u < UB; u++) {            // UB independent row gathers in flight
                    if (q0 + u < nloc) {
                        yy[u] = *reinterpret_cast<const double2 *>(a.yrec + (size_t)iv[u] * 2);
                        const double *Ai = a.A + (size_t)iv[u] * strideA;
#pragma unroll
                        for (int q = 0; q < KCH; q++) {
                            const int s = lane + 32 * q;
#pragma unroll
                            for (int r = 0; r < NA; r++) Av[u][q][r] = (s < k) ? Ai[(size_t)r * k + s] : 0.0;
                        }
                    }
                }
#pragma unroll
                for (int u = 0; u < UB; u++) {
                    if (q0 + u < nloc) {
                        const double x = xv[u];
                        const double dl = sp_dloss_rt(loss, yy[u].x, yy[u].y);
#pragma unroll
                        for (int q = 0; q < KCH; q++) {
                            double last;
                            if (KIND == PK_FM) {
                                double dprev = x;                          // pbcd.py:9-15
#pragma unroll
                                for (int r = 1; r < ND; r++) dprev = x * (Av[u][q][r - 1] - pold[q] * dprev);
                                last = dprev;
                            } else {
                                last = x * Av[u][q][0] / (1.0 + x * pold[q]);   // pbcd_all.py:51
                            }
                            if (lane + 32 * q < k) {
                                g[q] += dl * last;                          // pbcd.py:65-67
                                h[q] += last * last;
                            }
                        }
                    }
                }
            }
        }
        if (W > 1) {
#pragma unroll
            for (int q = 0; q < KCH; q++) {
                const int s = lane + 32 * q;
                if (s < k) red[(size_t)warp * k + s] = make_double2(g[q], h[q]);
            }
            __syncthreads();
#pragma unroll
            for (int q = 0; q < KCH; q++) {
                const int s = lane + 32 * q;
                g[q] = 0.0; h[q] = 0.0;
                if (s < k)
                    for (int w = 0; w < W; w++) { const double2 v = red[(size_t)w * k + s]; g[q] += v.x; h[q] += v.y; }
            }
        }
        if (C > 1) {
            const int par = t & 1;
            double2 *box = mbox + (size_t)par * C * k;
            for (int r = warp; r < C; r += W) {             // warp r-th pushes this CTA's vector to CTA r
                const uint32_t rbar = mapa_u32(smem_u32(&mbar[par]), (uint32_t)r);
#pragma unroll
                for (int q = 0; q < KCH; q++) {
                    const int s = lane + 32 * q;
                    if (s < k)
                        st_async_2f64(mapa_u32(smem_u32(&box[(size_t)c * k + s]), (uint32_t)r), g[q], h[q], rbar);
                }
            }
            mbar_wait(smem_u32(&mbar[par]), (uint32_t)((t >> 1) & 1));
#pragma unroll
            for (int q = 0; q < KCH; q++) {
                const int s = lane + 32 * q;
                g[q] = 0.0; h[q] = 0.0;
                if (s < k)
                    for (int r = 0; r < C; r++) { const double2 v = box[(size_t)r * k + s]; g[q] += v.x; h[q] += v.y; }
            }
        }

        // ------------------------------------------------ block step (redundant in every warp)
        double inv = 0.0;
#pragma unroll
        for (int q = 0; q < KCH; q++) inv += h[q];
        inv = sp_warp_allsum(inv);                            // pbcd.py:68-72
        inv = inv * mu;
        inv = inv + beta;
        double pnew[KCH];
#pragma unroll
        for (int q = 0; q < KCH; q++) {
            double gr = g[q] * lam[q];                        // pbcd.py:74-78
            gr = gr + beta * pold[q];
            gr = gr / inv;
            pnew[q] = pold[q] - eta * gr;
        }
        double strength = eta * gamma / inv;
        // ---- prox_bcd (l1.py:44-45, l21.py:33-38, squaredl21.py:45-55, omegacs.py:83-106)
        if (reg == SP_REG_L1) {
#pragma unroll
            for (int q = 0; q < KCH; q++) pnew[q] = sp_soft_threshold(pnew[q], strength);
        } else {
            if (reg == SP_REG_SQL21) {
                const double den = 1.0 + 2.0 * strength;
#pragma unroll
                for (int q = 0; q < KCH; q++) pnew[q] = pnew[q] / den;
            }
            double dot = 0.0;
#pragma unroll
            for (int q = 0; q < KCH; q++) dot += pnew[q] * pnew[q];
            dot = sp_warp_allsum(dot);
            const double l2 = sqrt(dot);
            double dc[NC + 1];
#pragma unroll
            for (int u = 0; u <= NC; u++) dc[u] = 0.0;
            double norm_j = norm_old;
            if (reg == SP_REG_SQL21) {
                if (cache[0] < norm_j) cache[0] = warp_sum_array(a.norms, d);
                const double dcache = cache[0] - norm_j;
                strength = 2.0 * dcache * strength / (1.0 + 2.0 * strength);
            } else if (reg == SP_REG_OMEGACS) {
                if (KIND == PK_FM) {
                    dc[1] = 1.0;
                    bool neg = false;
#pragma unroll
                    for (int deg = 2; deg <= DEG; deg++) {
                        double v = cache[deg - 1];
                        v = v - dc[deg - 1] * norm_j;
                        dc[deg] = v;
                        neg = neg || (v < 0.0);
                    }
                    if (neg) {                                // omegacs.py:90-96 recovery branch
                        norm_j = 0.0;
                        double ec[DEG + 1];
                        warp_esp<DEG>(a.norms, d, j0, DEG - 1, ec);
#pragma unroll
                        for (int u = 0; u <= DEG; u++) cache[u] = ec[u];
                        dc[0] = 0.0; dc[1] = 1.0;
#pragma unroll
                        for (int deg = 2; deg <= DEG; deg++) dc[deg] = cache[DEG - 1];
                    }
                    strength = strength * dc[DEG];
                } else {
                    cache[0] = cache[0] / (1.0 + norm_j);
                    strength = strength * cache[0];
                }
            }
            if (l2 > strength) {
                const double sc = 1.0 - strength / l2;
#pragma unroll
                for (int q = 0; q < KCH; q++) pnew[q] = pnew[q] * sc;
            } else {
#pragma unroll
                for (int q = 0; q < KCH; q++) pnew[q] = 0.0;
            }
            // ---- update_cache_pbcd (squaredl21.py:40-43, omegacs.py:68-81)
            if (reg == SP_REG_SQL21 || reg == SP_REG_OMEGACS) {
                double dn = 0.0;
#pragma unroll
                for (int q = 0; q < KCH; q++) dn += pnew[q] * pnew[q];
                dn = sp_warp_allsum(dn);
                const double l2n = sqrt(dn);
                if (reg == SP_REG_SQL21) {
                    cache[0] = cache[0] - norm_j;
                    cache[0] = cache[0] + l2n;
                } else if (KIND == PK_FM) {
                    bool neg = false;
#pragma unroll
                    for (int deg = 1; deg <= DEG; deg++) {
                        cache[deg] = cache[deg] + dc[deg] * l2n;
                        cache[deg] = cache[deg] - dc[deg] * norm_j;
                    }
#pragma unroll
                    for (int deg = 0; deg <= DEG; deg++) neg = neg || (cache[deg] < 0.0);
                    if (neg) {                                // omegacs.py:75-76: full recompute
                        if (c == 0 && tid == 0) a.norms[j0] = l2n;
                        // every warp recomputes from global norms with entry j0 := l2n
                        double ec[DEG + 1], e2[DEG + 1];
                        warp_esp<DEG>(a.norms, d, j0, DEG, ec);
                        e2[0] = ec[0];
#pragma unroll
                        for (int u = 1; u <= DEG; u++) e2[u] = ec[u] + ec[u - 1] * l2n;
#pragma unroll
                        for (int u = 0; u <= DEG; u++) cache[u] = e2[u];
                    }
                } else {
                    cache[0] = cache[0] * (1.0 + l2n);
                }
                if (c == 0 && tid == 0) a.norms[j0] = l2n;
            }
        }
        double upd[KCH], l1 = 0.0;
        bool moved = false;
#pragma unroll
        for (int q = 0; q < KCH; q++) {
            upd[q] = pold[q] - pnew[q];
            l1 += fabs(upd[q]);
            moved = moved || (upd[q] != 0.0);
        }
        viol += sp_warp_allsum(l1);                           // pbcd.py:146 norm(updates, 1)
        moved = __any_sync(0xffffffffu, moved);
        if (c == 0 && warp == 0) {
#pragma unroll
            for (int q = 0; q < KCH; q++) {
                const int s = lane + 32 * q;
                if (s < k) a.P[(size_t)j0 * k + s] = pnew[q];
            }
        }

        // ------------------------------------------------ synchronize predictions and caches
        if (KIND == PK_ALL || moved) {
            for (int qb = 0; qb < nq; qb += 32) {
                const int ql = qb + lane;
                int idx_l = 0;
                double x_l = 0.0;
                if (ql < nq) {
                    const int e = s0 + warp + W * ql;
                    idx_l = a.flag_idx[e] & SP_ROW_MASK;
                    x_l = a.data[e];
                }
                const int nloc = min(32, nq - qb);
                for (int q0 = 0; q0 < nloc; q0 += UB) {
                    int iv[UB];
                    double xv[UB], Av[UB][KCH][NA], ypv[UB];
#pragma unroll
                    for (int u = 0; u < UB; u++) {
                        iv[u] = __shfl_sync(0xffffffffu, idx_l, (q0 + u) & 31);
                        xv[u] = sp_shfl(x_l, (q0 + u) & 31);
                    }
#pragma unroll
                    for (int u = 0; u < UB; u++) {
                        if (q0 + u < nloc) {
                            ypv[u] = a.yrec[(size_t)iv[u] * 2];
                            const double *Ai = a.A + (size_t)iv[u] * strideA;
#pragma unroll
                            for (int q = 0; q < KCH; q++) {
                                const int s = lane + 32 * q;
#pragma unroll
                                for (int r = 0; r < NA; r++) Av[u][q][r] = (s < k) ? Ai[(size_t)r * k + s] : 0.0;
                            }
                        }
                    }
#pragma unroll
                    for (int u = 0; u < UB; u++) {
                        if (q0 + u < nloc) {
                            const double x = xv[u];
                            double *Ai = a.A + (size_t)iv[u] * strideA;
                            double dy = 0.0, dy2 = 0.0;
#pragma unroll
                            for (int q = 0; q < KCH; q++) {
                                const int s = lane + 32 * q;
                                if (s < k) {
                                    if (KIND == PK_FM) {
                                        double dprev = x;                  // pbcd.py:138-144
#pragma unroll
                                        for (int r = 1; r < ND; r++) {
                                            const double Aold = Av[u][q][r - 1];
                                            const double dcur = x * (Aold - pold[q] * dprev);
                                            Ai[(size_t)(r - 1) * k + s] = Aold - upd[q] * dprev;
                                            dprev = dcur;
                                        }
                                        dy += (lam[q] * upd[q]) * dprev;
                                    } else {
                                        double Aval = Av[u][q][0];         // pbcd_all.py:121-126
                                        dy += lam[q] * Aval;
                                        Aval = Aval / (1.0 + x * pold[q]);
                                        Aval = Aval * (1.0 + x * pnew[q]);
                                        Ai[s] = Aval;
                                        dy2 += lam[q] * Aval;
                                    }
                                }
                            }
                            dy = sp_warp_allsum(dy);
                            if (KIND == PK_ALL) dy2 = sp_warp_allsum(dy2);
                            if (lane == 0) {
                                double yp = ypv[u] - dy;
                                if (KIND == PK_ALL) yp = yp + dy2;
                                a.yrec[(size_t)iv[u] * 2] = yp;
                            }
                        }
                    }
                }
            }
        }
        if (W > 1) __syncthreads(); else __syncwarp();
    }

    if (c == 0 && tid == 0) {
        *a.viol = viol;
#pragma unroll
        for (int t = 0; t < NC; t++) a.regstate[t] = cache[t];
    }
    if (C > 1) cluster_sync_all();
}

// n_tab clusters of C CTAs run the device table; every entry has the same k
template <int KIND, int DEG, int KCH>
int launch_block(const BlockArgs *table, int n_tab, int C, int k, int threads, cudaStream_t st) {
    const size_t smem = ((size_t)PB_MAX_THREADS / 32 + 2 * (size_t)C) * k * sizeof(double2);
    auto kern = pbcd_sweep_kernel<KIND, DEG, KCH>;
    SP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (C > 8) SP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)C * (unsigned)n_tab, 1, 1);
    cfg.blockDim = dim3((unsigned)threads, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    sp_prof_begin(SP_PROF_SWEEP_PBCD, st);
    cudaError_t le = cudaLaunchKernelEx(&cfg, kern, table, C);
    sp_prof_end(st);
    return sp_check_cuda(le, "pbcd_sweep_kernel launch");
}

template <int KIND, int DEG>
int dispatch_kch(const BlockArgs *table, int n_tab, int C, int k, int threads, cudaStream_t st) {
    if (k <= 32) return launch_block<KIND, DEG, 1>(table, n_tab, C, k, threads, st);
    if (k <= 64) return launch_block<KIND, DEG, 2>(table, n_tab, C, k, threads, st);
    return launch_block<KIND, DEG, 4>(table, n_tab, C, k, threads, st);      // k <= 128 (check_args)
}

int dispatch_degree(int degree, const BlockArgs *table, int n_tab, int C, int k, int threads, cudaStream_t st) {
    switch (degree) {
    case -1: return dispatch_kch<PK_ALL, 1>(table, n_tab, C, k, threads, st);
    case 2: return dispatch_kch<PK_FM, 2>(table, n_tab, C, k, threads, st);
    case 3: return dispatch_kch<PK_FM, 3>(table, n_tab, C, k, threads, st);
    case 4: return dispatch_kch<PK_FM, 4>(table, n_tab, C, k, threads, st);
    case 5: return dispatch_kch<PK_FM, 5>(table, n_tab, C, k, threads, st);
    }
    return SP_ERR_UNSUPPORTED;
}

// The checks of sp_pbcd_epoch and sp_pbcd_epoch_multi.  A window plan needs only the order (idx_feat), and its
// geometry is not used.
int check_args(const sp_dataset *ds, int n_cta, int threads, const sp_wplan *win, const sp_pbcd_model *models,
               int n_models, int k, int degree, int loss, const char *who) {
    if (!ds || !ds->csc_data || !ds->csr_indptr || (win && !ds->csc_indptr) || k <= 0 || n_models < 0 ||
        n_models > PB_MULTI_MAX_MODELS || (n_models > 0 && !models) || (win && n_models != 1)) {
        sp_set_error("%s: invalid argument (n_models must be 0..%d, 1 with a window plan)", who, PB_MULTI_MAX_MODELS);
        return SP_ERR_INVALID;
    }
    if (!win && (n_cta < 1 || n_cta > PB_MAX_CTAS || (n_cta & (n_cta - 1)) || threads < 32 ||
                 threads > PB_MAX_THREADS || threads % 32)) {
        sp_set_error("%s: bad plan (n_cta power of two <= %d, threads multiple of 32 <= %d)", who, PB_MAX_CTAS,
                     PB_MAX_THREADS);
        return SP_ERR_INVALID;
    }
    for (int b = 0; b < n_models; b++) {
        const sp_pbcd_model &m = models[b];
        if (!m.idx_feat || (!win && (!m.pos_ptr || !m.flag_idx)) || !m.P || !m.lams || !m.yrec || !m.A ||
            !m.reg_norms || !m.regstate || !m.viol) {
            sp_set_error("%s: invalid argument (model %d)", who, b);
            return SP_ERR_INVALID;
        }
        if (m.reg != SP_REG_L1 && m.reg != SP_REG_L21 && m.reg != SP_REG_SQL21 && m.reg != SP_REG_OMEGACS) {
            sp_set_error("regularizer id %d does not implement the pbcd protocol (use l1, l21, squaredl21 or omegacs)",
                         m.reg);
            return SP_ERR_UNSUPPORTED;
        }
        if (m.reg == SP_REG_SQL21 && degree != 2) {
            sp_set_error(degree == -1 ? "squaredl21 is not available for all-subsets models"
                                      : "SquaredL21 supports only degree=2.");
            return SP_ERR_UNSUPPORTED;
        }
    }
    if (!(degree == -1 || (degree >= 2 && degree <= SP_MAXDEG))) {
        sp_set_error("pbcd degree %d is not supported by the CUDA backend (2..%d or -1)", degree, SP_MAXDEG);
        return SP_ERR_UNSUPPORTED;
    }
    if (k > 128) {
        sp_set_error("pbcd: n_components=%d > 128 is not supported by the CUDA backend", k);
        return SP_ERR_UNSUPPORTED;
    }
    if (loss < SP_LOSS_SQUARED || loss > SP_LOSS_SQHINGE) { sp_set_error("unknown loss id %d", loss); return SP_ERR_INVALID; }
    return SP_OK;
}

// regularizer-cache mode of reg_cache_kernel for the row norms (squaredl21: sum, omegacs: ESP or product)
int reg_cache_mode(int reg, int degree) { return (reg == SP_REG_SQL21) ? 0 : (degree == -1 ? 2 : 1); }

// One order of a list of models on one design matrix (DESIGN.md 3.3), in at most four launches, each covering all of
// them: the row DP (one block row per model), the row norms and the regularizer caches (squaredl21 / omegacs models
// only) and the block sweep (one cluster per model); sp_pbcd_epoch runs a list of one.  A window plan (one model
// only) replaces the cluster sweep by sp_pbcd_wsweep.
int pbcd_epoch(const sp_dataset *ds, int n_cta, int threads, const sp_wplan *win, const sp_pbcd_model *models,
               int n_models, int k, int degree, int loss, cudaStream_t st, const char *who) {
    int rc = check_args(ds, n_cta, threads, win, models, n_models, k, degree, loss, who);
    if (rc) return rc;
    const int d = ds->n_features;
    if (d == 0 || n_models == 0) return SP_OK;

    // Tables in model order: the sweep arguments and row-DP entries (every model), the row-norm and
    // regularizer-cache entries (squaredl21 / omegacs models: l1 and l21 need neither).
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
        row_norms_kernel<<<dim3((unsigned)row_norms_blocks(d), (unsigned)nn), 256, 0, st>>>(d, k, dnw);
        sp_prof_end(st);
        rc = sp_check_cuda(cudaGetLastError(), "row_norms_kernel");
        if (!rc) rc = sp_launch_reg_cache_multi(drg, nn, degree, d, st);
    }
    if (!rc) {
        const BlockArgs &a = sw[0];
        rc = win ? sp_pbcd_wsweep(ds, win, a.idx_feat, a.P, k, a.lams, degree, a.beta, a.gamma, a.eta, a.reg, loss,
                                  a.yrec, a.A, a.norms, a.regstate, a.viol, st)
                 : dispatch_degree(degree, dsw, n_models, n_cta, k, threads, st);
    }
    cudaFreeAsync(dbuf, st);
    return rc;
}

}  // namespace

extern "C" int sp_pbcd_epoch(const sp_dataset *ds, const sp_plan *plan, double *P_dk, int k,
                             const double *lams, int degree, double beta, double gamma, double eta,
                             int reg, int loss, double *yrec, double *A, double *reg_norms,
                             double *regstate, double *viol, sp_stream stream) {
    if (!plan) { sp_set_error("sp_pbcd_epoch: invalid argument"); return SP_ERR_INVALID; }
    sp_pbcd_model m = {};
    m.pos_ptr = plan->pos_ptr; m.flag_idx = plan->flag_idx; m.idx_feat = plan->idx_feat;
    m.P = P_dk; m.lams = lams; m.beta = beta; m.gamma = gamma; m.eta = eta; m.reg = reg;
    m.yrec = yrec; m.A = A; m.reg_norms = reg_norms; m.regstate = regstate; m.viol = viol;
    return pbcd_epoch(ds, plan->n_cta, plan->threads, plan->win, &m, 1, k, degree, loss, (cudaStream_t)stream,
                      "sp_pbcd_epoch");
}

extern "C" int sp_pbcd_epoch_multi(const sp_dataset *ds, int n_cta, int threads, const sp_pbcd_model *models,
                                   int n_models, int k, int degree, int loss, sp_stream stream) {
    return pbcd_epoch(ds, n_cta, threads, nullptr, models, n_models, k, degree, loss, (cudaStream_t)stream,
                      "sp_pbcd_epoch_multi");
}
