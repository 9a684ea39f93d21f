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


// Clusters along x: cluster b runs the sweep of table[b] (a single fit is a table of one entry).
template <int KIND, int DEG, int LOSS, int NZ>
__global__ void __launch_bounds__(SWEEP_MAX_THREADS + 32) sweep_kernel(const SweepArgs *__restrict__ table, int width) {
    const SweepArgs &a = table[blockIdx.x / width];   // read in place: no register copy of the entry
    constexpr int NA = (KIND == KIND_FM) ? DEG - 1 : (KIND == KIND_ALL ? 1 : 0);
    constexpr int R = 2 + NA;                                // doubles used per record
    constexpr int NCH = (R + 1) / 2;                         // 16-byte chunks staged per record
    constexpr int ND = (KIND == KIND_FM) ? DEG : 1;
    constexpr int NC = (KIND == KIND_FM) ? DEG : 1;          // regularizer cache scalars

    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ __align__(8) unsigned long long mbar[MBOX_DEPTH];   // partials of position q have landed
    __shared__ __align__(8) unsigned long long rbar[MBOX_DEPTH];   // result of position q is published
    __shared__ double2 res[MBOX_DEPTH];                             // (upd, pnew) of position q

    // warp roles: warps 0..W-1 gather (stage, terms, push, write-back); warp W runs the scalar chain
    const int T = blockDim.x - 32, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, W = T >> 5;
    const bool scalar_role = warp == W;
    const int C = a.C, d = a.d;
    const int c = (C > 1) ? (int)cluster_ctarank() : 0;
    const int NP = C * W;                                    // partials per position
    const int stride = a.stride;
    const double lam = (KIND == KIND_LINEAR) ? 1.0 : *a.lam_ptr;

    // dynamic smem carve-up
    double2 *recbuf = reinterpret_cast<double2 *>(smem_raw);                 // [2][NZ][NCH][T]
    double *xbuf = reinterpret_cast<double *>(recbuf + (size_t)2 * NZ * NCH * T);   // [3][NZ][T]
    double2 *mbox = reinterpret_cast<double2 *>(xbuf + (size_t)3 * NZ * T);  // [MBOX_DEPTH][NP]
    int *idxbuf = reinterpret_cast<int *>(mbox + (size_t)MBOX_DEPTH * NP);   // [3][NZ][T]

    if (tid == 0) {
#pragma unroll
        for (int b = 0; b < MBOX_DEPTH; b++) {
            mbar_init(smem_u32(&mbar[b]), 1);
            mbar_init(smem_u32(&rbar[b]), 1);
        }
        fence_mbar_init();
    }
    __syncthreads();
    if (C > 1) cluster_sync_all();

    // ------------------------------------------------------------------ per-position table
    MetaChunk mcur, mnxt, mnx2;
    meta_load_ptr(mcur, a, 0, c, lane);
    meta_load_ptr(mnxt, a, 32, c, lane);
    meta_load_ptr(mnx2, a, 64, c, lane);
    meta_load_val<KIND>(mcur, a, 0, lane);
    meta_load_val<KIND>(mnxt, a, 32, lane);
    int chunk_base = 0;
    auto meta_se = [&](int q, int &s, int &e) {
        const int l = q & 31;
        const int s1 = __shfl_sync(0xffffffffu, mcur.s, l), e1 = __shfl_sync(0xffffffffu, mcur.e, l);
        const int s2 = __shfl_sync(0xffffffffu, mnxt.s, l), e2 = __shfl_sync(0xffffffffu, mnxt.e, l);
        const bool in_cur = (q - chunk_base) < 32;
        s = in_cur ? s1 : s2; e = in_cur ? e1 : e2;
        if (q >= d) { s = 0; e = 0; }
    };
    auto meta_val = [&](int q, int &jf, double &pold, double &cn) {
        const int l = q & 31;
        const bool in_cur = (q - chunk_base) < 32;
        const int j1 = __shfl_sync(0xffffffffu, mcur.jf, l), j2 = __shfl_sync(0xffffffffu, mnxt.jf, l);
        const double p1 = sp_shfl(mcur.pold, l), p2 = sp_shfl(mnxt.pold, l);
        jf = in_cur ? j1 : j2; pold = in_cur ? p1 : p2;
        if (KIND == KIND_LINEAR) {
            const double c1 = sp_shfl(mcur.cn, l), c2 = sp_shfl(mnxt.cn, l);
            cn = in_cur ? c1 : c2;
        } else cn = 0.0;
    };
    auto meta_advance = [&](int t_next) {                     // entering the next chunk of positions
        if ((t_next & 31) == 0) {
            chunk_base = t_next;
            mcur = mnxt;
            mnxt = mnx2;
            meta_load_val<KIND>(mnxt, a, chunk_base + 32, lane);
            meta_load_ptr(mnx2, a, chunk_base + 64, c, lane);
        }
    };

    if (scalar_role) {
        // =============================================================== scalar-chain warp
        const double mu = sp_mu<LOSS>();
        const double ab = a.ab, gamma = a.gamma, eta = a.eta;
        const int reg = a.reg;
        double viol = *a.viol;
        double cache[NC];
#pragma unroll
        for (int t = 0; t < NC; t++) cache[t] = a.regstate[t];
        if (lane == 0) {
#pragma unroll
            for (int b = 0; b < MBOX_DEPTH; b++)
                if (b < d) mbar_arrive_expect_tx(smem_u32(&mbar[b]), 16u * (uint32_t)NP);
        }
        for (int t = 0; t < d; t++) {
            int jf0;
            double pold0, cn0;
            meta_val(t, jf0, pold0, cn0);
            const int b = t & (MBOX_DEPTH - 1);
            mbar_wait(smem_u32(&mbar[b]), (uint32_t)((t >> 2) & 1));
            double g0 = 0.0, h0 = 0.0, g1 = 0.0, h1 = 0.0;
            {
                const double2 *box = mbox + b * NP;
                int r = 0;
                for (; r + 1 < NP; r += 2) {
                    const double2 v = box[r], u = box[r + 1];
                    g0 += v.x; h0 += v.y; g1 += u.x; h1 += u.y;
                }
                if (r < NP) { const double2 v = box[r]; g0 += v.x; h0 += v.y; }
            }
            __syncwarp();
            // the mailbox has been read by every lane: re-arm it for position t+4
            if (lane == 0 && t + MBOX_DEPTH < d) mbar_arrive_expect_tx(smem_u32(&mbar[b]), 16u * (uint32_t)NP);
            const double tg = g0 + g1, th = h0 + h1;
            const int j0 = jf0 & 0x7fffffff;

            double pnew, upd;
            if (KIND == KIND_LINEAR) {
                double u = tg + ab * pold0;                       // cd_linear.py:19-22
                const double inv = mu * cn0 + ab;
                u = u / inv;
                pnew = pold0 - u;
                upd = u;
            } else {
                double inv = th * mu;                             // pcd.py:59-68 / pcd_all.py:34-41
                inv = inv + ab;
                double u = tg * lam;
                u = u + ab * pold0;
                u = u / inv;
                double p = pold0 - eta * u;
                double strength = eta * gamma / inv;
                const double a_old = fabs(pold0);
                if (reg == SP_REG_L1) {                           // l1.py:32-33
                    pnew = sp_soft_threshold(p, strength);
                } else if (reg == SP_REG_SQL12) {                 // squaredl12.py:52-57, :47-50
                    const double dcache = cache[0] - a_old;
                    p = p / (1.0 + 2.0 * strength);
                    const double sign = p > 0.0 ? 1.0 : -1.0;
                    double m = fabs(p) - 2.0 * strength * dcache / (1.0 + 2.0 * strength);
                    if (!(m > 0.0)) m = 0.0;
                    pnew = sign * m;
                    cache[0] = cache[0] - a_old;
                    cache[0] = cache[0] + fabs(pnew);
                } else {                                          // omegati.py:82-104
                    const double sign = p > 0.0 ? 1.0 : -1.0;
                    if (KIND == KIND_FM) {
                        double dc[DEG + 1];
                        dc[0] = 0.0; dc[1] = 1.0;
#pragma unroll
                        for (int deg = 2; deg <= DEG; deg++) {
                            double v = cache[deg - 1];
                            v = v - dc[deg - 1] * a_old;
                            if (v < 0.0) v = 0.0;
                            dc[deg] = v;
                        }
                        strength = strength * dc[DEG];
                        double m = fabs(p) - strength;
                        if (!(m > 0.0)) m = 0.0;
                        pnew = sign * m;
                        const double a_new = fabs(pnew);
#pragma unroll
                        for (int deg = 1; deg < DEG; deg++) cache[deg] = dc[deg + 1] + dc[deg] * a_new;
                    } else {
                        cache[0] = cache[0] / (1.0 + a_old);
                        strength = strength * cache[0];
                        double m = fabs(p) - strength;
                        if (!(m > 0.0)) m = 0.0;
                        pnew = sign * m;
                        cache[0] = cache[0] * (1.0 + fabs(pnew));
                    }
                }
                upd = pold0 - pnew;
            }
            viol += fabs(upd);
            if (lane == 0) {
                res[b] = make_double2(upd, pnew);
                asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&rbar[b])) : "memory");
                if (c == 0) a.prow[j0] = pnew;
            }
            meta_advance(t + 1);
        }
        if (c == 0 && lane == 0) {
            *a.viol = viol;
            if (KIND != KIND_LINEAR) {
#pragma unroll
                for (int t = 0; t < NC; t++) a.regstate[t] = cache[t];
            }
        }
    } else {
        // =============================================================== gather warps
        auto issue_idxval = [&](int q, int s, int e) {            // idx / value of position q -> stage q%3
            const int st3 = q % 3;
#pragma unroll
            for (int z = 0; z < NZ; z++) {
                const int g = s + z * T + tid;
                if (g < e) {
                    cp_async4(&idxbuf[(st3 * NZ + z) * T + tid], a.flag_idx + g);
                    cp_async8(&xbuf[(st3 * NZ + z) * T + tid], a.data + g);
                }
            }
        };
        auto issue_rec = [&](int q, int s, int e) {               // records of position q -> stage q%2
            const int st3 = q % 3, st2 = q & 1;
#pragma unroll
            for (int z = 0; z < NZ; z++) {
                if (s + z * T + tid < e) {
                    const int i = idxbuf[(st3 * NZ + z) * T + tid] & SP_ROW_MASK;
                    const double *src = a.rec + (size_t)i * stride;
#pragma unroll
                    for (int h = 0; h < NCH; h++)
                        cp_async16(&recbuf[((st2 * NZ + z) * NCH + h) * T + tid], src + 2 * h);
                }
            }
        };
        // pending position (terms computed, waiting for its scalar chain + write-back)
        int pi[NZ];
        double px[NZ], pr[NZ][R], pdA[NZ][ND];
#pragma unroll
        for (int z = 0; z < NZ; z++) pi[z] = -1;
        // gradient / curvature terms of position q; `late` = after the write-back of position q-1
        // (then bit31-tagged records are re-read as well)
        auto terms = [&](int q, int s, int e, double pold, bool late, double &tg, double &th) {
            const int st3 = q % 3, st2 = q & 1;
            tg = 0.0; th = 0.0;
#pragma unroll
            for (int z = 0; z < NZ; z++) {
                pi[z] = -1;
                if (s + z * T + tid < e) {
                    const int fi = idxbuf[(st3 * NZ + z) * T + tid];
                    const int i = fi & SP_ROW_MASK;
                    const unsigned stale = (unsigned)fi & (late ? (SP_FLAG_BIT | SP_FLAG2_BIT) : SP_FLAG2_BIT);
                    pi[z] = i;
                    px[z] = xbuf[(st3 * NZ + z) * T + tid];
                    if (stale) {
                        load_rec<R>(a.rec + (size_t)i * stride, pr[z]);
                    } else {
#pragma unroll
                        for (int h = 0; h < NCH; h++) {
                            const double2 v = recbuf[((st2 * NZ + z) * NCH + h) * T + tid];
                            pr[z][2 * h] = v.x;
                            if (2 * h + 1 < R) pr[z][2 * h + 1] = v.y;
                        }
                    }
                    nz_terms<KIND, DEG, LOSS, R, ND>(pr[z], px[z], pold, pdA[z], tg, th);
                }
            }
            for (int g = s + NZ * T + tid; g < e; g += T) {       // slices longer than NZ*T (rare)
                double rr[R], dd[ND];
                load_rec<R>(a.rec + (size_t)(a.flag_idx[g] & SP_ROW_MASK) * stride, rr);
                nz_terms<KIND, DEG, LOSS, R, ND>(rr, a.data[g], pold, dd, tg, th);
            }
            tg = sp_warp_allsum(tg);
            if (KIND != KIND_LINEAR) th = sp_warp_allsum(th);
        };
        // all-to-all: every gather warp writes its partial into every CTA's mailbox q%4
        auto push = [&](int q, double tg, double th) {
            const int b = q & (MBOX_DEPTH - 1);
            if (C > 1) {
                if (lane < C)
                    st_async_2f64(mapa_u32(smem_u32(&mbox[b * NP + c * W + warp]), (uint32_t)lane), tg, th,
                                  mapa_u32(smem_u32(&mbar[b]), (uint32_t)lane));
            } else if (lane == 0) {
                st_async_2f64(smem_u32(&mbox[b * NP + warp]), tg, th, smem_u32(&mbar[b]));
            }
        };
        auto gather_barrier = [&]() {
            if (W > 1) asm volatile("bar.sync 1, %0;" ::"r"(T) : "memory");
            else __syncwarp();
        };

        // ---- prologue
        int s0, e0, s1, e1, s2, e2, s3 = 0, e3 = 0;
        meta_se(0, s0, e0); meta_se(1, s1, e1); meta_se(2, s2, e2);
        int jf0, jf1 = 0;
        double pold0, cn0, pold1 = 0.0, cn1 = 0.0;
        meta_val(0, jf0, pold0, cn0);
        issue_idxval(0, s0, e0); issue_idxval(1, s1, e1); issue_idxval(2, s2, e2);
        cp_async_commit(); cp_async_wait_all();
        issue_rec(0, s0, e0); issue_rec(1, s1, e1);
        cp_async_commit(); cp_async_wait_all();
        if (d > 0) {
            double tg, th;
            terms(0, s0, e0, pold0, false, tg, th);
            push(0, tg, th);
        }
        for (int t = 0; t < d; t++) {
            // ---- staged data of t+1 (records) and t+2 (indices) has landed; stage the next ones
            cp_async_wait_all();
            meta_se(t + 3, s3, e3);
            issue_rec(t + 2, s2, e2);
            issue_idxval(t + 3, s3, e3);
            cp_async_commit();
            meta_val(t + 1, jf1, pold1, cn1);
            const bool have_next = t + 1 < d;
            const bool conf1 = jf1 < 0;
            // keep position t's pending registers: the terms of t+1 overwrite pi/px/pr/pdA
            int ci[NZ];
            double cx[NZ], cr[NZ][R], cdA[NZ][ND];
#pragma unroll
            for (int z = 0; z < NZ; z++) {
                ci[z] = pi[z]; cx[z] = px[z];
#pragma unroll
                for (int u = 0; u < R; u++) cr[z][u] = pr[z][u];
#pragma unroll
                for (int u = 0; u < ND; u++) cdA[z][u] = pdA[z][u];
            }
            // ---- early partial sums of t+1 (columns t and t+1 sample-disjoint)
            if (have_next && !conf1) {
                double tg, th;
                terms(t + 1, s1, e1, pold1, false, tg, th);
                push(t + 1, tg, th);
            }
            // ---- result of position t from the scalar warp, write-back
            const int b = t & (MBOX_DEPTH - 1);
            mbar_wait(smem_u32(&rbar[b]), (uint32_t)((t >> 2) & 1));
            const double2 rs = res[b];
            const double upd = rs.x, pnew = rs.y;
            if (KIND == KIND_ALL || upd != 0.0) {
#pragma unroll
                for (int z = 0; z < NZ; z++)
                    if (ci[z] >= 0)
                        nz_scatter<KIND, DEG, R, ND>(a.rec + (size_t)ci[z] * stride, cr[z], cdA[z], cx[z], lam, upd,
                                                     pold0, pnew);
                for (int g = s0 + NZ * T + tid; g < e0; g += T) {
                    double rr[R], dd[ND];
                    double *p = a.rec + (size_t)(a.flag_idx[g] & SP_ROW_MASK) * stride;
                    const double x = a.data[g];
                    load_rec<R>(p, rr);
                    dd[0] = x;
                    if (KIND == KIND_FM) {
#pragma unroll
                        for (int u = 1; u < ND; u++) dd[u] = x * (rr[1 + u] - pold0 * dd[u - 1]);
                    }
                    nz_scatter<KIND, DEG, R, ND>(p, rr, dd, x, lam, upd, pold0, pnew);
                }
            }
            // ---- the write-back must be visible before tagged records are re-read / re-staged
            gather_barrier();
            // ---- late partial sums of t+1 (the columns share samples)
            if (have_next && conf1) {
                double tg2, th2;
                terms(t + 1, s1, e1, pold1, true, tg2, th2);
                push(t + 1, tg2, th2);
            }
            s0 = s1; e0 = e1; s1 = s2; e1 = e2; s2 = s3; e2 = e3;
            jf0 = jf1; pold0 = pold1; cn0 = cn1;
            meta_advance(t + 1);
        }
        cp_async_wait_all();
    }
    __syncthreads();
    if (C > 1) cluster_sync_all();   // no CTA may exit while peers can still write its smem
}

// n_tab clusters of C CTAs run the device table
template <int KIND, int DEG, int LOSS, int NZ>
int launch_sweep(const SweepArgs *table, int n_tab, int C, int threads, cudaStream_t st) {
    constexpr int NA = (KIND == KIND_FM) ? DEG - 1 : (KIND == KIND_ALL ? 1 : 0);
    constexpr int NCH = (2 + NA + 1) / 2;
    const int W = threads / 32;
    const size_t smem = (size_t)2 * NZ * NCH * threads * 16 + (size_t)3 * NZ * threads * 8 +
                        (size_t)MBOX_DEPTH * C * W * 16 + (size_t)3 * NZ * threads * 4;
    auto kern = sweep_kernel<KIND, DEG, LOSS, NZ>;
    SP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (C > 8) SP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)C * (unsigned)n_tab, 1, 1);
    cfg.blockDim = dim3((unsigned)threads + 32, 1, 1);      // gather warps + the scalar-chain warp
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    sp_prof_begin(SP_PROF_SWEEP_PCD, st);
    cudaError_t le = cudaLaunchKernelEx(&cfg, kern, table, C);
    sp_prof_end(st);
    return sp_check_cuda(le, "sweep_kernel launch");
}

template <int KIND, int DEG>
int dispatch_loss(int loss, const SweepArgs *table, int n_tab, int C, int threads, int nz, cudaStream_t st) {
#define SP_DISPATCH_NZ(L)                                                                    \
    return nz >= 2 ? launch_sweep<KIND, DEG, L, 2>(table, n_tab, C, threads, st)             \
                   : launch_sweep<KIND, DEG, L, 1>(table, n_tab, C, threads, st)
    switch (loss) {
    case SP_LOSS_SQUARED: SP_DISPATCH_NZ(SP_LOSS_SQUARED);
    case SP_LOSS_LOGISTIC: SP_DISPATCH_NZ(SP_LOSS_LOGISTIC);
    case SP_LOSS_SQHINGE: SP_DISPATCH_NZ(SP_LOSS_SQHINGE);
    default: sp_set_error("unknown loss id %d", loss); return SP_ERR_INVALID;
    }
#undef SP_DISPATCH_NZ
}

int dispatch_degree(int degree, int loss, const SweepArgs *table, int n_tab, int C, int threads, int nz,
                    cudaStream_t st) {
    switch (degree) {
    case -1: return dispatch_loss<KIND_ALL, 1>(loss, table, n_tab, C, threads, nz, st);
    case 2: return dispatch_loss<KIND_FM, 2>(loss, table, n_tab, C, threads, nz, st);
    case 3: return dispatch_loss<KIND_FM, 3>(loss, table, n_tab, C, threads, nz, st);
    case 4: return dispatch_loss<KIND_FM, 4>(loss, table, n_tab, C, threads, nz, st);
    case 5: return dispatch_loss<KIND_FM, 5>(loss, table, n_tab, C, threads, nz, st);
    default: sp_set_error("pcd degree %d is not supported by the CUDA backend (2..%d or -1)", degree, SP_MAXDEG);
             return SP_ERR_UNSUPPORTED;
    }
}

// nonzeros per thread staged through shared memory: 2 when the mean slice exceeds the CTA
int pick_nz(const sp_dataset *ds, int n_cta, int threads) {
    const double avg = (double)ds->nnz / (ds->n_features > 0 ? ds->n_features : 1);
    return (avg / n_cta > 0.8 * threads) ? 2 : 1;
}

// flags[b*k + s] = 1 when row s of the [k,d] matrix Ps[b] has a nonzero entry (grid k x models)
__global__ void row_any_nonzero_kernel(const double *const *__restrict__ Ps, int d, int k, int *flags) {
    const double *row = Ps[blockIdx.y] + (size_t)blockIdx.x * d;
    __shared__ int s_any;
    if (threadIdx.x == 0) s_any = 0;
    __syncthreads();
    int any = 0;
    for (int j = threadIdx.x; j < d; j += blockDim.x) any |= (row[j] != 0.0);
    if (any) s_any = 1;
    __syncthreads();
    if (threadIdx.x == 0) flags[(size_t)blockIdx.y * k + blockIdx.x] = s_any;
}

// Pinned host staging of the argument tables (also used by pbcd.cu).  It is rewritten only after the copy that last
// read it has completed: `copied` is recorded behind every copy out of it.
struct Staging {
    unsigned char *host = nullptr;
    size_t cap = 0;
    cudaEvent_t copied = nullptr;
    int device = -1;
};
thread_local Staging g_stage;

}  // namespace

int sp_min_rec_stride(int degree) {   // record = {y_pred, y, A^1..A^{m-1}}, multiple of 4 doubles
    const int r = (degree == -1) ? 3 : (degree < 1 ? 2 : degree + 1);
    return (r + 3) & ~3;
}

extern "C" int sp_rec_stride(int degree) { return sp_min_rec_stride(degree); }

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

// ------------------------------------------------------------------------------------------------
// One order of a list of models on one design matrix (DESIGN.md 3.2).  Each launch covers all of them (one cluster,
// one row-DP block row, one regularizer-cache block per model), so the number of launches does not depend on the
// number of models; sp_pcd_epoch / sp_cd_linear_epoch run a list of one.  A window plan (one model only) replaces
// the cluster sweep by sp_wsweep.
namespace {

constexpr int MULTI_MAX_MODELS = 65535;   // gridDim.y of the row-DP and dead-scan launches

// The checks of every pcd / linear entry point.  A window plan needs only the order (idx_feat): SweepPlan leaves the
// cluster fields NULL then, and its geometry is not used.
int check_args(const sp_dataset *ds, int n_cta, int threads, const sp_wplan *win, const sp_pcd_model *models,
               int n_models, bool linear, int k, int degree, int loss, int rec_stride, const char *who) {
    if (!ds || n_models < 0 || n_models > MULTI_MAX_MODELS || (n_models > 0 && !models) || (win && n_models != 1)) {
        sp_set_error("%s: invalid argument (n_models must be 0..%d, 1 with a window plan)", who, MULTI_MAX_MODELS);
        return SP_ERR_INVALID;
    }
    if (!ds->csc_data || (win && !ds->csc_indptr) || (!linear && (k <= 0 || !ds->csr_indptr))) {
        sp_set_error("%s: invalid argument", who);
        return SP_ERR_INVALID;
    }
    if (!win && (n_cta < 1 || n_cta > SWEEP_MAX_CTAS || (n_cta & (n_cta - 1)))) {
        sp_set_error("%s: plan.n_cta must be a power of two in 1..%d", who, SWEEP_MAX_CTAS);
        return SP_ERR_INVALID;
    }
    if (!win && (threads < 32 || threads > SWEEP_MAX_THREADS || threads % 32)) {
        sp_set_error("%s: plan.threads must be a multiple of 32 in 32..%d", who, SWEEP_MAX_THREADS);
        return SP_ERR_INVALID;
    }
    for (int b = 0; b < n_models; b++) {
        const sp_pcd_model &m = models[b];
        if (!m.idx_feat || (!win && (!m.pos_ptr || !m.flag_idx || !m.pos_conf))) {
            sp_set_error("%s: dataset/plan pointers missing", who);
            return SP_ERR_INVALID;
        }
        if (!m.P || !m.rec || !m.viol || (!linear && (!m.lams || !m.regstate || !m.idx_comp_host))) {
            sp_set_error("%s: invalid argument (model %d)", who, b);
            return SP_ERR_INVALID;
        }
        if (linear) continue;
        // solver x regularizer x degree support matrix (reference README.md:25-31; the reference
        // fails with a numba TypingError / ValueError inside the jitclass for the others)
        if (m.reg != SP_REG_L1 && m.reg != SP_REG_SQL12 && m.reg != SP_REG_OMEGATI) {
            sp_set_error("regularizer id %d does not implement the pcd protocol (use l1, squaredl12 or omegati)", m.reg);
            return SP_ERR_UNSUPPORTED;
        }
        if (m.reg == SP_REG_SQL12 && degree != 2) {
            sp_set_error(degree == -1 ? "squaredl12 is not available for all-subsets models"
                                      : "SquaredL12 supports only degree=2.");
            return SP_ERR_UNSUPPORTED;
        }
        for (int ss = 0; ss < k; ss++) {
            const int s = m.idx_comp_host[ss];
            if (s < 0 || s >= k) {
                sp_set_error("%s: bad component index %d", who, s);
                return SP_ERR_INVALID;
            }
        }
    }
    if (!linear && !(degree == -1 || (degree >= 2 && degree <= SP_MAXDEG))) {
        sp_set_error("pcd degree %d is not supported by the CUDA backend (2..%d or -1)", degree, SP_MAXDEG);
        return SP_ERR_UNSUPPORTED;
    }
    if (rec_stride < (linear ? 2 : sp_min_rec_stride(degree)) || (rec_stride & 1)) {
        sp_set_error("%s: rec_stride %d too small for degree %d", who, rec_stride, linear ? 1 : degree);
        return SP_ERR_INVALID;
    }
    if (loss < SP_LOSS_SQUARED || loss > SP_LOSS_SQHINGE) { sp_set_error("unknown loss id %d", loss); return SP_ERR_INVALID; }
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

// the model a single-model entry point describes by its plan
sp_pcd_model plan_model(const sp_plan *plan) {
    sp_pcd_model m = {};
    m.pos_ptr = plan->pos_ptr; m.flag_idx = plan->flag_idx; m.idx_feat = plan->idx_feat; m.pos_conf = plan->pos_conf;
    return m;
}

int cd_linear_epoch(const sp_dataset *ds, int n_cta, int threads, const sp_wplan *win, const double *col_norm_sq,
                    const sp_pcd_model *models, int n_models, int loss, int rec_stride, cudaStream_t st,
                    const char *who) {
    int rc = check_args(ds, n_cta, threads, win, models, n_models, true, 0, 1, loss, rec_stride, who);
    if (rc) return rc;
    if (!col_norm_sq) {
        sp_set_error("%s: invalid argument", who);
        return SP_ERR_INVALID;
    }
    if (ds->n_features == 0 || n_models == 0) return SP_OK;
    if (win) {
        const sp_pcd_model &m = models[0];
        return sp_wsweep(ds, win, m.idx_feat, 1, m.P, col_norm_sq, nullptr, m.ab, 0.0, 1.0, SP_REG_L1, loss, m.rec,
                         rec_stride, m.viol, m.viol, st);
    }
    const size_t bytes = sizeof(SweepArgs) * n_models;
    unsigned char *h = nullptr;
    rc = sp_stage_acquire(bytes, &h);
    if (rc) return rc;
    SweepArgs *tab = reinterpret_cast<SweepArgs *>(h);
    for (int b = 0; b < n_models; b++) {
        SweepArgs a = model_args(ds, n_cta, models[b], rec_stride);
        a.prow = models[b].P; a.cns = col_norm_sq; a.lam_ptr = nullptr;
        a.gamma = 0.0; a.eta = 1.0; a.reg = SP_REG_L1; a.regstate = models[b].viol;
        tab[b] = a;
    }
    SweepArgs *dtab = nullptr;
    SP_CUDA(cudaMallocAsync((void **)&dtab, bytes, st));
    rc = sp_stage_upload(dtab, bytes, st);
    if (!rc)
        rc = dispatch_loss<KIND_LINEAR, 1>(loss, dtab, n_models, n_cta, threads, pick_nz(ds, n_cta, threads), st);
    cudaFreeAsync(dtab, st);
    return rc;
}

int pcd_epoch(const sp_dataset *ds, int n_cta, int threads, const sp_wplan *win, const sp_pcd_model *models,
              int n_models, int k, int degree, int loss, int rec_stride, cudaStream_t st, const char *who) {
    int rc = check_args(ds, n_cta, threads, win, models, n_models, false, k, degree, loss, rec_stride, who);
    if (rc) return rc;
    const int d = ds->n_features;
    if (d == 0 || n_models == 0) return SP_OK;

    // Dead components (ANOVA, degree >= 2, beta > 0): when row P[s,:] is entirely zero, A^t_i = 0 for every
    // t >= 1, so dA[m-1] = x (A^{m-1} - p dA[m-2]) = 0 on every nonzero, g = h = 0, the step is
    // (lams*0 + beta*0) / beta = 0 and the prox of 0 is 0 for l1 / squaredl12 / omegati: the reference's sweep
    // over that component (pcd.py:33-68, :92-135) changes nothing and adds 0 to the violation.  It is skipped
    // exactly; with beta == 0 the reference divides 0/0, so there the sweep runs as usual.  One scan of every
    // (model, component) row, one copy back and ONE stream synchronisation per call (the only one this library
    // makes inside an epoch).
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
            row_any_nonzero_kernel<<<dim3((unsigned)k, (unsigned)ns), 256, 0, st>>>(dP, d, k, flags);
            e1 = cudaGetLastError();
            if (e1 == cudaSuccess) e1 = cudaMemcpyAsync(f.data(), flags, sizeof(int) * ns * k, cudaMemcpyDeviceToHost, st);
            if (e1 == cudaSuccess) e1 = cudaStreamSynchronize(st);
        }
        cudaFreeAsync(buf, st);
        if (rc) return rc;
        if (e1 != cudaSuccess) return sp_check_cuda(e1, "dead-component scan");
        for (int i = 0; i < ns; i++)
            for (int s = 0; s < k; s++) alive[(size_t)scanned[i] * k + s] = f[(size_t)i * k + s];
    }

    // Tables, by position ss of the component order and then in model order: the sweep arguments and the
    // row-DP entries (one per live (model, component) pair, same index), the regularizer-cache entries
    // (pairs of models other than l1: l1 needs no cache).
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
    const int nz = win ? 1 : pick_nz(ds, n_cta, threads);
    for (int ss = 0; ss < k && !rc; ss++) {
        const int n = sw_off[ss + 1] - sw_off[ss], nr = rg_off[ss + 1] - rg_off[ss];
        if (n == 0) continue;
        rc = sp_rows_precompute_multi(ds, drw + sw_off[ss], n, degree, rec_stride, st);    // pcd.py:94 / pcd_all.py:65
        if (!rc && nr > 0) rc = sp_launch_reg_cache_multi(drg + rg_off[ss], nr, degree, d, st);   // pcd.py:96
        if (rc) break;
        if (win) {
            const SweepArgs &a = sw[sw_off[ss]];
            rc = sp_wsweep(ds, win, a.idx_feat, degree, a.prow, nullptr, a.lam_ptr, a.ab, a.gamma, a.eta, a.reg, loss,
                           a.rec, rec_stride, a.regstate, a.viol, st);
        } else {
            rc = dispatch_degree(degree, loss, dsw + sw_off[ss], n, n_cta, threads, nz, st);
        }
    }
    cudaFreeAsync(dbuf, st);
    return rc;
}

}  // namespace

extern "C" int sp_cd_linear_epoch(const sp_dataset *ds, const sp_plan *plan, double *w,
                                  const double *col_norm_sq, double alpha, int loss, double *rec,
                                  int rec_stride, double *viol, sp_stream stream) {
    if (!plan) { sp_set_error("sp_cd_linear_epoch: invalid argument"); return SP_ERR_INVALID; }
    sp_pcd_model m = plan_model(plan);
    m.P = w; m.ab = alpha; m.rec = rec; m.viol = viol;
    return cd_linear_epoch(ds, plan->n_cta, plan->threads, plan->win, col_norm_sq, &m, 1, loss, rec_stride,
                           (cudaStream_t)stream, "sp_cd_linear_epoch");
}

extern "C" int sp_pcd_epoch(const sp_dataset *ds, const sp_plan *plan, double *P_kd, int k,
                            const double *lams, int degree, double beta, double gamma, double eta,
                            int reg, int loss, double *rec, int rec_stride, double *regstate,
                            double *viol, const int32_t *idx_comp_host, sp_stream stream) {
    if (!plan) { sp_set_error("sp_pcd_epoch: invalid argument"); return SP_ERR_INVALID; }
    sp_pcd_model m = plan_model(plan);
    m.P = P_kd; m.lams = lams; m.ab = beta; m.gamma = gamma; m.eta = eta; m.reg = reg;
    m.rec = rec; m.regstate = regstate; m.viol = viol; m.idx_comp_host = idx_comp_host;
    return pcd_epoch(ds, plan->n_cta, plan->threads, plan->win, &m, 1, k, degree, loss, rec_stride,
                     (cudaStream_t)stream, "sp_pcd_epoch");
}

extern "C" int sp_cd_linear_epoch_multi(const sp_dataset *ds, int n_cta, int threads, const double *col_norm_sq,
                                        const sp_pcd_model *models, int n_models, int loss, int rec_stride,
                                        sp_stream stream) {
    return cd_linear_epoch(ds, n_cta, threads, nullptr, col_norm_sq, models, n_models, loss, rec_stride,
                           (cudaStream_t)stream, "sp_cd_linear_epoch_multi");
}

extern "C" int sp_pcd_epoch_multi(const sp_dataset *ds, int n_cta, int threads, const sp_pcd_model *models,
                                  int n_models, int k, int degree, int loss, int rec_stride, sp_stream stream) {
    return pcd_epoch(ds, n_cta, threads, nullptr, models, n_models, k, degree, loss, rec_stride, (cudaStream_t)stream,
                     "sp_pcd_epoch_multi");
}
