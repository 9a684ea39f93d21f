// Planned proximal minibatch SGD (reference optimizer/psgd.py:9-199) for the regularizers whose prox is
// a column-wise soft threshold: l1 (l1.py:50-51) and squaredl12 (squaredl12.py:66-78, utils.py:26-70).
//
// The reference scatters every sample's gradient into a dense grad_P [n_orders,d,k] and then sweeps
// P, grad_P and the prox over all d*k entries once per minibatch.  Here a minibatch is two GATHER
// passes over a precomputed plan and nothing is ever scattered:
//
//   rows  (psgd_rows_kernel)  one group of lanes per sample (lane = component): psgd._pred
//                             (psgd.py:47-57) -> the sample's ANOVA table rows A^1..A^(m-1) and
//                             dloss go to a small per-minibatch buffer (L2 resident);
//   cols  (psgd_cols_kernel)  the minibatch's nonzeros regrouped by feature (the "batch CSC" plan,
//                             built once per sample order): for every touched feature j the terms of
//                             psgd._update_grads (psgd.py:60-91) are summed in ascending sample order
//                             -- the reference's own order, no atomics, deterministic -- and the SGD
//                             step of psgd._update_params (psgd.py:94-117) is applied to row P[j,:]
//                             right there.  Work is cut into chunks of SP_PSGD_CHUNK nonzeros; a
//                             feature that spans several chunks (dense columns) leaves partial sums
//                             that psgd_split_kernel adds in chunk order.
//   untouched rows are never read or written by the step: the divisions by (1 + eta*beta) and the
//   prox thresholds are kept LAZY in a per-column frame  value = soft_threshold(raw, T_c) / C
//   (shrink-then-scale maps compose), so a minibatch rewrites only the rows it touches.
//   stats (psgd_stats_kernel) squaredl12 only: one read-only streaming pass over the raw matrix collects,
//                             per column, (count, sum) of |value| above a band around the predicted
//                             threshold and the band's values;
//   solve (psgd_solve_kernel) runs the fixed-point iteration tau <- 2 s S(tau) / (1 + 2 s C(tau)) over each
//                             band (members in registers, exact order-independent sums) to the (theta, S)
//                             that the reference's randomized-pivot search finds (utils.py:26-70); generic
//                             read-only passes when a band misses.
//
// Sharded over G ranks (one process per GPU, samples sharded, P sharded by rows j % G): the ranks PULL
// the raw rows their minibatch touches from the owners' HBM over NVLink peer memory (psgd_pull_kernel, on
// the context's own stream: minibatch m+1's rows travel while minibatch m's selection runs),
// PUSH their partial gradient rows into the owners' inboxes (cols kernel epilogue), the owner adds
// them in rank order and updates its rows (psgd_owner_kernel), and the column statistics are
// exchanged through peer memory as well -- no NCCL on the data path.
#include <cooperative_groups.h>
#include <math.h>
#include <stdlib.h>

#include <vector>

#include "common.cuh"
#include "sparsepoly_b200.h"

namespace cg = cooperative_groups;

namespace {

constexpr int PL_THREADS = 256;
constexpr int CH = SP_PSGD_CHUNK;
constexpr int BAND_CAP = SP_PSGD_BAND_CAP;          // band values per column and rank
constexpr int BAND_TOTAL = 2048;                    // band values per column over all ranks (shared memory)
constexpr int STAT_PART_MAX = 148 * 3;              // most blocks of the statistics pass
constexpr double BAND_DELTA = 0.02;
constexpr unsigned long long SPIN_TIMEOUT_NS = 20ull * 1000ull * 1000ull * 1000ull;

__device__ __forceinline__ double st_true(double r, double T, double invC) {
    double m = fabs(r) - T;                                  // value = soft_threshold(raw, T) / C
    if (!(m > 0.0)) return 0.0;
    m = m * invC;
    return r > 0.0 ? m : -m;
}
// raw representation of `v` in the frame (Cn, T)
__device__ __forceinline__ double to_raw(double v, double T, double Cn) {
    if (v == 0.0) return 0.0;
    const double a = fabs(v) * Cn + T;
    return v > 0.0 ? a : -a;
}

template <int DEG, int NORD> struct ARows {          // rows A^1..A^(deg_o-1) kept per sample, all orders
    static constexpr int value = (DEG - 1) + ARows<DEG - 1, NORD - 1>::value;
};
template <int DEG> struct ARows<DEG, 0> { static constexpr int value = 0; };
template <int DEG, int NORD> __device__ __forceinline__ constexpr int arow_off(int o) {
    int off = 0;
    for (int q = 0; q < o; q++) off += DEG - q - 1;
    return off;
}

template <int G> __device__ __forceinline__ unsigned group_mask() {
    return (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) & ~(G - 1)));
}

// ------------------------------------------------------------------------------------ rows
struct RowsArgs {
    int k, d;
    const int32_t *indptr, *colidx;      // colidx: feature ids, or (STAGED) slots in the minibatch's column list
    const double *data, *y;
    const double *Psrc, *wsrc;           // raw P [n_orders,d,k] / raw w [d]; STAGED: staged raw rows [U][n_orders][k] / [U]
    const double *lams, *thr;
    double invC, invCw;
    int loss, fit_linear;
    const int32_t *idx;
    int b0, b1;
    double *bufA, *bufdL, *sloss;        // [b1-b0][AROWS*k], [b1-b0], [n_local]
};

template <int DEG, int NORD, int G, int KCH, bool STAGED>
__global__ void __launch_bounds__(PL_THREADS, 3) psgd_rows_kernel(const RowsArgs a) {
    constexpr int AR = ARows<DEG, NORD>::value;
    const int lane = threadIdx.x & (G - 1);
    const unsigned gmask = group_mask<G>();
    const int gpb = PL_THREADS / G;
    const int n_groups = gridDim.x * gpb;
    const int k = a.k;
    const size_t dk = (size_t)a.d * k;
    // The inner loop is branch-free: lanes past a row's end carry (column 0, x = 0), whose terms vanish, and
    // lanes that own no component (s >= k) read a valid dummy address and are never written back.
    double lam[KCH], thr[KCH][NORD];
    const double *Pl[KCH][NORD];                       // lane's element of row 0 of every order
    const double invC = a.invC, invCw = a.invCw;
    const size_t rstride = STAGED ? (size_t)NORD * k : (size_t)k;
#pragma unroll
    for (int c = 0; c < KCH; c++) {
        const int s = lane + G * c;
        lam[c] = s < k ? a.lams[s] : 0.0;
#pragma unroll
        for (int o = 0; o < NORD; o++) {
            thr[c][o] = s < k ? a.thr[o * k + s] : 0.0;
            Pl[c][o] = a.Psrc + (s < k ? (STAGED ? (size_t)o * k + s : o * dk + s) : 0);
        }
    }
    const bool lin = a.fit_linear != 0;
    // software pipeline over the group's samples: (row bounds) of sample b + 2 n_groups and (first block of column
    // ids / values) of sample b + n_groups are in flight while sample b is processed
    const int bfirst = a.b0 + blockIdx.x * gpb + threadIdx.x / G;
    int i_c = 0, st_c = 0, en_c = 0, i_n = 0, st_n = 0, en_n = 0, i_nn = 0, st_nn = 0, en_nn = 0;
    int jl_c = 0, jl_n = 0;
    double xl_c = 0.0, xl_n = 0.0;
    if (bfirst < a.b1) { i_c = a.idx[bfirst]; st_c = a.indptr[i_c]; en_c = a.indptr[i_c + 1]; }
    if (bfirst + n_groups < a.b1) { i_n = a.idx[bfirst + n_groups]; st_n = a.indptr[i_n]; en_n = a.indptr[i_n + 1]; }
    if (st_c + lane < en_c) { jl_c = a.colidx[st_c + lane]; xl_c = a.data[st_c + lane]; }
    for (int b = bfirst; b < a.b1; b += n_groups) {
        const int i = i_c;
        const int st = st_c, en = en_c;
        // stage loads for the following samples
        i_nn = 0; st_nn = 0; en_nn = 0;
        if (b + 2 * n_groups < a.b1) { i_nn = a.idx[b + 2 * n_groups]; st_nn = a.indptr[i_nn]; en_nn = a.indptr[i_nn + 1]; }
        jl_n = 0; xl_n = 0.0;
        if (st_n + lane < en_n) { jl_n = a.colidx[st_n + lane]; xl_n = a.data[st_n + lane]; }
        double A[KCH][NORD][DEG + 1];
#pragma unroll
        for (int c = 0; c < KCH; c++)
#pragma unroll
            for (int o = 0; o < NORD; o++) {
                A[c][o][0] = 1.0;
#pragma unroll
                for (int t = 1; t <= DEG; t++) A[c][o][t] = 0.0;
            }
        double ypred = 0.0;                                   // _pred, psgd.py:47-57
        int jl = jl_c;
        double xl = xl_c;
        for (int base = st; base < en; base += G) {
            int jn = 0;                                       // the next block of (column, value): in flight during this one
            double xn = 0.0;
            if (base + G + lane < en) { jn = a.colidx[base + G + lane]; xn = a.data[base + G + lane]; }
            if (lin) ypred += xl * (a.wsrc[jl] * invCw);
            const int cnt = min(G, en - base);
            constexpr int UBR = 16 / (KCH * NORD);
            constexpr int UB = UBR >= 8 ? 8 : (UBR >= 4 ? 4 : (UBR >= 2 ? 2 : 1));
            for (int q0 = 0; q0 < cnt; q0 += UB) {
                double pv[UB][KCH][NORD], xv[UB];
#pragma unroll
                for (int u = 0; u < UB; u++) {                // UB independent row gathers in flight
                    const size_t at = (size_t)__shfl_sync(gmask, jl, q0 + u, G) * rstride;
                    xv[u] = __shfl_sync(gmask, xl, q0 + u, G);
#pragma unroll
                    for (int c = 0; c < KCH; c++)
#pragma unroll
                        for (int o = 0; o < NORD; o++) pv[u][c][o] = Pl[c][o][at];
                }
#pragma unroll
                for (int u = 0; u < UB; u++)
#pragma unroll
                    for (int c = 0; c < KCH; c++)
#pragma unroll
                        for (int o = 0; o < NORD; o++) {
                            const double p = st_true(pv[u][c][o], thr[c][o], invC);
#pragma unroll
                            for (int t = 0; t < DEG - o; t++)           // _anova, psgd.py:34-44
                                A[c][o][DEG - o - t] += (A[c][o][DEG - o - t - 1] * xv[u]) * p;
                        }
            }
            jl = jn; xl = xn;
        }
#pragma unroll
        for (int m = G / 2; m > 0; m >>= 1) ypred += __shfl_xor_sync(gmask, ypred, m, G);
#pragma unroll
        for (int o = 0; o < NORD; o++) {                      // y_pred += dot(lams, A[order, deg])
            double v = 0.0;
#pragma unroll
            for (int c = 0; c < KCH; c++) v += lam[c] * A[c][o][DEG - o];
#pragma unroll
            for (int m = G / 2; m > 0; m >>= 1) v += __shfl_xor_sync(gmask, v, m, G);
            ypred += v;
        }
        const double yi = a.y[i];
        double *row = a.bufA + (size_t)(b - a.b0) * AR * k;
#pragma unroll
        for (int c = 0; c < KCH; c++) {
            const int s = lane + G * c;
            if (s < k) {
#pragma unroll
                for (int o = 0; o < NORD; o++)
#pragma unroll
                    for (int t = 1; t < DEG - o; t++) row[(size_t)(arow_off<DEG, NORD>(o) + t - 1) * k + s] = A[c][o][t];
            }
        }
        if (lane == 0) {
            a.bufdL[b - a.b0] = sp_dloss_rt(a.loss, ypred, yi);
            a.sloss[b] = sp_loss_rt(a.loss, ypred, yi);        // psgd.py:155 (summed in fixed order at epoch end)
        }
        i_c = i_n; st_c = st_n; en_c = en_n; jl_c = jl_n; xl_c = xl_n;
        i_n = i_nn; st_n = st_nn; en_n = en_nn;
    }
}

// ------------------------------------------------------------------------------------ cols
enum { MODE_APPLY = 0, MODE_PUSH = 1 };

struct StepArgs {                        // psgd._update_params for one row (psgd.py:94-117) in the lazy frame
    double cP, denP, CnP;                // eta_P / batch, 1 + eta_P*beta, C * denP
    double cw, denw, Cnw;
    double rP, rw;                       // 1 / denP, 1 / denw (host, correctly rounded)
    double invC, invCw;                  // frame the rows are read in
    int fit_linear;
};

struct ColsArgs {
    int k, d;                            // d: rows of P (this rank's rows when sharded)
    const int32_t *e_pos;                // ABSOLUTE entry arrays: position of the sample inside its minibatch, value
    const double *e_x;
    const int32_t *u_feat;               // ABSOLUTE column arrays
    const int64_t *u_ptr;
    long long u_base;                    // absolute column offset of the minibatch
    const int32_t *sg_u, *sg_feat, *sg_pos;   // minibatch-relative lists: columns of ONE nonzero (column, feature, position,
    const double *sg_x;                       // value) ...
    int n_single;
    const int64_t *sc_ptr;               // ... short columns (2..SP_PSGD_SHORT nonzeros): offsets into the compact
    const int32_t *sc_u, *sc_feat, *sc_pos;   // nonzero arrays sc_pos / sc_x, column, feature ...
    const double *sc_x;
    int n_short;
    const int32_t *lc_u, *lc_feat, *lc_cnt;   // ... chunks of the long columns (column, feature, nonzeros | 2^30 when
    const int64_t *lc_e0;                     // the column has one chunk only, first nonzero) ...
    int n_chunks;
    const int32_t *ml_u, *ml_c0;         // ... and the long columns of several chunks (column, its first chunk)
    int n_multi;
    const double *bufA, *bufdL;
    const double *lams, *thr;
    double *P, *w;                       // APPLY: raw model (read + written)
    const double *stage, *stage_w;       // PUSH: staged true values [U][n_orders][k], [U]
    double *part_g, *part_w;             // partial sums of the chunks [n_chunks][n_orders*k], [n_chunks]
    StepArgs s;
    // PUSH: owner inboxes (peer memory)
    int world, rank;
    int owner_start[SP_MAX_RANKS + 1];   // first minibatch-relative column of every owner
    double *inbox_g[SP_MAX_RANKS];       // owner's inbox region of THIS rank: [cap][n_orders*k]
    double *inbox_w[SP_MAX_RANKS];       // [cap]
};

// v / den for a divisor that is the same for the whole minibatch: q = RN(v r), one fused residual correction
// (Markstein): the correctly rounded quotient, in 3 instructions instead of the ~35 of a generic fp64 division
__device__ __forceinline__ double div_const(double v, double den, double r) {
    const double q = v * r;
    const double rem = fma(-q, den, v);
    return fma(rem, r, q);
}

// psgd._update_params on one row: P = (P - (eta/b) g) / (1 + eta beta), written back in the frame (CnP, T)
template <int NORD, int G, int KCH>
__device__ __forceinline__ void apply_row(const StepArgs &s, double *P, double *w, int d, int k, int j, int lane,
                                          const double (&g)[KCH][NORD], double gw, const double (&pold)[KCH][NORD],
                                          double wraw, const double (&thr)[KCH][NORD]) {
    const size_t dk = (size_t)d * k;
#pragma unroll
    for (int c = 0; c < KCH; c++) {
        const int sidx = lane + G * c;
        if (sidx < k) {
#pragma unroll
            for (int o = 0; o < NORD; o++) {
                double gg = g[c][o] * s.cP;                 // grad *= eta / batch          psgd.py:113
                double v = pold[c][o] - gg;                 // P -= grad                    psgd.py:114
                v = div_const(v, s.denP, s.rP);             // P /= 1 + eta*beta            psgd.py:115
                P[o * dk + (size_t)j * k + sidx] = to_raw(v, thr[c][o], s.CnP);
            }
        }
    }
    if (s.fit_linear && lane == 0) {                        // psgd.py:109-112
        const double wold = wraw * s.invCw;                   // (raw value gathered together with the row)
        double gg = gw * s.cw;
        double v = wold - gg;
        v = div_const(v, s.denw, s.rw);
        w[j] = v * s.Cnw;
    }
}

// a column's gradient row is complete: apply the step (single rank) or push it to the owner's inbox
template <int NORD, int G, int KCH, int MODE>
__device__ __forceinline__ void finish_column(const ColsArgs &a, int lane, int ucol, int feat, const double (&g)[KCH][NORD],
                                              double gw, const double (&pold)[KCH][NORD], double wraw,
                                              const double (&thr)[KCH][NORD]) {
    const int k = a.k;
    if (MODE == MODE_APPLY) {
        apply_row<NORD, G, KCH>(a.s, a.P, a.w, a.d, k, feat, lane, g, gw, pold, wraw, thr);
    } else {
        const int su = (int)(ucol - a.u_base);
        const int owner = feat % a.world;
        const size_t at = (size_t)(su - a.owner_start[owner]);
        double *dst = a.inbox_g[owner] + at * NORD * k;
#pragma unroll
        for (int c = 0; c < KCH; c++) {
            const int sidx = lane + G * c;
            if (sidx < k) {
#pragma unroll
                for (int o = 0; o < NORD; o++) dst[o * k + sidx] = g[c][o];
            }
        }
        if (lane == 0) a.inbox_w[owner][at] = gw;
    }
}

// RAW gather of row `feat` (single rank) / of the staged raw row of slot `su` (sharded); row_values() turns
// the raw values into the true (pre-update) ones afterwards, so that the gathers of a batch are issued back to back
template <int NORD, int G, int KCH, int MODE>
__device__ __forceinline__ void load_row(const ColsArgs &a, int lane, int feat, long long su, double (&p)[KCH][NORD],
                                         double &wraw, const double (&thr)[KCH][NORD]) {
    const int k = a.k;
    const size_t dk = (size_t)a.d * k;
    wraw = (MODE == MODE_APPLY && a.s.fit_linear) ? a.w[feat] : 0.0;     // the row's w entry travels with it
#pragma unroll
    for (int c = 0; c < KCH; c++) {
        const int sidx = (lane + G * c) < k ? lane + G * c : 0;          // (lanes without a component: a valid dummy element)
#pragma unroll
        for (int o = 0; o < NORD; o++)
            p[c][o] = (MODE == MODE_APPLY) ? a.P[o * dk + (size_t)feat * k + sidx] : a.stage[((size_t)su * NORD + o) * k + sidx];
    }
    (void)thr;
}
template <int NORD, int G, int KCH, int MODE>
__device__ __forceinline__ void row_values(const ColsArgs &a, double (&p)[KCH][NORD], const double (&thr)[KCH][NORD]) {
#pragma unroll
    for (int c = 0; c < KCH; c++)
#pragma unroll
        for (int o = 0; o < NORD; o++) p[c][o] = st_true(p[c][o], thr[c][o], a.s.invC);
}

// one term of psgd._update_grads (psgd.py:60-91) for nonzero x of a sample with table rows av, dloss dl
template <int DEG, int NORD, int KCH, int AR>
__device__ __forceinline__ void add_term(double (&g)[KCH][NORD], double &gw, double x, double dl, const double (&av)[KCH][AR],
                                         const double (&pold)[KCH][NORD], const double (&lam)[KCH]) {
    gw += dl * x;                                             // psgd.py:86
#pragma unroll
    for (int c = 0; c < KCH; c++)
#pragma unroll
        for (int o = 0; o < NORD; o++) {
            double dprev = x;                                 // _grad_anova, psgd.py:25-31
#pragma unroll
            for (int t = 1; t < DEG - o; t++) dprev = x * (av[c][arow_off<DEG, NORD>(o) + t - 1] - pold[c][o] * dprev);
            g[c][o] += (dl * lam[c]) * dprev;                 // psgd.py:91
        }
}

// ---- columns of a single nonzero (70 % of a Criteo-shaped minibatch's columns): the plan stores (feature, position,
// value) per column, a group of G lanes fetches G of them at once and finishes UBC at a time -- row of P, table row
// and dloss of all UBC in flight together, no dependence between them
template <int DEG, int NORD, int G, int KCH, int MODE>
__device__ __forceinline__ void cols_single_part(const ColsArgs &a, int bidx, int nblk) {
    constexpr int AR = ARows<DEG, NORD>::value;
    constexpr int UBR = 8 / (KCH * (AR + NORD));                // (register budget: no spills at 3 blocks / SM)
    constexpr int UBC = UBR >= 4 ? 4 : (UBR >= 2 ? 2 : 1);
    const int lane = threadIdx.x & (G - 1);
    const unsigned gmask = group_mask<G>();
    const int gpb = PL_THREADS / G;
    const int k = a.k;
    double lam[KCH], thr[KCH][NORD];
    const double *Al[KCH];
#pragma unroll
    for (int c = 0; c < KCH; c++) {
        const int s = lane + G * c;
        lam[c] = s < k ? a.lams[s] : 0.0;
        Al[c] = a.bufA + (s < k ? s : 0);
#pragma unroll
        for (int o = 0; o < NORD; o++) thr[c][o] = s < k ? a.thr[o * k + s] : 0.0;
    }
    const size_t astride = (size_t)AR * k;
    for (int qb = (bidx * gpb + threadIdx.x / G) * G; qb < a.n_single; qb += nblk * gpb * G) {
        int u_l = (int)a.u_base, feat_l = 0, pos_l = 0;       // (lanes past the end: a valid dummy column, never finished)
        double x_l = 0.0;
        if (qb + lane < a.n_single) {
            u_l = a.sg_u[qb + lane]; feat_l = a.sg_feat[qb + lane]; pos_l = a.sg_pos[qb + lane]; x_l = a.sg_x[qb + lane];
        }
        const int ncol = (a.n_single - qb < G) ? a.n_single - qb : G;
        for (int c0 = 0; c0 < ncol; c0 += UBC) {
            double pold[UBC][KCH][NORD], av[UBC][KCH][AR], dl[UBC], xv[UBC], wraw[UBC];
            int uu[UBC], ff[UBC];
#pragma unroll
            for (int t = 0; t < UBC; t++) {                     // gathers of UBC columns in flight
                const int cc = (c0 + t) & (G - 1);
                uu[t] = __shfl_sync(gmask, u_l, cc, G);
                ff[t] = __shfl_sync(gmask, feat_l, cc, G);
                const int pos = __shfl_sync(gmask, pos_l, cc, G);
                xv[t] = __shfl_sync(gmask, x_l, cc, G);
                load_row<NORD, G, KCH, MODE>(a, lane, ff[t], uu[t] - a.u_base, pold[t], wraw[t], thr);
                dl[t] = a.bufdL[pos];
#pragma unroll
                for (int c = 0; c < KCH; c++)
#pragma unroll
                    for (int r = 0; r < AR; r++) av[t][c][r] = Al[c][(size_t)pos * astride + (size_t)r * k];
            }
#pragma unroll
            for (int t = 0; t < UBC; t++) {
                if (c0 + t >= ncol) break;
                double g[KCH][NORD];
                double gw = 0.0;
#pragma unroll
                for (int c = 0; c < KCH; c++)
#pragma unroll
                    for (int o = 0; o < NORD; o++) g[c][o] = 0.0;
                row_values<NORD, G, KCH, MODE>(a, pold[t], thr);
                add_term<DEG, NORD, KCH, AR>(g, gw, xv[t], dl[t], av[t], pold[t], lam);
                finish_column<NORD, G, KCH, MODE>(a, lane, uu[t], ff[t], g, gw, pold[t], wraw[t], thr);
            }
        }
    }
}

// ---- short columns (2..SP_PSGD_SHORT nonzeros; a quarter of a Criteo-shaped minibatch's columns).  The plan keeps
// their nonzeros in compact arrays (sc_ptr / sc_pos / sc_x), so a column's work is three dependent gathers:
// descriptor -> its nonzeros -> their table rows.  A group of lanes walks its columns with the three stages of
// three consecutive columns in flight (software pipeline): one memory round trip per column instead of three.
// Terms are added in sample order (the reference's).
template <int DEG, int NORD, int G, int KCH, int MODE>
__device__ __forceinline__ void cols_short_part(const ColsArgs &a, int bidx, int nblk) {
    constexpr int AR = ARows<DEG, NORD>::value;
    constexpr int SH = SP_PSGD_SHORT;
    static_assert(SH <= 8 && G >= 8, "a group's lanes hold a column's nonzeros");
    const int lane = threadIdx.x & (G - 1);
    const unsigned gmask = group_mask<G>();
    const int gpb = PL_THREADS / G;
    const int ngroups = nblk * gpb;
    const int k = a.k;
    double lam[KCH], thr[KCH][NORD];
    const double *Al[KCH];
#pragma unroll
    for (int c = 0; c < KCH; c++) {
        const int s = lane + G * c;
        lam[c] = s < k ? a.lams[s] : 0.0;
        Al[c] = a.bufA + (s < k ? s : 0);
#pragma unroll
        for (int o = 0; o < NORD; o++) thr[c][o] = s < k ? a.thr[o * k + s] : 0.0;
    }
    const size_t astride = (size_t)AR * k;
    const int q0 = bidx * gpb + threadIdx.x / G;
    // stage 1 (descriptor) of column q, stage 2 (nonzeros) of column q - ngroups, stage 3 (rows) of q - 2 ngroups
    long long p0_1 = 0, p0_2 = 0;
    int len_1 = 0, u_1 = 0, f_1 = 0, len_2 = 0, u_2 = 0, f_2 = 0, len_3 = 0, u_3 = 0, f_3 = 0;
    int ep_2 = 0;
    double ex_2 = 0.0;
    double pold[KCH][NORD], av[SH][KCH][AR], dl[SH], xv[SH], wraw = 0.0;
    for (int q = q0; q < a.n_short + 2 * ngroups; q += ngroups) {
        // ---- stage 3 loads: rows of the column whose nonzeros arrived in the previous iteration
        len_3 = len_2; u_3 = u_2; f_3 = f_2;
        if (len_3 > 0) {
            load_row<NORD, G, KCH, MODE>(a, lane, f_3, u_3 - a.u_base, pold, wraw, thr);
#pragma unroll
            for (int t = 0; t < SH; t++) {
                const int pos = __shfl_sync(gmask, ep_2, t, G);       // (nonzeros past the column's end: position 0, x = 0)
                xv[t] = __shfl_sync(gmask, ex_2, t, G);
                if (t < len_3) {
                    dl[t] = a.bufdL[pos];
#pragma unroll
                    for (int c = 0; c < KCH; c++)
#pragma unroll
                        for (int r = 0; r < AR; r++) av[t][c][r] = Al[c][(size_t)pos * astride + (size_t)r * k];
                }
            }
        }
        // ---- stage 2 loads: nonzeros of the column whose descriptor arrived in the previous iteration
        len_2 = len_1; u_2 = u_1; f_2 = f_1; p0_2 = p0_1;
        ep_2 = 0; ex_2 = 0.0;
        if (lane < len_2) { ep_2 = a.sc_pos[p0_2 + lane]; ex_2 = a.sc_x[p0_2 + lane]; }
        // ---- stage 1 loads: descriptor of column q
        len_1 = 0;
        if (q < a.n_short) {
            p0_1 = a.sc_ptr[q];
            len_1 = (int)(a.sc_ptr[q + 1] - p0_1);
            u_1 = a.sc_u[q];
            f_1 = a.sc_feat[q];
        }
        // ---- finish the stage-3 column
        if (len_3 > 0) {
            double g[KCH][NORD];
            double gw = 0.0;
#pragma unroll
            for (int c = 0; c < KCH; c++)
#pragma unroll
                for (int o = 0; o < NORD; o++) g[c][o] = 0.0;
            row_values<NORD, G, KCH, MODE>(a, pold, thr);
#pragma unroll
            for (int t = 0; t < SH; t++)
                if (t < len_3) add_term<DEG, NORD, KCH, AR>(g, gw, xv[t], dl[t], av[t], pold, lam);
            finish_column<NORD, G, KCH, MODE>(a, lane, u_3, f_3, g, gw, pold, wraw, thr);
        }
    }
}

// ---- long columns: cut into chunks of SP_PSGD_CHUNK nonzeros of ONE column -- a pure streaming sum, no column
// bookkeeping inside; the gathers of the next UB nonzeros are in flight while the current UB are being added.
// A column of one chunk is finished right here, the others leave one partial per chunk.
template <int DEG, int NORD, int G, int KCH, int MODE>
__global__ void __launch_bounds__(PL_THREADS, 2) psgd_cols_long_kernel(const ColsArgs a) {
    constexpr int AR = ARows<DEG, NORD>::value;
    constexpr int SETS = CH / G;                               // (position, value) pairs held per lane
    constexpr int UBR = 16 / (KCH * AR);
    constexpr int UB = UBR >= 8 ? 8 : (UBR >= 4 ? 4 : (UBR >= 2 ? 2 : 1));
    constexpr int NB = CH / UB;
    static_assert(G % UB == 0, "a batch never straddles two sets");
    const int lane = threadIdx.x & (G - 1);
    const unsigned gmask = group_mask<G>();
    const int gpb = PL_THREADS / G;
    const int chunk = blockIdx.x * gpb + threadIdx.x / G;
    if (chunk >= a.n_chunks) return;
    const int k = a.k;
    const int u = a.lc_u[chunk];
    const long long ce0 = a.lc_e0[chunk];
    const int cdesc = a.lc_cnt[chunk];
    const int cnt = cdesc & 0x3fffffff;
    const bool single = (cdesc & 0x40000000) != 0;
    const int feat = a.lc_feat[chunk];
    int ep[SETS];
    double ex[SETS];
#pragma unroll
    for (int sidx = 0; sidx < SETS; sidx++) {                  // nonzeros past the chunk's end: x = 0 and dloss = 0 below,
        const int q = sidx * G + lane;                         // so their terms vanish without a branch
        ep[sidx] = 0; ex[sidx] = 0.0;
        if (q < cnt) { ep[sidx] = a.e_pos[ce0 + q]; ex[sidx] = a.e_x[ce0 + q]; }
    }
    double lam[KCH], thr[KCH][NORD], pold[KCH][NORD], g[KCH][NORD];
    double gw = 0.0, wraw = 0.0;
#pragma unroll
    for (int c = 0; c < KCH; c++) {
        const int s = lane + G * c;
        lam[c] = s < k ? a.lams[s] : 0.0;
#pragma unroll
        for (int o = 0; o < NORD; o++) { thr[c][o] = s < k ? a.thr[o * k + s] : 0.0; g[c][o] = 0.0; }
    }
    load_row<NORD, G, KCH, MODE>(a, lane, feat, u - a.u_base, pold, wraw, thr);
    // nonzeros past the chunk's end carry (position 0, x = 0): every one of their terms is a product with x, so the
    // gathers below need no predicate; lanes that own no component read a valid dummy address and are not stored
    const double *Al[KCH];
#pragma unroll
    for (int c = 0; c < KCH; c++) Al[c] = a.bufA + ((lane + G * c) < k ? lane + G * c : 0);
    const size_t astride = (size_t)AR * k;
    double av[2][UB][KCH][AR], dl[2][UB], xv[2][UB];
    auto load_batch = [&](int buf, int b) {
#pragma unroll
        for (int t = 0; t < UB; t++) {
            const int q = b * UB + t;
            const int pos = __shfl_sync(gmask, ep[q / G], q & (G - 1), G);
            xv[buf][t] = __shfl_sync(gmask, ex[q / G], q & (G - 1), G);
            dl[buf][t] = a.bufdL[pos];
#pragma unroll
            for (int c = 0; c < KCH; c++)
#pragma unroll
                for (int r = 0; r < AR; r++) av[buf][t][c][r] = Al[c][(size_t)pos * astride + (size_t)r * k];
        }
    };
    auto add_batch = [&](int buf) {
#pragma unroll
        for (int t = 0; t < UB; t++) add_term<DEG, NORD, KCH, AR>(g, gw, xv[buf][t], dl[buf][t], av[buf][t], pold, lam);
    };
    load_batch(0, 0);
    row_values<NORD, G, KCH, MODE>(a, pold, thr);
#pragma unroll
    for (int b = 0; b < NB; b += 2) {
        if (b + 1 < NB && (b + 1) * UB < cnt) load_batch(1, b + 1);
        add_batch(0);
        if ((b + 1) * UB >= cnt) break;
        if (b + 2 < NB && (b + 2) * UB < cnt) load_batch(0, b + 2);
        add_batch(1);
        if ((b + 2) * UB >= cnt) break;
    }
    if (single) {
        finish_column<NORD, G, KCH, MODE>(a, lane, u, feat, g, gw, pold, wraw, thr);
    } else {
#pragma unroll
        for (int c = 0; c < KCH; c++) {
            const int s = lane + G * c;
            if (s < k) {
#pragma unroll
                for (int o = 0; o < NORD; o++) a.part_g[((size_t)chunk * NORD + o) * k + s] = g[c][o];
            }
        }
        if (lane == 0) a.part_w[chunk] = gw;
    }
}

// long columns of several chunks: one block per column adds the chunks' partial sums -- group w the chunks w,
// w+G', ... in order, then the groups' sums in group order (a fixed association: deterministic) -- and finishes it
constexpr int CB_THREADS = PL_THREADS;
template <int DEG, int NORD, int G, int KCH, int MODE>
__device__ __forceinline__ void cols_combine_part(const ColsArgs &a, int bidx, double *cb_sh) {
    constexpr int GPB = CB_THREADS / G;
    constexpr int ROW = KCH * G * NORD + 1;
    const int lane = threadIdx.x & (G - 1), grp = threadIdx.x / G;
    const int k = a.k;
    const int u = a.ml_u[bidx];
    const int c0 = a.ml_c0[bidx];
    const int np = (int)((a.u_ptr[u + 1] - a.u_ptr[u] + CH - 1) / CH);
    double g[KCH][NORD];
    double gw = 0.0;
#pragma unroll
    for (int c = 0; c < KCH; c++)
#pragma unroll
        for (int o = 0; o < NORD; o++) g[c][o] = 0.0;
    for (int pc = grp; pc < np; pc += GPB) {
        const size_t slot = (size_t)(c0 + pc);
#pragma unroll
        for (int c = 0; c < KCH; c++) {
            const int s = lane + G * c;
            if (s < k) {
#pragma unroll
                for (int o = 0; o < NORD; o++) g[c][o] += a.part_g[(slot * NORD + o) * k + s];
            }
        }
        gw += a.part_w[slot];
    }
#pragma unroll
    for (int c = 0; c < KCH; c++)
#pragma unroll
        for (int o = 0; o < NORD; o++) cb_sh[grp * ROW + (c * NORD + o) * G + lane] = g[c][o];
    if (lane == 0) cb_sh[grp * ROW + ROW - 1] = gw;
    __syncthreads();
    if (grp != 0) return;
    const int ngrp = np < GPB ? np : GPB;
    for (int w = 1; w < ngrp; w++) {
#pragma unroll
        for (int c = 0; c < KCH; c++)
#pragma unroll
            for (int o = 0; o < NORD; o++) g[c][o] += cb_sh[w * ROW + (c * NORD + o) * G + lane];
        gw += cb_sh[w * ROW + ROW - 1];
    }
    double thr[KCH][NORD], pold[KCH][NORD], wraw = 0.0;
#pragma unroll
    for (int c = 0; c < KCH; c++)
#pragma unroll
        for (int o = 0; o < NORD; o++) {
            const int s = lane + G * c;
            thr[c][o] = s < k ? a.thr[o * k + s] : 0.0;
        }
    const int feat = a.u_feat[u];
    load_row<NORD, G, KCH, MODE>(a, lane, feat, u - a.u_base, pold, wraw, thr);
    row_values<NORD, G, KCH, MODE>(a, pold, thr);
    finish_column<NORD, G, KCH, MODE>(a, lane, u, feat, g, gw, pold, wraw, thr);
}

// One launch for everything that follows the long-column chunks: blocks [0, n_multi) combine the multi-chunk
// columns (latency-bound: scheduled first, hidden behind the rest), the next nb_single blocks finish the
// single-nonzero columns, the remaining ones the short columns.
template <int DEG, int NORD, int G, int KCH, int MODE>
__global__ void __launch_bounds__(PL_THREADS, 3) psgd_cols_tail_kernel(const ColsArgs a, int nb_single, int nb_short) {
    constexpr int ROW = KCH * G * NORD + 1;
    __shared__ double cb_sh[(PL_THREADS / G) * ROW];
    const int b = blockIdx.x;
    if (b < a.n_multi) cols_combine_part<DEG, NORD, G, KCH, MODE>(a, b, cb_sh);
    else if (b < a.n_multi + nb_single) cols_single_part<DEG, NORD, G, KCH, MODE>(a, b - a.n_multi, nb_single);
    else cols_short_part<DEG, NORD, G, KCH, MODE>(a, b - a.n_multi - nb_single, nb_short);
}

// ------------------------------------------------------------------------------------ sharded: pull / owner
struct PullArgs {
    int k, d_own, world, n_cols;
    const int32_t *u_feat;               // the minibatch's columns (minibatch-relative pointer)
    const double *peer_P[SP_MAX_RANKS];  // owners' raw rows [n_orders][d_own][k]
    const double *peer_w[SP_MAX_RANKS];  // owners' raw w [d_own]
    int n_orders, fit_linear;
    double *stage, *stage_w;             // [n_cols][n_orders][k], [n_cols]
};

// RAW rows this rank's minibatch touches, read from the owners' HBM (NVLink peer loads; .cv: peer lines must
// not be served from a stale L1).  Raw, because the pull of minibatch m+1 runs on its own stream WHILE the
// selection of minibatch m runs: that only moves the frame (thresholds, scale), which the readers of the stage apply.  One warp per row batch, lane = element of the row, 8 rows in flight per
// warp: the latency of a peer load (~2 us) is covered by ~130 KB in flight per SM, so the pass is NVLink-bound.
__global__ void __launch_bounds__(PL_THREADS) psgd_pull_kernel(const PullArgs a) {
    const int k = a.k, rowlen = a.n_orders * k;
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = (gridDim.x * blockDim.x) >> 5;
    constexpr int UB = 8;
    for (int u0 = warp * UB; u0 < a.n_cols; u0 += nwarps * UB) {
        int jl = 0;
        if (lane < UB && u0 + lane < a.n_cols) jl = a.u_feat[u0 + lane];
        for (int e0 = 0; e0 < rowlen; e0 += 32) {
            const int e = e0 + lane;
            const int o = e / k, s = e - o * k;
            double raw[UB];
#pragma unroll
            for (int t = 0; t < UB; t++) {
                const int j = __shfl_sync(0xffffffffu, jl, t);
                const int owner = j % a.world, q = j / a.world;
                raw[t] = (e < rowlen && u0 + t < a.n_cols) ? __ldcv(a.peer_P[owner] + ((size_t)o * a.d_own + q) * k + s) : 0.0;
            }
            if (e < rowlen) {
#pragma unroll
                for (int t = 0; t < UB; t++)
                    if (u0 + t < a.n_cols) a.stage[(size_t)(u0 + t) * rowlen + e] = raw[t];
            }
        }
        if (a.fit_linear && lane < UB && u0 + lane < a.n_cols)
            a.stage_w[u0 + lane] = __ldcv(a.peer_w[jl % a.world] + jl / a.world);
    }
}

struct OwnerArgs {
    int k, d_own, world, n_rows;         // rows of this owner touched by the global minibatch
    const int32_t *own_q;                // [n_rows] local row index (feature / world)
    const int32_t *own_src;              // [n_rows][world] index in the inbox region of every rank, or -1
    const double *inbox_g[SP_MAX_RANKS]; // local inbox regions [cap][n_orders*k]
    const double *inbox_w[SP_MAX_RANKS];
    const double *thr;
    double *P, *w;
    StepArgs s;
};

// A group of lanes walks its rows: the next row's descriptor (local row, inbox index of every rank) is fetched while
// the current row's partial rows -- all ranks' at once, absent ranks contribute +0.0 -- are gathered and added in
// rank order (deterministic), then the step is applied.
template <int NORD, int G, int KCH>
__global__ void __launch_bounds__(PL_THREADS, 3) psgd_owner_kernel(const OwnerArgs a) {
    const int lane = threadIdx.x & (G - 1);
    const unsigned gmask = group_mask<G>();
    const int gpb = PL_THREADS / G;
    const int ngroups = gridDim.x * gpb;
    const int k = a.k, world = a.world;
    const size_t dk = (size_t)a.d_own * k;
    double thr[KCH][NORD];
#pragma unroll
    for (int c = 0; c < KCH; c++)
#pragma unroll
        for (int o = 0; o < NORD; o++) thr[c][o] = (lane + G * c) < k ? a.thr[o * k + lane + G * c] : 0.0;
    int r = blockIdx.x * gpb + threadIdx.x / G;
    int q_n = 0, at_n = -1;
    if (r < a.n_rows) {
        q_n = a.own_q[r];
        if (lane < world) at_n = a.own_src[(size_t)r * world + lane];
    }
    for (; r < a.n_rows; r += ngroups) {
        const int q = q_n, at_l = at_n;
        q_n = 0; at_n = -1;
        if (r + ngroups < a.n_rows) {
            q_n = a.own_q[r + ngroups];
            if (lane < world) at_n = a.own_src[(size_t)(r + ngroups) * world + lane];
        }
        double g[KCH][NORD], pold[KCH][NORD];
        double gw = 0.0;
        const double wraw = a.s.fit_linear ? a.w[q] : 0.0;
#pragma unroll
        for (int c = 0; c < KCH; c++)
#pragma unroll
            for (int o = 0; o < NORD; o++) {
                const int s = (lane + G * c) < k ? lane + G * c : 0;
                g[c][o] = 0.0;
                pold[c][o] = a.P[o * dk + (size_t)q * k + s];
            }
        constexpr int SB = 4;                                 // ranks gathered together
        for (int s0 = 0; s0 < world; s0 += SB) {
            double gi[SB][KCH][NORD], gwi[SB];
#pragma unroll
            for (int t = 0; t < SB; t++) {
                const int at = (s0 + t < world) ? __shfl_sync(gmask, at_l, (s0 + t) & (G - 1), G) : -1;
                gwi[t] = at >= 0 ? a.inbox_w[s0 + t][at] : 0.0;
#pragma unroll
                for (int c = 0; c < KCH; c++)
#pragma unroll
                    for (int o = 0; o < NORD; o++) {
                        const int s = (lane + G * c) < k ? lane + G * c : 0;
                        gi[t][c][o] = at >= 0 ? a.inbox_g[s0 + t][((size_t)at * NORD + o) * k + s] : 0.0;
                    }
            }
#pragma unroll
            for (int t = 0; t < SB; t++) {                    // fixed rank order
                gw += gwi[t];
#pragma unroll
                for (int c = 0; c < KCH; c++)
#pragma unroll
                    for (int o = 0; o < NORD; o++) g[c][o] += gi[t][c][o];
            }
        }
#pragma unroll
        for (int c = 0; c < KCH; c++)
#pragma unroll
            for (int o = 0; o < NORD; o++) pold[c][o] = st_true(pold[c][o], thr[c][o], a.s.invC);
        apply_row<NORD, G, KCH>(a.s, a.P, a.w, a.d_own, k, q, lane, g, gw, pold, wraw, thr);
    }
}

// ------------------------------------------------------------------------------------ cross-rank flags
struct XArgs {
    int world, rank, chan;
    unsigned long long seq;
    uint64_t *peer_flags[SP_MAX_RANKS];   // every rank's flag array [SP_PSGD_CHANNELS][SP_MAX_RANKS]
    uint64_t *my_flags;
    int *err;                                        // set to 1 on a timeout
};

__device__ __forceinline__ void flag_store(uint64_t *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long flag_load(const uint64_t *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ unsigned long long now_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// thread r < world: tell rank r that this rank reached `seq` on channel `chan`
__device__ __forceinline__ void x_signal(const XArgs &x, int r) {
    __threadfence_system();
    flag_store(x.peer_flags[r] + (size_t)x.chan * SP_MAX_RANKS + x.rank, x.seq);
}
// thread r < world: wait until rank r reached `seq`
__device__ __forceinline__ void x_wait(const XArgs &x, int r) {
    const uint64_t *f = x.my_flags + (size_t)x.chan * SP_MAX_RANKS + r;
    const unsigned long long t0 = now_ns();
    while (flag_load(f) < x.seq) {
        if (*reinterpret_cast<volatile int *>(x.err) != 0) break;      // a wait already timed out: do not stack timeouts
        __nanosleep(64);
        if (now_ns() - t0 > SPIN_TIMEOUT_NS) { *x.err = 1; break; }
    }
    __threadfence_system();
}
__global__ void psgd_xbarrier_kernel(const XArgs x) {       // signal + wait: everything the ranks wrote into
    const int r = threadIdx.x;                              // each other's memory before is visible after
    if (r < x.world) { x_signal(x, r); x_wait(x, r); }
}

// ------------------------------------------------------------------------------------ statistics + solve
// statbox of one source rank (doubles): sum[ncol] | cnt[ncol] | band_n[ncol] | band[ncol][BAND_CAP]
__host__ __device__ inline size_t statbox_doubles(size_t ncol) { return ncol * (3 + (size_t)BAND_CAP); }

struct StatArgs {
    const double *P;                     // raw rows [n_orders][d][k] (this rank's rows)
    int n_orders, d, k;
    double invC;                         // frame AFTER the update
    double strength;
    const double *thr;
    int reg;
    double *psum, *pcnt;                 // [STAT_PART_MAX][ncol] per-block partials
    double *band;                        // [ncol][BAND_CAP] (this rank)
    int *band_n;                         // [ncol] counters (zeroed before the launch) | [ncol] ticket
    double *state;                       // persistent: [0] previous strength, [1] calls, [2]/[3] band hits / generic
                                         // passes, [4] band half-width, [8+c] tau of the last call, [8+ncol+c] the one before
    double *tau;                         // [ncol] thresholds of the generic passes (value units); NULL: band pass
    int world, rank;
    double *statbox[SP_MAX_RANKS];       // every rank's statbox region of THIS rank (peer memory; [rank] is local)
    int *err;
};

__device__ __forceinline__ double predict_tau(const double *state, int ncol, int c, double strength) {
    const double last = state[8 + c], older = state[8 + ncol + c];
    double ratio = strength / state[0];
    if (state[1] >= 2.0 && older > 0.0) ratio = last / older;
    if (ratio < 0.5) ratio = 0.5;
    if (ratio > 2.0) ratio = 2.0;
    return last * ratio;
}

// One read-only pass over this rank's rows: per-block (sum, count) of the values above the statistics
// threshold of every column -- the band's upper edge (band pass) or a.tau[c] (generic pass) -- and, in a
// band pass, the values inside the band.  Partials are combined in fixed order.  VEC = 2: a thread owns two
// adjacent columns and streams 16-byte loads, 8 in flight (needs an even k); ssum / scnt hold VEC*blockDim.
constexpr int BAND_BLK = 16;                        // band values a block stages per column before one global reservation
template <int VEC>
__device__ __forceinline__ void stats_pass(const StatArgs &a, double *ssum, double *scnt, bool band_pass,
                                           int *s_bn = nullptr, double *s_bv = nullptr) {
    const int tid = threadIdx.x, T = blockDim.x, nblk = gridDim.x, k = a.k, d = a.d;
    const int ncol = a.n_orders * k;
    const int tpr = k / VEC;                        // threads per row (host: k <= 128, k % VEC == 0)
    const int rpp = T / tpr;
    const int cq = tid % tpr, row0 = tid / tpr;
    const bool act = tid < tpr * rpp;
    const double bdelta = a.state[4] > 0.0 ? a.state[4] : BAND_DELTA;
    for (int o = 0; o < a.n_orders; o++) {
        const double *P = a.P + (size_t)o * d * k;
        double Tc[VEC], hi[VEC], lo[VEC], lsum[VEC], lcnt[VEC];
        bool band_on[VEC];
        if (s_bn != nullptr) {                                 // per-block staging of the band values of this order's columns
            for (int c = tid; c < k; c += T) s_bn[c] = 0;
            __syncthreads();
        }
#pragma unroll
        for (int v = 0; v < VEC; v++) {
            const int cidx = o * k + (act ? cq * VEC + v : 0);
            Tc[v] = a.thr[cidx];
            band_on[v] = false;
            if (band_pass) {
                const double last = a.state[8 + cidx];
                band_on[v] = a.state[0] > 0.0 && a.strength > 0.0 && last > 0.0;
                const double tp = band_on[v] ? predict_tau(a.state, ncol, cidx, a.strength) : 0.0;
                hi[v] = band_on[v] ? tp * (1.0 + bdelta) : 0.0;
                lo[v] = band_on[v] ? tp * (1.0 - bdelta) : 0.0;
            } else {
                hi[v] = lo[v] = a.tau[cidx];
            }
            lsum[v] = 0.0; lcnt[v] = 0.0;
        }
        auto take = [&](double raw, int v) {                  // branch-free on the common paths (zero entry / counted entry)
            const double val = (fabs(raw) - Tc[v]) * a.invC;   // <= 0 for entries the lazy threshold has zeroed
            const bool above = val > hi[v];
            lsum[v] += above ? val : 0.0;
            lcnt[v] += above ? 1.0 : 0.0;
            if (band_on[v] && !above && val > lo[v]) {          // (rare: inside the band)
                const int cl = cq * VEC + v, cidx = o * k + cl;
                int sb = BAND_BLK;
                if (s_bn != nullptr) sb = atomicAdd(s_bn + cl, 1);          // shared-memory slot first: the global counter
                if (sb < BAND_BLK) s_bv[cl * BAND_BLK + sb] = val;          // of a column would serialise thousands of atomics
                else {
                    const int bi = atomicAdd(a.band_n + cidx, 1);
                    if (bi < BAND_CAP) a.band[(size_t)cidx * BAND_CAP + bi] = val;
                }
            }
        };
        if (act) {
            const long long step = (long long)nblk * rpp;
            long long r = (long long)blockIdx.x * rpp + row0;
            if (VEC == 2) {
                const double2 *P2 = reinterpret_cast<const double2 *>(P);
                const int k2 = k / 2;
                for (; r + 7 * step < d; r += 8 * step) {       // 8 independent 16-byte loads in flight
                    double2 rv[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) rv[u] = P2[(size_t)(r + u * step) * k2 + cq];
#pragma unroll
                    for (int u = 0; u < 8; u++) { take(rv[u].x, 0); take(rv[u].y, VEC - 1); }
                }
                for (; r < d; r += step) {
                    const double2 rv = P2[(size_t)r * k2 + cq];
                    take(rv.x, 0); take(rv.y, VEC - 1);
                }
            } else {
                for (; r + 7 * step < d; r += 8 * step) {
                    double rv[8];
#pragma unroll
                    for (int u = 0; u < 8; u++) rv[u] = P[(size_t)(r + u * step) * k + cq];
#pragma unroll
                    for (int u = 0; u < 8; u++) take(rv[u], 0);
                }
                for (; r < d; r += step) take(P[(size_t)r * k + cq], 0);
            }
        }
#pragma unroll
        for (int v = 0; v < VEC; v++) { ssum[v * T + tid] = lsum[v]; scnt[v * T + tid] = lcnt[v]; }
        __syncthreads();
        if (tid < k) {                                        // fixed-order combine over the block's rows
            const int q = tid / VEC, v = tid % VEC;
            double sm = 0.0, n = 0.0;
            for (int r = 0; r < rpp; r++) { sm += ssum[v * T + r * tpr + q]; n += scnt[v * T + r * tpr + q]; }
            a.psum[(size_t)blockIdx.x * ncol + o * k + tid] = sm;
            a.pcnt[(size_t)blockIdx.x * ncol + o * k + tid] = n;
            if (s_bn != nullptr) {                             // flush the block's staged band values: one reservation per column
                const int nb = s_bn[tid] < BAND_BLK ? s_bn[tid] : BAND_BLK;
                if (nb > 0) {
                    const int base = atomicAdd(a.band_n + o * k + tid, nb);
                    for (int q2 = 0; q2 < nb; q2++)
                        if (base + q2 < BAND_CAP) a.band[(size_t)(o * k + tid) * BAND_CAP + base + q2] = s_bv[tid * BAND_BLK + q2];
                }
            }
        }
        __syncthreads();
    }
}

// reduce the per-block partials of column cidx in fixed order (whole block cooperates)
__device__ __forceinline__ void reduce_partials(const StatArgs &a, int cidx, int npart, double *ssum, double *scnt,
                                                double *osum, double *ocnt) {
    const int tid = threadIdx.x, T = blockDim.x;
    const int ncol = a.n_orders * a.k;
    double s = 0.0, n = 0.0;
    for (int b = tid; b < npart; b += T) { s += a.psum[(size_t)b * ncol + cidx]; n += a.pcnt[(size_t)b * ncol + cidx]; }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) { s += __shfl_down_sync(0xffffffffu, s, off); n += __shfl_down_sync(0xffffffffu, n, off); }
    if ((tid & 31) == 0) { ssum[tid >> 5] = s; scnt[tid >> 5] = n; }
    __syncthreads();
    s = 0.0; n = 0.0;
    for (int w = 0; w < T / 32; w++) { s += ssum[w]; n += scnt[w]; }
    *osum = s; *ocnt = n;
    __syncthreads();
}

// band pass as its own streaming launch
__global__ void __launch_bounds__(PL_THREADS, 3) psgd_stats_kernel(const StatArgs a) {
    __shared__ double ssum[2 * PL_THREADS], scnt[2 * PL_THREADS];
    __shared__ int s_bn[128];                                  // (k <= 128)
    __shared__ double s_bv[128 * BAND_BLK];
    if ((a.k & 1) == 0) stats_pass<2>(a, ssum, scnt, true, s_bn, s_bv);
    else stats_pass<1>(a, ssum, scnt, true, s_bn, s_bv);
}

// sharded: block c reduces column c's partials (fixed order) and publishes this rank's statistics + band to
// every rank's statbox; the band counter is reset for the next minibatch
__global__ void __launch_bounds__(PL_THREADS) psgd_stats_publish_kernel(const StatArgs a, int npart) {
    __shared__ double ssum[PL_THREADS], scnt[PL_THREADS];
    const int ncol = a.n_orders * a.k, cidx = blockIdx.x;
    double s, n;
    reduce_partials(a, cidx, npart, ssum, scnt, &s, &n);
    const int nb = a.band_n[cidx];
    const int nv = nb < BAND_CAP ? nb : BAND_CAP;
    for (int r = 0; r < a.world; r++) {
        double *box = a.statbox[r];
        if (threadIdx.x == 0) { box[cidx] = s; box[ncol + cidx] = n; box[2 * ncol + cidx] = (double)nb; }
        for (int q = threadIdx.x; q < nv; q += blockDim.x)
            box[3 * (size_t)ncol + (size_t)cidx * BAND_CAP + q] = a.band[(size_t)cidx * BAND_CAP + q];
    }
    __syncthreads();
    if (threadIdx.x == 0) a.band_n[cidx] = 0;
}

struct SolveArgs {
    StatArgs st;                         // generic passes reuse the statistics pass (st.tau = tau)
    double Cn;                           // frame scale after the update: T[c] += Cn * tau[c]
    double *thr;                         // [ncol] raw-space thresholds (updated)
    double *tau;                         // [ncol] scratch: new thresholds in value units
    double *colres;                      // [2*ncol] reduced (sum, cnt) of a generic pass
    int *fail;                           // [2] = call_id when a column could not use its band / overflowed in THIS call
    int call_id;                         // > 0, different in every call (no reset between launches)
    int npart;                           // single rank: rows of st.psum / st.pcnt the statistics pass wrote
    const double *statbox_all;           // local statboxes of all ranks [world][statbox_doubles]
    double *xbuf[SP_MAX_RANKS];          // every rank's exchange buffer region of THIS rank [2][2*ncol] (generic passes)
    const double *xbuf_local;            // local exchange buffers of all ranks [world][2][2*ncol]
    XArgs x;                             // channel of the generic-pass exchanges (seq = first free sequence number)
    unsigned long long *seq_out;         // device counter: sequence numbers consumed (host adds a bound instead)
    int max_iter;
};

constexpr int SOLVE_THREADS = 512;

__global__ void __launch_bounds__(SOLVE_THREADS) psgd_solve_kernel(const SolveArgs a) {
    cg::grid_group grid = cg::this_grid();
    __shared__ double ssum[SOLVE_THREADS], scnt[SOLVE_THREADS];
    __shared__ double sband[BAND_TOTAL];
    __shared__ uint4 sred[2 * (SOLVE_THREADS / 32)];
    const StatArgs &st = a.st;
    const int tid = threadIdx.x, T = SOLVE_THREADS, nblk = gridDim.x;
    const int ncol = st.n_orders * st.k, world = st.world;
    const size_t boxlen = statbox_doubles(ncol);
    const double bdelta = st.state[4] > 0.0 ? st.state[4] : BAND_DELTA;
    const bool band_on = st.state[0] > 0.0 && st.strength > 0.0;
    // ---- band path: every column's fixed point from (statistics above the band) + (the band's values)
    if (!band_on) {
        if (blockIdx.x == 0) {
            if (tid == 0) a.fail[0] = a.call_id;
            if (world == 1) for (int c = tid; c < ncol; c += T) st.band_n[c] = 0;
        }
    } else {
        for (int cidx = blockIdx.x; cidx < ncol; cidx += nblk) {
            double sumA = 0.0, cntA = 0.0;
            int nbv = 0;
            bool ok = st.state[8 + cidx] > 0.0;
            if (world == 1) {                                    // partials + band straight from the statistics pass
                reduce_partials(st, cidx, a.npart, ssum, scnt, &sumA, &cntA);
                const int nb = st.band_n[cidx];
                if (nb > BAND_CAP) { ok = false; if (tid == 0) a.fail[1] = a.call_id; }
                nbv = nb < BAND_CAP ? nb : BAND_CAP;
            } else {
                for (int r = 0; r < world; r++) {                // rank order: identical on every rank
                    const double *box = a.statbox_all + (size_t)r * boxlen;
                    sumA += box[cidx]; cntA += box[ncol + cidx];
                    const int nb = (int)box[2 * ncol + cidx];
                    if (nb > BAND_CAP) { ok = false; if (tid == 0) a.fail[1] = a.call_id; }
                    nbv += nb < BAND_CAP ? nb : BAND_CAP;
                }
            }
            if (nbv > BAND_TOTAL) { ok = false; if (tid == 0) a.fail[1] = a.call_id; }
            if (tid == 0) st.state[8 + 2 * ncol + cidx] = (double)nbv;
            if (ok) {
                const double tau_pred = predict_tau(st.state, ncol, cidx, st.strength);
                const double b_hi = tau_pred * (1.0 + bdelta), b_lo = tau_pred * (1.0 - bdelta);
                if (world == 1) {
                    for (int q = tid; q < nbv; q += T) sband[q] = st.band[(size_t)cidx * BAND_CAP + q];
                } else {
                    int at = 0;
                    for (int r = 0; r < world; r++) {
                        const double *box = a.statbox_all + (size_t)r * boxlen;
                        const int nb0 = (int)box[2 * ncol + cidx];
                        const int nb = nb0 < BAND_CAP ? nb0 : BAND_CAP;
                        for (int q = tid; q < nb; q += T) sband[at + q] = box[3 * (size_t)ncol + (size_t)cidx * BAND_CAP + q];
                        at += nb;
                    }
                }
                __syncthreads();
                // The prox keeps the values above tau = 2 s S / (1 + 2 s theta), S / theta the sum / number of the kept
                // values (utils.py:26-70).  Everything above the band is kept whenever tau lands inside the band, so
                // only the band's members are undecided: start with all of them kept and drop the ones at or below
                // tau until none drops (the kept set only shrinks, tau only rises, and the fixed point is the set
                // utils.py selects).  The band arrives in no particular order (atomic reservations), so its sums
                // are taken EXACTLY: all members lie in (2^(E-2), 2^E) -- the band is at most +-10 % wide -- hence
                // v * 2^(54-E) is an integer below 2^54, summed as three 18-bit limbs in 32-bit integers
                // (<= 2048 members) and rounded once.  The result does not depend on the order.
                constexpr int VPT = BAND_TOTAL / SOLVE_THREADS;
                const int E = ilogb(b_hi) + 1;
                const double up = scalbn(1.0, 54 - E), down = scalbn(1.0, E - 54);
                const double vmin = scalbn(1.0, E - 2), vmax = scalbn(1.0, E);
                double bv[VPT];
                unsigned l0[VPT], l1[VPT], l2[VPT];
                bool bad = !(bdelta <= 0.1) || E - 54 < -1000 || 54 - E < -1000;
#pragma unroll
                for (int i = 0; i < VPT; i++) {
                    const int q = tid + i * T;
                    bv[i] = -1.0; l0[i] = l1[i] = l2[i] = 0u;
                    if (q < nbv) {
                        const double b = sband[q];
                        if (!(b > vmin && b < vmax)) bad = true;
                        else {
                            const unsigned long long I = (unsigned long long)(b * up);
                            bv[i] = b;
                            l0[i] = (unsigned)(I & 0x3ffffull); l1[i] = (unsigned)((I >> 18) & 0x3ffffull); l2[i] = (unsigned)(I >> 36);
                        }
                    }
                }
                double tau = b_lo;                                   // every member of the band is above b_lo
                int prev_n = -1;
                bool conv = false;
                for (int iter = 0; iter < 64; iter++) {
                    unsigned c = bad ? 1u << 20 : 0u, s0 = 0u, s1 = 0u, s2 = 0u;
#pragma unroll
                    for (int i = 0; i < VPT; i++) {
                        const bool act = bv[i] > tau;
                        c += act ? 1u : 0u; s0 += act ? l0[i] : 0u; s1 += act ? l1[i] : 0u; s2 += act ? l2[i] : 0u;
                    }
                    c = __reduce_add_sync(0xffffffffu, c); s0 = __reduce_add_sync(0xffffffffu, s0);
                    s1 = __reduce_add_sync(0xffffffffu, s1); s2 = __reduce_add_sync(0xffffffffu, s2);
                    uint4 *red = sred + (iter & 1) * (SOLVE_THREADS / 32);
                    if ((tid & 31) == 0) red[tid >> 5] = make_uint4(c, s0, s1, s2);
                    __syncthreads();
                    unsigned long long t0 = 0, t1 = 0, t2 = 0;
                    unsigned n = 0;
#pragma unroll
                    for (int w = 0; w < SOLVE_THREADS / 32; w++) { const uint4 r = red[w]; n += r.x; t0 += r.y; t1 += r.z; t2 += r.w; }
                    if (n >= (1u << 20)) break;                        // a member outside the exact range: generic path
                    if ((int)n == prev_n) { conv = true; break; }      // nothing dropped: tau is the fixed point
                    prev_n = (int)n;
                    const double sum = ((double)t2 * 68719476736.0 + (double)((t1 << 18) + t0)) * down;
                    tau = 2.0 * st.strength * (sumA + sum) / (1.0 + 2.0 * st.strength * (cntA + (double)n));
                }
                ok = conv && tau > b_lo && tau <= b_hi;
                if (ok && tid == 0) a.tau[cidx] = tau;
                __syncthreads();
            }
            if (!ok && tid == 0) a.fail[0] = a.call_id;
            if (world == 1) {                                    // this column's band counter: ready for the next minibatch
                __syncthreads();                                 // (only the block that owns the column touches it)
                if (tid == 0) st.band_n[cidx] = 0;
            }
        }
    }
    __threadfence();
    grid.sync();
    const bool fb = *reinterpret_cast<volatile int *>(a.fail) == a.call_id;
    const bool over = *reinterpret_cast<volatile int *>(a.fail + 1) == a.call_id;
    if (!fb) {
        if (blockIdx.x == 0) {
            for (int c = tid; c < ncol; c += T) {
                st.state[8 + ncol + c] = st.state[8 + c];
                st.state[8 + c] = a.tau[c];
                a.thr[c] = a.thr[c] + a.Cn * a.tau[c];
            }
            if (tid == 0) { st.state[0] = st.strength; st.state[1] += 1.0; st.state[2] += 1.0; }
        }
        return;
    }
    // ---- generic path: Michelot iteration from tau = 0 with one read-only pass per step; the active set
    //      {v > tau} only shrinks and tau rises monotonically to the fixed point the reference finds
    for (int c = blockIdx.x * T + tid; c < ncol; c += nblk * T) a.tau[c] = 0.0;
    __threadfence();
    grid.sync();
    StatArgs sp = st;
    sp.tau = a.tau;
    double prev_total = -1.0;
    XArgs x = a.x;
    for (int it = 0; it < a.max_iter; it++) {
        stats_pass<1>(sp, ssum, scnt, false);
        __threadfence();
        grid.sync();
        for (int cidx = blockIdx.x; cidx < ncol; cidx += nblk) {
            double s, n;
            reduce_partials(sp, cidx, nblk, ssum, scnt, &s, &n);
            if (tid == 0) { a.colres[cidx] = s; a.colres[ncol + cidx] = n; }
        }
        __threadfence();
        grid.sync();
        if (world > 1) {                                            // sum over the ranks through peer memory
            const int par = it & 1;
            if (blockIdx.x == 0) {
                for (int r = 0; r < world; r++)
                    for (int q = tid; q < 2 * ncol; q += T) a.xbuf[r][(size_t)par * 2 * ncol + q] = a.colres[q];
                __threadfence_system();
                __syncthreads();
                if (tid < world) { x_signal(x, tid); x_wait(x, tid); }
                __syncthreads();
            }
            x.seq += 1;
            grid.sync();
        }
        // every block derives the same new thresholds and the same convergence decision
        double total = 0.0;
        for (int c = tid; c < ncol; c += T) {
            double s = 0.0, n = 0.0;
            if (world > 1) {
                for (int r = 0; r < world; r++) {
                    const double *xb = a.xbuf_local + ((size_t)r * 2 + (it & 1)) * 2 * ncol;
                    s += __ldcg(xb + c); n += __ldcg(xb + ncol + c);
                }
            } else { s = a.colres[c]; n = a.colres[ncol + c]; }
            total += n;
            if (blockIdx.x == 0) a.tau[c] = 2.0 * st.strength * s / (1.0 + 2.0 * st.strength * n);   // = 2*strength*S (utils.py:69-70)
        }
        ssum[tid] = total;
        __syncthreads();
        for (int off = T / 2; off > 0; off >>= 1) { if (tid < off) ssum[tid] += ssum[tid + off]; __syncthreads(); }
        total = ssum[0];
        __syncthreads();
        __threadfence();
        grid.sync();
        if (total == prev_total) break;                           // no column lost an element: fixed point
        prev_total = total;
    }
    if (blockIdx.x == 0) {
        for (int c = tid; c < ncol; c += T) {
            st.state[8 + ncol + c] = st.state[8 + c];
            st.state[8 + c] = a.tau[c];
            a.thr[c] = a.thr[c] + a.Cn * a.tau[c];
        }
        if (tid == 0) {
            st.state[0] = st.strength; st.state[1] += 1.0; st.state[3] += 1.0;
            if (band_on) {                                          // adapt the band's half-width
                double nd = over ? bdelta * 0.5 : bdelta * 2.0;
                if (nd < 0.002) nd = 0.002;
                if (nd > 0.1) nd = 0.1;
                st.state[4] = nd;
            }
        }
    }
}

// l1: every column's threshold is `strength` (l1.py:50-51)
__global__ void psgd_thr_advance_kernel(double *thr, int ncol, double add) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c < ncol) thr[c] = thr[c] + add;
}

// P <- true values (soft_threshold(raw, T) / C), w likewise; thresholds back to 0: the stored matrix is
// the model again
__global__ void psgd_materialize_kernel(double *P, int n_orders, size_t d, int k, const double *thr, double invC,
                                        double *w, double invCw, int fit_linear) {
    const size_t n = (size_t)n_orders * d * k, stride = (size_t)gridDim.x * blockDim.x;
    for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
        const int o = (int)(e / (d * k));
        P[e] = st_true(P[e], thr[o * k + (int)(e % k)], invC);
    }
    if (fit_linear)
        for (size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x; e < d; e += stride) w[e] = w[e] * invCw;
}
// the model the frame represents, written out in the component-major [n_orders, k, d] layout of P_: a 32 x 32 tile
// of (feature, component) per block, read along k and written along d; the value expressions are those of
// psgd_materialize_kernel, so the result equals materialise + transpose bit for bit
constexpr int READ_TILE = 32, READ_ROWS = 8;
__global__ void psgd_read_kernel(const double *P, int d, int k, const double *thr, double invC, double *P_out) {
    __shared__ double tile[READ_TILE][READ_TILE + 1];
    const int o = blockIdx.z, s = blockIdx.y * READ_TILE + threadIdx.x;
    const long long j0 = (long long)blockIdx.x * READ_TILE;
    const double *Po = P + (size_t)o * d * k;
    if (s < k) {
        const double T = thr[o * k + s];
        for (int r = threadIdx.y; r < READ_TILE; r += READ_ROWS) {
            const long long j = j0 + r;
            if (j < d) tile[r][threadIdx.x] = st_true(Po[(size_t)j * k + s], T, invC);
        }
    }
    __syncthreads();
    const long long j = j0 + threadIdx.x;
    if (j < d)
        for (int r = threadIdx.y; r < READ_TILE; r += READ_ROWS) {
            const int s2 = blockIdx.y * READ_TILE + r;
            if (s2 < k) P_out[((size_t)o * k + s2) * d + j] = tile[threadIdx.x][r];
        }
}
__global__ void psgd_read_w_kernel(const double *w, int d, double invCw, int fit_linear, double *w_out) {
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < d; j += gridDim.x * blockDim.x)
        w_out[j] = fit_linear ? w[j] * invCw : w[j];
}
__global__ void psgd_zero_kernel(double *p, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = 0.0;
}

// fixed-order sum of the per-sample losses of positions [b0, b1) (epoch end): LOSS_BLOCKS grid-strided block sums,
// then one block adds them to *out -- the same association for the same n on every run
constexpr int LOSS_BLOCKS = 148;
__global__ void __launch_bounds__(1024) psgd_loss_part_kernel(const double *sloss, long long b0, long long b1, double *part) {
    __shared__ double sh[1024];
    double acc = 0.0;
    for (long long b = b0 + (long long)blockIdx.x * 1024 + threadIdx.x; b < b1; b += (long long)LOSS_BLOCKS * 1024) acc += sloss[b];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int off = 512; off > 0; off >>= 1) { if ((int)threadIdx.x < off) sh[threadIdx.x] += sh[threadIdx.x + off]; __syncthreads(); }
    if (threadIdx.x == 0) part[blockIdx.x] = sh[0];
}
__global__ void __launch_bounds__(256) psgd_loss_sum_kernel(const double *part, double *out) {
    __shared__ double sh[256];
    sh[threadIdx.x] = (int)threadIdx.x < LOSS_BLOCKS ? part[threadIdx.x] : 0.0;
    __syncthreads();
    for (int off = 128; off > 0; off >>= 1) { if ((int)threadIdx.x < off) sh[threadIdx.x] += sh[threadIdx.x + off]; __syncthreads(); }
    if (threadIdx.x == 0) out[0] = out[0] + sh[0];
}

int grid_for(long long groups, int G) {
    const int gpb = PL_THREADS / G;
    long long blocks = (groups + gpb - 1) / gpb;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

}  // namespace

// ============================================================================================ host side
struct PlanMb {                          // one minibatch of the plan, resolved on the host
    long long e0, e1, u0, u1, sg0, sg1, sh0, sh1, lc0, lc1, ml0, ml1;
    int b0, b1;
};

static inline PlanMb plan_mb(const sp_psgd_plan *pl, int m) {
    PlanMb q;
    q.e0 = pl->mb_eptr_host[m]; q.e1 = pl->mb_eptr_host[m + 1];
    q.u0 = pl->mb_uptr_host[m]; q.u1 = pl->mb_uptr_host[m + 1];
    q.sg0 = pl->mb_sgptr_host[m]; q.sg1 = pl->mb_sgptr_host[m + 1];
    q.sh0 = pl->mb_shptr_host[m]; q.sh1 = pl->mb_shptr_host[m + 1];
    q.lc0 = pl->mb_lcptr_host[m]; q.lc1 = pl->mb_lcptr_host[m + 1];
    q.ml0 = pl->mb_mlptr_host[m]; q.ml1 = pl->mb_mlptr_host[m + 1];
    q.b0 = m * pl->batch_local;
    q.b1 = q.b0 + pl->batch_local < pl->n_local ? q.b0 + pl->batch_local : pl->n_local;
    return q;
}

template <int DEG, int NORD, int G, int KCH>
static int launch_minibatch(const sp_psgd_ctx *cx, const sp_dataset *ds, const sp_psgd_plan *pl, const double *y,
                            const int32_t *idx, const PlanMb &mb, const StepArgs &sa, cudaStream_t st) {
    const bool sharded = cx->world > 1;
    RowsArgs ra;
    ra.k = cx->k; ra.d = cx->d_rows;
    ra.indptr = ds->csr_indptr;
    ra.colidx = sharded ? pl->csr_slot : ds->csr_indices;
    ra.data = ds->csr_data; ra.y = y;
    ra.Psrc = sharded ? cx->stage : cx->P; ra.wsrc = sharded ? cx->stage_w : cx->w;
    ra.lams = cx->lams; ra.thr = cx->thr;
    ra.invC = sa.invC; ra.invCw = sa.invCw;
    ra.loss = cx->loss; ra.fit_linear = cx->fit_linear;
    ra.idx = idx; ra.b0 = mb.b0; ra.b1 = mb.b1;
    ra.bufA = cx->bufA; ra.bufdL = cx->bufdL; ra.sloss = cx->sample_loss;
    long long groups = mb.b1 - mb.b0;
    int blocks = grid_for(groups, G);
    if (blocks > 148 * 16) blocks = 148 * 16;
    sp_prof_begin(SP_PROF_PSGD_GRAD, st);
    if (sharded) psgd_rows_kernel<DEG, NORD, G, KCH, true><<<blocks, PL_THREADS, 0, st>>>(ra);
    else psgd_rows_kernel<DEG, NORD, G, KCH, false><<<blocks, PL_THREADS, 0, st>>>(ra);
    sp_prof_end(st);
    SP_LAUNCH_CHECK("psgd_rows_kernel");

    ColsArgs ca;
    ca.k = cx->k; ca.d = cx->d_rows;
    ca.e_pos = pl->e_pos; ca.e_x = pl->e_x;
    ca.u_feat = pl->u_feat; ca.u_ptr = pl->u_ptr;
    ca.u_base = mb.u0;
    ca.sg_u = pl->sg_u + mb.sg0; ca.sg_feat = pl->sg_feat + mb.sg0; ca.sg_pos = pl->sg_pos + mb.sg0; ca.sg_x = pl->sg_x + mb.sg0;
    ca.n_single = (int)(mb.sg1 - mb.sg0);
    ca.sc_ptr = pl->sc_ptr + mb.sh0; ca.sc_u = pl->sc_u + mb.sh0; ca.sc_feat = pl->sc_feat + mb.sh0;
    ca.sc_pos = pl->sc_pos; ca.sc_x = pl->sc_x;
    ca.n_short = (int)(mb.sh1 - mb.sh0);
    ca.lc_u = pl->lc_u + mb.lc0; ca.lc_e0 = pl->lc_e0 + mb.lc0; ca.n_chunks = (int)(mb.lc1 - mb.lc0);
    ca.lc_feat = pl->lc_feat + mb.lc0; ca.lc_cnt = pl->lc_cnt + mb.lc0;
    ca.ml_u = pl->ml_u + mb.ml0; ca.ml_c0 = pl->ml_c0 + mb.ml0; ca.n_multi = (int)(mb.ml1 - mb.ml0);
    ca.bufA = cx->bufA; ca.bufdL = cx->bufdL;
    ca.lams = cx->lams; ca.thr = cx->thr;
    ca.P = cx->P; ca.w = cx->w;
    ca.stage = cx->stage; ca.stage_w = cx->stage_w;
    ca.part_g = cx->part_g; ca.part_w = cx->part_w;
    ca.s = sa;
    ca.world = cx->world; ca.rank = cx->rank;
    for (int r = 0; r <= SP_MAX_RANKS; r++) ca.owner_start[r] = 0;
    for (int r = 0; r < SP_MAX_RANKS; r++) { ca.inbox_g[r] = nullptr; ca.inbox_w[r] = nullptr; }
    if (sharded) {
        const int m = mb.b0 / pl->batch_local;
        for (int r = 0; r <= cx->world; r++) ca.owner_start[r] = pl->mb_owner_start_host[(size_t)m * (cx->world + 1) + r];
        for (int r = 0; r < cx->world; r++) { ca.inbox_g[r] = cx->peer_inbox_g[r]; ca.inbox_w[r] = cx->peer_inbox_w[r]; }
    }
    sp_prof_begin(SP_PROF_PSGD_STEP, st);
    if (ca.n_chunks > 0) {                                   // long columns first: their tail (combine) overlaps nothing else
        const int cb = grid_for(ca.n_chunks, G);
        if (sharded) psgd_cols_long_kernel<DEG, NORD, G, KCH, MODE_PUSH><<<cb, PL_THREADS, 0, st>>>(ca);
        else psgd_cols_long_kernel<DEG, NORD, G, KCH, MODE_APPLY><<<cb, PL_THREADS, 0, st>>>(ca);
        SP_LAUNCH_CHECK("psgd_cols_long_kernel");
    }
    {
        int nb_single = ca.n_single > 0 ? grid_for((ca.n_single + G - 1) / G, G) : 0;
        if (nb_single > 148 * 12) nb_single = 148 * 12;
        int nb_short = ca.n_short > 0 ? grid_for((ca.n_short + 3) / 4, G) : 0;      // ~4 columns per group: enough to fill the pipeline
        if (nb_short > 148 * 3) nb_short = 148 * 3;
        const int nb = ca.n_multi + nb_single + nb_short;
        if (nb > 0) {
            if (sharded) psgd_cols_tail_kernel<DEG, NORD, G, KCH, MODE_PUSH><<<nb, PL_THREADS, 0, st>>>(ca, nb_single, nb_short);
            else psgd_cols_tail_kernel<DEG, NORD, G, KCH, MODE_APPLY><<<nb, PL_THREADS, 0, st>>>(ca, nb_single, nb_short);
            SP_LAUNCH_CHECK("psgd_cols_tail_kernel");
        }
    }
    sp_prof_end(st);
    return SP_OK;
}

template <int NORD, int G, int KCH>
static int launch_owner(const sp_psgd_ctx *cx, const sp_psgd_plan *pl, int m, const StepArgs &sa, cudaStream_t st) {
    OwnerArgs oa;
    const long long o0 = pl->mb_optr_host[m], o1 = pl->mb_optr_host[m + 1];
    oa.k = cx->k; oa.d_own = cx->d_rows; oa.world = cx->world; oa.n_rows = (int)(o1 - o0);
    oa.own_q = pl->own_q + o0;
    oa.own_src = pl->own_src + o0 * cx->world;
    for (int r = 0; r < SP_MAX_RANKS; r++) { oa.inbox_g[r] = nullptr; oa.inbox_w[r] = nullptr; }
    for (int r = 0; r < cx->world; r++) { oa.inbox_g[r] = cx->inbox_g + (size_t)r * cx->inbox_cap * cx->n_orders * cx->k; oa.inbox_w[r] = cx->inbox_w + (size_t)r * cx->inbox_cap; }
    oa.thr = cx->thr; oa.P = cx->P; oa.w = cx->w; oa.s = sa;
    if (oa.n_rows > 0) {
        int ob = grid_for((oa.n_rows + 3) / 4, G);                 // ~4 rows per group
        if (ob > 148 * 3) ob = 148 * 3;
        psgd_owner_kernel<NORD, G, KCH><<<ob, PL_THREADS, 0, st>>>(oa);
        SP_LAUNCH_CHECK("psgd_owner_kernel");
    }
    return SP_OK;
}

static int xbarrier(const sp_psgd_ctx *cx, int chan, unsigned long long seq, cudaStream_t st) {
    XArgs x;
    x.world = cx->world; x.rank = cx->rank; x.chan = chan; x.seq = seq;
    for (int r = 0; r < SP_MAX_RANKS; r++) x.peer_flags[r] = r < cx->world ? cx->peer_flags[r] : nullptr;
    x.my_flags = cx->peer_flags[cx->rank];
    x.err = cx->err;
    psgd_xbarrier_kernel<<<1, 32, 0, st>>>(x);
    SP_LAUNCH_CHECK("psgd_xbarrier_kernel");
    return SP_OK;
}

// the context's own stream (high priority: its few blocks slot in between the statistics pass's) and events
static int aux_init(sp_psgd_ctx *cx) {
    if (cx->aux_stream != nullptr) return SP_OK;
    int lo = 0, hi = 0;
    SP_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    cudaStream_t s;
    SP_CUDA(cudaStreamCreateWithPriority(&s, cudaStreamNonBlocking, hi));
    cudaEvent_t e0, e1;
    SP_CUDA(cudaEventCreateWithFlags(&e0, cudaEventDisableTiming));
    SP_CUDA(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
    cx->aux_stream = s; cx->aux_event[0] = e0; cx->aux_event[1] = e1;
    return SP_OK;
}
extern "C" int sp_psgd_plan_release(sp_psgd_ctx *cx) {
    if (cx == nullptr) return SP_OK;
    if (cx->aux_stream != nullptr) { cudaStreamSynchronize((cudaStream_t)cx->aux_stream); cudaStreamDestroy((cudaStream_t)cx->aux_stream); }
    for (int i = 0; i < 2; i++) if (cx->aux_event[i] != nullptr) cudaEventDestroy((cudaEvent_t)cx->aux_event[i]);
    cx->aux_stream = nullptr; cx->aux_event[0] = cx->aux_event[1] = nullptr;
    return SP_OK;
}

// layout of cx->work (doubles)
struct WorkLayout {
    size_t psum, pcnt, colres, tau, state, band, statbox, xbuf, ints, total;
};
static WorkLayout work_layout(size_t ncol, int world) {
    WorkLayout L;
    size_t at = 0;
    L.psum = at; at += (size_t)STAT_PART_MAX * ncol;
    L.pcnt = at; at += (size_t)STAT_PART_MAX * ncol;
    L.colres = at; at += 2 * ncol;
    L.tau = at; at += ncol;
    L.state = at; at += 8 + 3 * ncol;                  // (+ the band size of every column at the last call: diagnostics)
    L.band = at; at += ncol * (size_t)BAND_CAP;
    L.ints = at; at += (ncol + 8) / 2 + 4;            // band counters + ticket | fail[2]
    L.total = at;
    (void)world;
    return L;
}

extern "C" size_t sp_psgd_plan_work_doubles(int n_orders, int k) {
    return work_layout((size_t)n_orders * k, 1).total + 64;
}
// peer-visible buffer of one rank (doubles): statboxes of all ranks | exchange buffers of all ranks
extern "C" size_t sp_psgd_plan_xwork_doubles(int n_orders, int k, int world) {
    const size_t ncol = (size_t)n_orders * k;
    return (size_t)world * statbox_doubles(ncol) + (size_t)world * 2 * 2 * ncol + 64;
}

static int solve_grid(int *nblk_out, int ncol) {
    int dev = 0, sms = 0, occ = 0;
    SP_CUDA(cudaGetDevice(&dev));
    SP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    SP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, psgd_solve_kernel, SOLVE_THREADS, 0));
    if (occ < 1) { sp_set_error("psgd_solve_kernel does not fit on an SM"); return SP_ERR_CUDA; }
    // one block per column is all the band path needs (a smaller cooperative grid launches and synchronises faster);
    // the generic passes -- first minibatches of a fit, a band miss every few thousand minibatches -- are
    // correspondingly slower, which is the right trade
    int nb = ncol < 16 ? 16 : ncol;
    *nblk_out = nb < sms ? nb : sms;
    return SP_OK;
}

static int ctx_check(const sp_psgd_ctx *cx) {
    if (!cx || !cx->P || !cx->w || !cx->lams || !cx->thr || !cx->bufA || !cx->bufdL || !cx->sample_loss || !cx->work ||
        !cx->part_g || !cx->part_w || cx->k <= 0 || cx->n_orders <= 0 || cx->world < 1 || cx->world > SP_MAX_RANKS ||
        cx->rank < 0 || cx->rank >= cx->world) {
        sp_set_error("sp_psgd_plan_*: invalid context");
        return SP_ERR_INVALID;
    }
    if (cx->reg != SP_REG_L1 && cx->reg != SP_REG_SQL12) {
        sp_set_error("the planned psgd path handles l1 and squaredl12 (use sp_psgd_epoch for l21 / squaredl21)");
        return SP_ERR_UNSUPPORTED;
    }
    if (cx->degree < 2 || cx->degree > SP_MAXDEG) {
        sp_set_error("psgd degree %d is not supported by the CUDA backend (2..%d)", cx->degree, SP_MAXDEG);
        return SP_ERR_UNSUPPORTED;
    }
    if (cx->n_orders != 1 && cx->n_orders != cx->degree - 1) {
        sp_set_error("psgd: n_orders must be 1 or degree-1 (got %d)", cx->n_orders);
        return SP_ERR_INVALID;
    }
    if (cx->k > 128) { sp_set_error("psgd: n_components=%d > 128 is not supported by the CUDA backend", cx->k); return SP_ERR_UNSUPPORTED; }
    if (cx->world > 1 && (!cx->stage || !cx->stage_w || !cx->inbox_g || !cx->inbox_w || !cx->err || !cx->xwork)) {
        sp_set_error("sp_psgd_plan_*: sharded context without peer buffers");
        return SP_ERR_INVALID;
    }
    return SP_OK;
}

// diagnostics of the squared-l1,2 selection since sp_psgd_plan_begin: out_host[0] = prox calls, [1] = solved from the
// band, [2] = needed the generic passes, [3] = current band half-width, [4] / [5] = mean / largest band size of the
// columns at the last call
extern "C" int sp_psgd_plan_solver_stats(const sp_psgd_ctx *cx, double *out_host, sp_stream stream) {
    int rc = ctx_check(cx);
    if (rc) return rc;
    if (!out_host) { sp_set_error("sp_psgd_plan_solver_stats: null pointer"); return SP_ERR_INVALID; }
    const WorkLayout L = work_layout((size_t)cx->n_orders * cx->k, cx->world);
    const size_t ncol = (size_t)cx->n_orders * cx->k;
    std::vector<double> st(8 + 3 * ncol);
    SP_CUDA(cudaMemcpyAsync(st.data(), cx->work + L.state, st.size() * sizeof(double), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    SP_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    out_host[0] = st[1]; out_host[1] = st[2]; out_host[2] = st[3]; out_host[3] = st[4] > 0.0 ? st[4] : BAND_DELTA;
    double mx = 0.0, sm = 0.0;
    for (size_t c = 0; c < ncol; c++) { const double v = st[8 + 2 * ncol + c]; sm += v; if (v > mx) mx = v; }
    out_host[4] = ncol ? sm / (double)ncol : 0.0; out_host[5] = mx;
    return SP_OK;
}

extern "C" int sp_psgd_plan_begin(sp_psgd_ctx *cx, sp_stream stream) {
    int rc = ctx_check(cx);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t ncol = (size_t)cx->n_orders * cx->k;
    const WorkLayout L = work_layout(ncol, cx->world);
    SP_CUDA(cudaMemsetAsync(cx->thr, 0, ncol * sizeof(double), st));
    SP_CUDA(cudaMemsetAsync(cx->work + L.state, 0, (L.total - L.state) * sizeof(double), st));
    cx->C = 1.0; cx->Cw = 1.0;
    return SP_OK;
}

// The lazy scales only grow (by 1 + eta * beta per minibatch): the frame is folded back into the storage as soon
// as C or Cw leaves (1e-100, 1e100), long before either can overflow.  The rule depends on the C trajectory alone,
// so every way of cutting the same minibatches into calls (epochs, partial_fit chunks) folds after the same ones.
constexpr double FRAME_MAX = 1e100;
static inline bool frame_in_range(double C, double Cw) {
    return 1.0 / FRAME_MAX < C && C < FRAME_MAX && 1.0 / FRAME_MAX < Cw && Cw < FRAME_MAX;
}

// P / w <- the model the frame represents, thresholds 0, scales 1; sharded: every rank's rows are folded before
// any rank reads a peer's rows again
static int fold_frame(sp_psgd_ctx *cx, cudaStream_t st) {
    const size_t n = (size_t)cx->n_orders * cx->d_rows * cx->k;
    if (n > 0) {
        size_t b = (n + 255) / 256;
        if (b > 148 * 16) b = 148 * 16;
        psgd_materialize_kernel<<<(int)b, 256, 0, st>>>(cx->P, cx->n_orders, (size_t)cx->d_rows, cx->k, cx->thr, 1.0 / cx->C,
                                                      cx->w, 1.0 / cx->Cw, cx->fit_linear);
        SP_LAUNCH_CHECK("psgd_materialize_kernel");
    }
    psgd_zero_kernel<<<1, 256, 0, st>>>(cx->thr, cx->n_orders * cx->k);
    SP_LAUNCH_CHECK("psgd_zero_kernel");
    cx->C = 1.0; cx->Cw = 1.0;
    if (cx->world > 1) { cx->seq += 1; return xbarrier(cx, 0, cx->seq, st); }
    return SP_OK;
}

// Minibatches [m_begin, m_end) of one epoch = the body of psgd.psgd_epoch (psgd.py:150-198) for them.
extern "C" int sp_psgd_plan_run(sp_psgd_ctx *cx, const sp_dataset *ds, const sp_psgd_plan *pl, const double *y,
                                const int32_t *idx_samples, double alpha, double beta, double gamma, double eta0,
                                int learning_rate, double power_t, int m_begin, int m_end, int64_t *it_io_host,
                                sp_stream stream) {
    int rc = ctx_check(cx);
    if (rc) return rc;
    if (!ds || !ds->csr_indptr || !pl || !y || !idx_samples || !it_io_host || m_begin < 0 || m_end > pl->n_minibatches ||
        m_begin > m_end) {
        sp_set_error("sp_psgd_plan_run: invalid argument");
        return SP_ERR_INVALID;
    }
    if (pl->chunk != CH || pl->short_max != SP_PSGD_SHORT) { sp_set_error("sp_psgd_plan_run: plan built for chunk %d / short %d, library uses %d / %d", pl->chunk, pl->short_max, CH, SP_PSGD_SHORT); return SP_ERR_INVALID; }
    if (cx->world > 1 && (!pl->csr_slot || !pl->own_q || !pl->own_src || !pl->mb_owner_start_host || !pl->mb_optr_host)) {
        sp_set_error("sp_psgd_plan_run: sharded run with a single-rank plan");
        return SP_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int k = cx->k, nord = cx->n_orders;
    const size_t ncol = (size_t)nord * k;
    const WorkLayout L = work_layout(ncol, cx->world);
    const bool sharded = cx->world > 1;
    int solve_blocks = 0;
    if (cx->reg == SP_REG_SQL12) { rc = solve_grid(&solve_blocks, (int)ncol); if (rc) return rc; }
    int64_t it = *it_io_host;
    // sharded: the raw rows minibatch m touches are pulled on the context's own stream -- for the first minibatch
    // of the call right away (every owner's rows are final: the previous step ended with a barrier), for the
    // others as soon as every rank's owner update of minibatch m-1 is done (flag barrier on channel 2 of that
    // stream), i.e. WHILE the statistics pass / selection of m-1 run here: those only move the frame.
    cudaStream_t s2 = nullptr;
    cudaEvent_t ev_own = nullptr, ev_pull = nullptr;
    auto pull = [&](int m) -> int {
        const PlanMb pm = plan_mb(pl, m);
        PullArgs pa;
        pa.k = k; pa.d_own = cx->d_rows; pa.world = cx->world; pa.n_cols = (int)(pm.u1 - pm.u0);
        pa.u_feat = pl->u_feat + pm.u0;
        for (int r = 0; r < SP_MAX_RANKS; r++) { pa.peer_P[r] = r < cx->world ? cx->peer_P[r] : nullptr; pa.peer_w[r] = r < cx->world ? cx->peer_w[r] : nullptr; }
        pa.n_orders = nord; pa.fit_linear = cx->fit_linear;
        pa.stage = cx->stage; pa.stage_w = cx->stage_w;
        if (pa.n_cols > 0) {
            long long blocks = ((long long)(pa.n_cols + 7) / 8 + 7) / 8;          // 8 rows per warp pass, 8 warps per block
            if (blocks > 148 * 8) blocks = 148 * 8;
            if (blocks < 1) blocks = 1;
            sp_prof_begin(SP_PROF_ROWS, s2);                                     // (sharded psgd: class 0 = pull)
            psgd_pull_kernel<<<(int)blocks, PL_THREADS, 0, s2>>>(pa);
            sp_prof_end(s2);
            SP_LAUNCH_CHECK("psgd_pull_kernel");
        }
        SP_CUDA(cudaEventRecord(ev_pull, s2));
        return SP_OK;
    };
    if (sharded) {
        rc = aux_init(cx);
        if (rc) return rc;
        s2 = (cudaStream_t)cx->aux_stream; ev_own = (cudaEvent_t)cx->aux_event[0]; ev_pull = (cudaEvent_t)cx->aux_event[1];
        if (m_begin < m_end) {
            SP_CUDA(cudaEventRecord(ev_own, st));
            SP_CUDA(cudaStreamWaitEvent(s2, ev_own, 0));
            rc = pull(m_begin);
            if (rc) return rc;
        }
    }
    for (int m = m_begin; m < m_end; m++) {
        const PlanMb mb = plan_mb(pl, m);
        const long long b_glob = (long long)(mb.b1 - mb.b0) * cx->world;
        double eta_P, eta_w;
        rc = sp_get_eta(learning_rate, eta0, alpha, beta, power_t, it, &eta_P, &eta_w);     // psgd.py:178
        if (rc) return rc;
        StepArgs sa;
        sa.cP = eta_P / (double)b_glob; sa.denP = 1.0 + eta_P * beta; sa.CnP = cx->C * sa.denP;
        sa.cw = eta_w / (double)b_glob; sa.denw = 1.0 + eta_w * alpha; sa.Cnw = cx->fit_linear ? cx->Cw * sa.denw : cx->Cw;
        sa.invC = 1.0 / cx->C; sa.invCw = 1.0 / cx->Cw;
        sa.rP = 1.0 / sa.denP; sa.rw = 1.0 / sa.denw;
        sa.fit_linear = cx->fit_linear;
        const double strength = gamma * eta_P / (1.0 + eta_P * beta);                     // psgd.py:122
        const bool fold = !frame_in_range(sa.CnP, sa.Cnw);                // the frame is folded after this minibatch
        if (sharded) SP_CUDA(cudaStreamWaitEvent(st, ev_pull, 0));          // this minibatch's rows are staged
#define SP_MB(D, N, GG, KC) rc = launch_minibatch<D, N, GG, KC>(cx, ds, pl, y, idx_samples, mb, sa, st)
#define SP_MB_K(D, N)                                                                      \
        if (k <= 8) SP_MB(D, N, 8, 1);                                                     \
        else if (k <= 16) SP_MB(D, N, 16, 1);                                              \
        else if (k <= 32) SP_MB(D, N, 32, 1);                                              \
        else if (k <= 64) SP_MB(D, N, 32, 2);                                              \
        else SP_MB(D, N, 32, 4)
        const bool ex = nord > 1;
        switch (cx->degree) {
        case 2: SP_MB_K(2, 1); break;
        case 3: if (ex) { SP_MB_K(3, 2); } else { SP_MB_K(3, 1); } break;
        case 4: if (ex) { SP_MB_K(4, 3); } else { SP_MB_K(4, 1); } break;
        default: if (ex) { SP_MB_K(5, 4); } else { SP_MB_K(5, 1); } break;
        }
#undef SP_MB_K
#undef SP_MB
        if (rc) return rc;
        if (sharded) {
            sp_prof_begin(SP_PROF_REGCACHE, st);                   // (sharded psgd: class 1 = inbox barrier, 2 = owner)
            cx->seq += 1;
            rc = xbarrier(cx, 0, cx->seq, st);                     // every rank's partial rows are in the inboxes
            sp_prof_end(st);
            if (rc) return rc;
            sp_prof_begin(SP_PROF_SWEEP_PCD, st);
#define SP_OW(N, GG, KC) rc = launch_owner<N, GG, KC>(cx, pl, m, sa, st)
#define SP_OW_K(N)                                                                         \
            if (k <= 8) SP_OW(N, 8, 1);                                                    \
            else if (k <= 16) SP_OW(N, 16, 1);                                             \
            else if (k <= 32) SP_OW(N, 32, 1);                                             \
            else if (k <= 64) SP_OW(N, 32, 2);                                             \
            else SP_OW(N, 32, 4)
            switch (nord) {
            case 1: SP_OW_K(1); break;
            case 2: SP_OW_K(2); break;
            case 3: SP_OW_K(3); break;
            default: SP_OW_K(4); break;
            }
#undef SP_OW_K
#undef SP_OW
            sp_prof_end(st);
            if (rc) return rc;
            if (m + 1 < m_end && !fold) {                          // next minibatch's rows: see above (after a fold they
                                                                   // are pulled once every rank's rows are folded)
                SP_CUDA(cudaEventRecord(ev_own, st));
                SP_CUDA(cudaStreamWaitEvent(s2, ev_own, 0));
                cx->seq_pull += 1;
                rc = xbarrier(cx, 2, cx->seq_pull, s2);
                if (rc) return rc;
                rc = pull(m + 1);
                if (rc) return rc;
            }
        }
        cx->C = sa.CnP; cx->Cw = sa.Cnw;
        const double invCn = 1.0 / cx->C;
        if (cx->reg == SP_REG_L1) {
            psgd_thr_advance_kernel<<<(int)((ncol + 127) / 128), 128, 0, st>>>(cx->thr, (int)ncol, cx->C * strength);
            SP_LAUNCH_CHECK("psgd_thr_advance_kernel");
            if (sharded) { cx->seq += 1; rc = xbarrier(cx, 0, cx->seq, st); if (rc) return rc; }   // owners' rows are final
        } else {
            StatArgs sg;
            sg.P = cx->P; sg.n_orders = nord; sg.d = cx->d_rows; sg.k = k;
            sg.invC = invCn; sg.strength = strength; sg.thr = cx->thr; sg.reg = cx->reg;
            sg.psum = cx->work + L.psum; sg.pcnt = cx->work + L.pcnt;
            sg.band = cx->work + L.band;
            sg.band_n = reinterpret_cast<int *>(cx->work + L.ints);
            sg.state = cx->work + L.state;
            sg.tau = nullptr;
            sg.world = cx->world; sg.rank = cx->rank;
            const size_t boxlen = statbox_doubles(ncol);
            for (int r = 0; r < SP_MAX_RANKS; r++) sg.statbox[r] = nullptr;
            if (sharded) { for (int r = 0; r < cx->world; r++) sg.statbox[r] = cx->peer_xwork[r] + (size_t)cx->rank * boxlen; }
            else sg.statbox[0] = cx->xwork;
            sg.err = cx->err;
            const int tpr = (k & 1) ? k : k / 2, rpp = PL_THREADS / tpr;
            long long nblk = ((long long)cx->d_rows + rpp - 1) / rpp;
            if (nblk > STAT_PART_MAX) nblk = STAT_PART_MAX;
            if (sharded && nblk > 148 * 2) nblk = 148 * 2;         // (leaves room on every SM for the early pull's blocks)
            if (nblk < 1) nblk = 1;
            sp_prof_begin(SP_PROF_PROX, st);
            psgd_stats_kernel<<<(int)nblk, PL_THREADS, 0, st>>>(sg);
            SP_LAUNCH_CHECK("psgd_stats_kernel");
            if (sharded) {
                psgd_stats_publish_kernel<<<(int)ncol, PL_THREADS, 0, st>>>(sg, (int)nblk);
                SP_LAUNCH_CHECK("psgd_stats_publish_kernel");
                cx->seq += 1;
                rc = xbarrier(cx, 0, cx->seq, st);
                if (rc) { sp_prof_end(st); return rc; }
            }
            sp_prof_end(st);
            sp_prof_begin(SP_PROF_PLAN, st);                       // (psgd: class 6 = statistics pass, class 7 = solve)
            SolveArgs so;
            so.st = sg;
            so.Cn = cx->C; so.thr = cx->thr; so.tau = cx->work + L.tau; so.colres = cx->work + L.colres;
            so.fail = reinterpret_cast<int *>(cx->work + L.ints) + ((ncol + 8) & ~1) ;
            so.npart = (int)nblk;
            so.statbox_all = cx->xwork;
            const size_t xoff = (size_t)cx->world * boxlen;
            for (int r = 0; r < SP_MAX_RANKS; r++) so.xbuf[r] = nullptr;
            if (sharded) for (int r = 0; r < cx->world; r++) so.xbuf[r] = cx->peer_xwork[r] + xoff + (size_t)cx->rank * 4 * ncol;
            so.xbuf_local = cx->xwork + xoff;
            so.x.world = cx->world; so.x.rank = cx->rank; so.x.chan = 1; so.x.seq = cx->seq_generic + 1;
            for (int r = 0; r < SP_MAX_RANKS; r++) so.x.peer_flags[r] = (sharded && r < cx->world) ? cx->peer_flags[r] : nullptr;
            so.x.my_flags = sharded ? cx->peer_flags[cx->rank] : nullptr;
            so.x.err = cx->err;
            so.seq_out = nullptr;
            so.max_iter = 500;
            cx->seq_generic += (unsigned long long)so.max_iter;     // sequence numbers reserved for this call's exchanges
            so.call_id = (int)((cx->seq_generic / (unsigned long long)so.max_iter) & 0x3fffffffull) + 1;
            void *args[] = {(void *)&so};
            cudaError_t e = cudaLaunchCooperativeKernel((void *)psgd_solve_kernel, dim3(solve_blocks), dim3(SOLVE_THREADS), args, 0, st);
            sp_prof_end(st);
            if (e != cudaSuccess) return sp_check_cuda(e, "psgd_solve_kernel launch");
        }
        if (fold) {
            rc = fold_frame(cx, st);
            if (rc) return rc;
            if (sharded && m + 1 < m_end) {                        // (fold_frame ended with a cross-rank barrier)
                SP_CUDA(cudaEventRecord(ev_own, st));
                SP_CUDA(cudaStreamWaitEvent(s2, ev_own, 0));
                rc = pull(m + 1);
                if (rc) return rc;
            }
        }
        it++;
    }
    *it_io_host = it;
    return SP_OK;
}

// epoch end: *loss_sum += sum of the epoch's per-sample losses (fixed order); the raw matrix becomes the
// model again (thresholds 0, scales 1) so that P / w can be read by anyone
extern "C" int sp_psgd_plan_end(sp_psgd_ctx *cx, int n_local, double *loss_sum, int materialize, sp_stream stream) {
    int rc = ctx_check(cx);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (loss_sum && n_local > 0) {
        const WorkLayout L = work_layout((size_t)cx->n_orders * cx->k, cx->world);
        double *part = cx->work + L.psum;                          // (free between minibatches; >= 444 doubles)
        psgd_loss_part_kernel<<<LOSS_BLOCKS, 1024, 0, st>>>(cx->sample_loss, 0, n_local, part);
        SP_LAUNCH_CHECK("psgd_loss_part_kernel");
        psgd_loss_sum_kernel<<<1, 256, 0, st>>>(part, loss_sum);
        SP_LAUNCH_CHECK("psgd_loss_sum_kernel");
    }
    if (materialize) return fold_frame(cx, st);
    return SP_OK;
}

// the model the lazy frame represents, for a caller that goes on training: the context is only read
extern "C" int sp_psgd_plan_read(const sp_psgd_ctx *cx, double *P_out, double *w_out, sp_stream stream) {
    int rc = ctx_check(cx);
    if (rc) return rc;
    if (cx->world > 1) { sp_set_error("sp_psgd_plan_read: single rank only (got world %d)", cx->world); return SP_ERR_UNSUPPORTED; }
    if (!P_out || !w_out) { sp_set_error("sp_psgd_plan_read: null pointer"); return SP_ERR_INVALID; }
    cudaStream_t st = (cudaStream_t)stream;
    const int d = cx->d_rows, k = cx->k;
    if (d > 0) {
        const dim3 grid((unsigned)((d + READ_TILE - 1) / READ_TILE), (unsigned)((k + READ_TILE - 1) / READ_TILE), (unsigned)cx->n_orders);
        psgd_read_kernel<<<grid, dim3(READ_TILE, READ_ROWS), 0, st>>>(cx->P, d, k, cx->thr, 1.0 / cx->C, P_out);
        SP_LAUNCH_CHECK("psgd_read_kernel");
        int b = (d + 255) / 256;
        if (b > 148 * 16) b = 148 * 16;
        psgd_read_w_kernel<<<b, 256, 0, st>>>(cx->w, d, 1.0 / cx->Cw, cx->fit_linear, w_out);
        SP_LAUNCH_CHECK("psgd_read_w_kernel");
    }
    return SP_OK;
}

// ------------------------------------------------------------------------------------ peer memory (CUDA IPC)
extern "C" int sp_shm_alloc(size_t bytes, void **out) {
    if (!out) { sp_set_error("sp_shm_alloc: null pointer"); return SP_ERR_INVALID; }
    SP_CUDA(cudaMalloc(out, bytes ? bytes : 8));
    SP_CUDA(cudaMemset(*out, 0, bytes ? bytes : 8));
    return SP_OK;
}
extern "C" int sp_shm_free(void *p) { return sp_check_cuda(cudaFree(p), "cudaFree"); }
extern "C" int sp_ipc_export(void *p, unsigned char *handle64) {
    if (!p || !handle64) { sp_set_error("sp_ipc_export: null pointer"); return SP_ERR_INVALID; }
    cudaIpcMemHandle_t h;
    SP_CUDA(cudaIpcGetMemHandle(&h, p));
    static_assert(sizeof(h) == 64, "cudaIpcMemHandle_t is 64 bytes");
    memcpy(handle64, &h, 64);
    return SP_OK;
}
extern "C" int sp_ipc_open(const unsigned char *handle64, void **out) {
    if (!handle64 || !out) { sp_set_error("sp_ipc_open: null pointer"); return SP_ERR_INVALID; }
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    SP_CUDA(cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess));
    return SP_OK;
}
extern "C" int sp_ipc_close(void *p) { return sp_check_cuda(cudaIpcCloseMemHandle(p), "cudaIpcCloseMemHandle"); }
extern "C" int sp_memcpy(void *dst, const void *src, size_t bytes, int kind, sp_stream stream) {
    const cudaMemcpyKind kd = kind == 0 ? cudaMemcpyHostToDevice : (kind == 1 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice);
    SP_CUDA(cudaMemcpyAsync(dst, src, bytes, kd, (cudaStream_t)stream));
    if (kind == 1) SP_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
    return SP_OK;
}
