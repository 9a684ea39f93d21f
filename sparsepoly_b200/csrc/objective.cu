// Objective evaluation: sum of losses, squared l2 norms and the regularizers' Omega(P).
//
// The reference's update rules minimise
//     sum_i loss(y_pred_i, y_i) + alpha/2 |w|^2 + beta/2 |P|^2 + gamma * Omega(P)
// (sparse_factorization_machines.py:181-188, :265-272) but no call site ever evaluates it; the
// regularizer classes carry `eval` methods (l1.py:17-18, l21.py:19-21, squaredl12.py:20-22,
// squaredl21.py:23-25, omegati.py:19-47, omegacs.py:22-39) that define Omega.  These kernels
// compute the same quantities on device so that a fit can be monitored / compared ("objective
// within 1e-9") without copying P and y_pred to the host.
//
// Every Omega is a fold over the feature rows j of a non-negative value v_jc (|p_js| per component
// column, or the row norm |p_j|_2) with one of two associative operations:
//   POLY(m): truncated product of the polynomials (1 + v z) mod z^(m+1)  -> e_0..e_m, the elementary
//            symmetric polynomials (m = 1: e_1 = the plain sum)
//   PROD   : product of (1 + v)                                          (all-subsets variants)
// so one streaming pass over P (HBM-bound: d*k*8 bytes read once, coalesced) produces per-block
// partial states that are combined in a fixed tree: deterministic, and well conditioned because
// all terms are >= 0.  The reference folds left to right; the difference is O(1e-16) relative.
#include "common.cuh"
#include "sparsepoly_b200.h"

namespace {
constexpr int OB_THREADS = 256;
constexpr int OB_MAXBLK = 148 * 4;
constexpr int OB_ST = SP_MAXDEG + 1;
constexpr int OB_CT = 640;               // combine kernel threads (>= OB_MAXBLK)
constexpr int OB_FT = 1024;              // final sum kernel threads (power of two >= OB_MAXBLK)

struct Poly { double e[OB_ST]; };

__device__ __forceinline__ void poly_init(Poly &p) {
    p.e[0] = 1.0;
#pragma unroll
    for (int t = 1; t < OB_ST; t++) p.e[t] = 0.0;
}
__device__ __forceinline__ void poly_fold(Poly &p, double v, int m, int prod) {
    if (prod) { p.e[0] *= 1.0 + v; return; }
#pragma unroll
    for (int t = OB_ST - 1; t >= 1; t--)
        if (t <= m) p.e[t] += p.e[t - 1] * v;
}
__device__ __forceinline__ Poly poly_mul(const Poly &l, const Poly &r, int m, int prod) {
    Poly o;
    poly_init(o);
    if (prod) { o.e[0] = l.e[0] * r.e[0]; return o; }
#pragma unroll
    for (int t = 0; t < OB_ST; t++) {
        if (t > m) break;
        double acc = 0.0;
#pragma unroll
        for (int u = 0; u < OB_ST; u++)
            if (u <= t) acc += l.e[u] * r.e[t - u];
        o.e[t] = acc;
    }
    return o;
}

// tree over `cnt` states stored at sh[(base + i*stride)], i = 0..cnt-1; result lands in i = 0
__device__ __forceinline__ void poly_tree(double (*sh)[OB_ST], int i, int cnt, int stride, int base,
                                          bool active, int m, int prod) {
    for (int off = 1; off < cnt; off <<= 1) {
        if (active && (i & (2 * off - 1)) == 0 && i + off < cnt) {
            Poly l, r;
#pragma unroll
            for (int t = 0; t < OB_ST; t++) {
                l.e[t] = sh[base + i * stride][t];
                r.e[t] = sh[base + (i + off) * stride][t];
            }
            Poly o = poly_mul(l, r, m, prod);
#pragma unroll
            for (int t = 0; t < OB_ST; t++) sh[base + i * stride][t] = o.e[t];
        }
        __syncthreads();
    }
}

// Table entry of one Omega evaluation: its P, its slices of the work buffer (per-block partial states, then one
// state per column), its output and its fold (m / prod / square), columns (k, or 1 for the row norms) and partition
// of the rows (nb blocks of rpb rows).  The tables travel as kernel parameters: no copy, no wait for one.
struct RegEntry {
    const double *P;
    double (*part)[OB_ST];
    double (*colres)[OB_ST];
    double *out;
    int m, prod, square, cols, nb, rpb;
};
struct RegTable { RegEntry e[SP_OBJECTIVE_MAX_ENTRIES]; };

// Per-column fold of |P[j,c]| of entry blockIdx.y: thread (r, c) = (tid / k, tid % k) walks rows j0+r, j0+r+R, ...
// (consecutive threads read consecutive addresses); part[(blk*k + c)] gets the block's state.
__global__ void __launch_bounds__(OB_THREADS) reg_partial_cols_kernel(const __grid_constant__ RegTable tab, int d,
                                                                      int k) {
    const RegEntry &e = tab.e[blockIdx.y];
    const double *__restrict__ P = e.P;
    const int m = e.m, prod = e.prod, rows_per_block = e.rpb;
    __shared__ double sh[OB_THREADS][OB_ST];
    const int tid = threadIdx.x, R = OB_THREADS / k, r = tid / k, c = tid - r * k;
    const bool active = r < R;
    Poly p;
    poly_init(p);
    if (active) {
        const int j0 = blockIdx.x * rows_per_block, j1 = min(d, j0 + rows_per_block);
        for (int j = j0 + r; j < j1; j += R) poly_fold(p, fabs(P[(size_t)j * k + c]), m, prod);
    }
#pragma unroll
    for (int t = 0; t < OB_ST; t++) sh[tid][t] = p.e[t];
    __syncthreads();
    poly_tree(sh, r, R, k, c, active, m, prod);
    if (active && r == 0) {
#pragma unroll
        for (int t = 0; t < OB_ST; t++) e.part[(size_t)blockIdx.x * k + c][t] = sh[c][t];
    }
}

// Fold of the row norms |P[j,:]|_2 of entry blockIdx.y: one group of G lanes per row (fixed butterfly for the sum of
// squares, lanes beyond k idle), every lane of the group folds the same value.
template <int G>
__global__ void __launch_bounds__(OB_THREADS) reg_partial_rows_kernel(const __grid_constant__ RegTable tab, int d,
                                                                      int k) {
    const RegEntry &e = tab.e[blockIdx.y];
    const double *__restrict__ P = e.P;
    const int m = e.m, prod = e.prod, rows_per_block = e.rpb;
    constexpr int NG = OB_THREADS / G;
    __shared__ double sh[NG][OB_ST];
    const int tid = threadIdx.x, g = tid / G, lane = tid % G;
    Poly p;
    poly_init(p);
    const int j0 = blockIdx.x * rows_per_block, j1 = min(d, j0 + rows_per_block);
    for (int jb = j0; jb < j1; jb += NG) {              // block-uniform trip count: the shuffles
        const int j = jb + g;                           // below need every lane of the warp
        double ss = 0.0;
        if (j < j1)
            for (int s = lane; s < k; s += G) {
                const double v = P[(size_t)j * k + s];
                ss += v * v;
            }
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) ss += sp_shfl_xor(ss, o);
        if (j < j1) poly_fold(p, sqrt(ss), m, prod);
    }
    if (lane == 0) {
#pragma unroll
        for (int t = 0; t < OB_ST; t++) sh[g][t] = p.e[t];
    }
    __syncthreads();
    poly_tree(sh, g, NG, 1, 0, lane == 0, m, prod);
    if (tid == 0) {
#pragma unroll
        for (int t = 0; t < OB_ST; t++) e.part[blockIdx.x][t] = sh[0][t];
    }
}

// block (c, y) combines the nb per-block states of column c of entry y; colres[c] = the column's state
__global__ void __launch_bounds__(OB_CT) reg_combine_kernel(const __grid_constant__ RegTable tab) {
    const RegEntry &e = tab.e[blockIdx.y];
    const int tid = threadIdx.x, c = blockIdx.x, nb = e.nb, cols = e.cols, m = e.m, prod = e.prod;
    if (c >= cols) return;                              // block-uniform: entries of fewer columns
    __shared__ double sh[OB_CT][OB_ST];
    if (tid < nb) {
#pragma unroll
        for (int t = 0; t < OB_ST; t++) sh[tid][t] = e.part[(size_t)tid * cols + c][t];
    }
    __syncthreads();
    poly_tree(sh, tid, nb, 1, 0, tid < nb, m, prod);
    if (tid == 0) {
#pragma unroll
        for (int t = 0; t < OB_ST; t++) e.colres[c][t] = sh[0][t];
    }
}

// final scalar of entry blockIdx.x: sum over the columns (ascending) of e_m, of e_1^2 (squared norms) or of the product
__global__ void reg_final_kernel(const __grid_constant__ RegTable tab) {
    if (threadIdx.x != 0) return;
    const RegEntry &e = tab.e[blockIdx.x];
    double acc = 0.0;
    for (int c = 0; c < e.cols; c++) {
        const double v = e.prod ? e.colres[c][0] : e.colres[c][e.m];
        acc += e.square ? v * v : v;
    }
    e.out[0] = acc;
}

// ------------------------------------------------------------------ plain sums
// Table entry of one sum: op 0..2: loss id (loss.py:13-71) of (a[i*sa], b[i*sb]); op 3: a[i*sa]^2
struct SumEntry { const double *a, *b; double *out; int op; };
struct SumTable { SumEntry e[SP_OBJECTIVE_MAX_ENTRIES]; };

// entry blockIdx.y; its per-block partials go to work[blockIdx.y * OB_MAXBLK + blockIdx.x]
__global__ void __launch_bounds__(OB_THREADS) sum_partial_kernel(const __grid_constant__ SumTable tab, int sa, int sb,
                                                                 long long n, double *work) {
    const SumEntry &e = tab.e[blockIdx.y];
    const double *__restrict__ a = e.a;
    const double *__restrict__ b = e.b;
    const int op = e.op;
    __shared__ double sh[OB_THREADS / 32];
    double acc = 0.0;
    for (long long i = (long long)blockIdx.x * OB_THREADS + threadIdx.x; i < n;
         i += (long long)gridDim.x * OB_THREADS) {
        if (op == 3) {
            const double v = a[i * sa];
            acc += v * v;
        } else {
            acc += sp_loss_rt(op, a[i * sa], b[i * sb]);
        }
    }
    acc = sp_warp_allsum(acc);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double s = 0.0;
        for (int w = 0; w < OB_THREADS / 32; w++) s += sh[w];
        work[(size_t)blockIdx.y * OB_MAXBLK + blockIdx.x] = s;
    }
}
// block y sums the nb partials of entry y
__global__ void __launch_bounds__(OB_FT) sum_final_kernel(const __grid_constant__ SumTable tab, int nb,
                                                          const double *work) {
    const double *part = work + (size_t)blockIdx.x * OB_MAXBLK;
    __shared__ double sh[OB_FT];
    const int tid = threadIdx.x;
    sh[tid] = tid < nb ? part[tid] : 0.0;
    __syncthreads();
    for (int off = OB_FT / 2; off > 0; off >>= 1) {
        if (tid < off) sh[tid] += sh[tid + off];
        __syncthreads();
    }
    if (tid == 0) tab.e[blockIdx.x].out[0] = sh[0];
}

int launch_sum(const SumTable &tab, int n_entries, int sa, int sb, long long n, double *work, cudaStream_t st) {
    if (n_entries == 0) return SP_OK;
    long long want = (n + OB_THREADS - 1) / OB_THREADS;
    const int nb = (int)(want < 1 ? 1 : (want > OB_MAXBLK ? OB_MAXBLK : want));
    sum_partial_kernel<<<dim3(nb, n_entries), OB_THREADS, 0, st>>>(tab, sa, sb, n, work);
    SP_LAUNCH_CHECK("sum_partial_kernel");
    sum_final_kernel<<<n_entries, OB_FT, 0, st>>>(tab, nb, work);
    SP_LAUNCH_CHECK("sum_final_kernel");
    return SP_OK;
}

bool table_fits(int n_entries, const char *who) {
    if (n_entries >= 0 && n_entries <= SP_OBJECTIVE_MAX_ENTRIES) return true;
    sp_set_error("%s: %d entries (at most %d per call)", who, n_entries, SP_OBJECTIVE_MAX_ENTRIES);
    return false;
}
}  // namespace

extern "C" size_t sp_sum_work_doubles(void) { return OB_MAXBLK; }

extern "C" size_t sp_reg_eval_work_doubles(int d, int k) {
    (void)d;
    const size_t cols = k > 0 ? (size_t)k : 1;
    return (size_t)(OB_MAXBLK + 1) * cols * OB_ST;
}

extern "C" int sp_loss_sum_multi(const sp_loss_entry *entries, int n_entries, int pred_stride, int y_stride, int n,
                                 double *work, sp_stream stream) {
    if (!table_fits(n_entries, "sp_loss_sum")) return SP_ERR_INVALID;
    if (!entries || !work || n < 0 || pred_stride <= 0 || y_stride <= 0) {
        sp_set_error("sp_loss_sum: invalid argument");
        return SP_ERR_INVALID;
    }
    SumTable tab;
    for (int b = 0; b < n_entries; b++) {
        const sp_loss_entry &e = entries[b];
        if (!e.y_pred || !e.y || !e.out || e.loss < 0 || e.loss > 2) {
            sp_set_error("sp_loss_sum: invalid argument");
            return SP_ERR_INVALID;
        }
        tab.e[b] = SumEntry{e.y_pred, e.y, e.out, e.loss};
    }
    return launch_sum(tab, n_entries, pred_stride, y_stride, n, work, (cudaStream_t)stream);
}

extern "C" int sp_loss_sum(const double *y_pred, int pred_stride, const double *y, int y_stride, int n,
                           int loss, double *work, double *out, sp_stream stream) {
    const sp_loss_entry e = {y_pred, y, loss, out};
    return sp_loss_sum_multi(&e, 1, pred_stride, y_stride, n, work, stream);
}

extern "C" int sp_sqnorm_multi(const sp_sqnorm_entry *entries, int n_entries, int64_t len, double *work,
                               sp_stream stream) {
    if (!table_fits(n_entries, "sp_sqnorm")) return SP_ERR_INVALID;
    if (!entries || !work || len < 0) {
        sp_set_error("sp_sqnorm: invalid argument");
        return SP_ERR_INVALID;
    }
    SumTable tab;
    for (int b = 0; b < n_entries; b++) {
        if (!entries[b].v || !entries[b].out) {
            sp_set_error("sp_sqnorm: invalid argument");
            return SP_ERR_INVALID;
        }
        tab.e[b] = SumEntry{entries[b].v, entries[b].v, entries[b].out, 3};
    }
    return launch_sum(tab, n_entries, 1, 1, len, work, (cudaStream_t)stream);
}

extern "C" int sp_sqnorm(const double *v, int64_t len, double *work, double *out, sp_stream stream) {
    const sp_sqnorm_entry e = {v, out};
    return sp_sqnorm_multi(&e, 1, len, work, stream);
}

extern "C" int sp_reg_eval_multi(const sp_reg_entry *entries, int n_entries, int d, int k, int degree, double *work,
                                 sp_stream stream) {
    if (!table_fits(n_entries, "sp_reg_eval")) return SP_ERR_INVALID;
    if (!entries || !work || d < 0 || k <= 0) {
        sp_set_error("sp_reg_eval: invalid argument");
        return SP_ERR_INVALID;
    }
    cudaStream_t st = (cudaStream_t)stream;
    // all entries, then the column-fold and the row-norm entries apart: one partial launch per kind
    RegTable all, by_cols, by_rows;
    int n_cols = 0, n_rows = 0, max_cols = 1;
    int nb_kind[2] = {0, 0};
    const size_t per_entry = sp_reg_eval_work_doubles(d, k);
    for (int b = 0; b < n_entries; b++) {
        const sp_reg_entry &in = entries[b];
        if ((!in.P_dk && d > 0) || !in.out) {
            sp_set_error("sp_reg_eval: invalid argument");
            return SP_ERR_INVALID;
        }
        int m = 1, prod = 0, rownorm = 0, square = 0;
        switch (in.reg) {
        case SP_REG_L1: break;                                   // sum_js |p_js|
        case SP_REG_L21: rownorm = 1; break;                     // sum_j |p_j|_2          (l21.py:19-21)
        case SP_REG_SQL12: square = 1; break;                    // sum_s (sum_j |p_js|)^2 (squaredl12.py:20-22)
        case SP_REG_SQL21: rownorm = 1; square = 1; break;       // (sum_j |p_j|_2)^2      (squaredl21.py:23-25)
        case SP_REG_OMEGATI:                                     // omegati.py:19-47
        case SP_REG_OMEGACS:                                     // omegacs.py:22-39
            rownorm = in.reg == SP_REG_OMEGACS;
            if (degree == -1) prod = 1;
            else if (degree >= 1 && degree <= SP_MAXDEG) m = degree;
            else {
                sp_set_error("degree must be a positive int (<= %d) or -1 (all).", SP_MAXDEG);
                return SP_ERR_UNSUPPORTED;
            }
            break;
        default: sp_set_error("sp_reg_eval: unknown regularizer id %d", in.reg); return SP_ERR_INVALID;
        }
        if (!rownorm && k > OB_THREADS) {
            sp_set_error("sp_reg_eval: n_components=%d > %d is not supported", k, OB_THREADS);
            return SP_ERR_UNSUPPORTED;
        }
        const int cols = rownorm ? 1 : k;
        // rows per block: at least one full step of the block's row stride, at most OB_MAXBLK blocks
        const int step = rownorm ? OB_THREADS / 8 : (OB_THREADS / k);
        int rpb = (d + OB_MAXBLK - 1) / OB_MAXBLK;
        rpb = ((rpb + step - 1) / step) * step;
        if (rpb < step * 4) rpb = step * 4;
        int nb = (d + rpb - 1) / rpb;
        if (nb < 1) nb = 1;
        double (*part)[OB_ST] = reinterpret_cast<double (*)[OB_ST]>(work + (size_t)b * per_entry);
        const RegEntry e = {in.P_dk, part, part + (size_t)OB_MAXBLK * cols, in.out, m, prod, square, cols, nb, rpb};
        all.e[b] = e;
        if (rownorm) by_rows.e[n_rows++] = e;
        else by_cols.e[n_cols++] = e;
        nb_kind[rownorm] = nb;
        if (cols > max_cols) max_cols = cols;
    }
    if (n_entries == 0) return SP_OK;
    if (n_cols > 0) reg_partial_cols_kernel<<<dim3(nb_kind[0], n_cols), OB_THREADS, 0, st>>>(by_cols, d, k);
    if (n_rows > 0) {
        const dim3 grid(nb_kind[1], n_rows);
        if (k > 16) reg_partial_rows_kernel<32><<<grid, OB_THREADS, 0, st>>>(by_rows, d, k);
        else if (k > 8) reg_partial_rows_kernel<16><<<grid, OB_THREADS, 0, st>>>(by_rows, d, k);
        else reg_partial_rows_kernel<8><<<grid, OB_THREADS, 0, st>>>(by_rows, d, k);
    }
    SP_LAUNCH_CHECK("reg_partial_kernel");
    reg_combine_kernel<<<dim3(max_cols, n_entries), OB_CT, 0, st>>>(all);
    SP_LAUNCH_CHECK("reg_combine_kernel");
    reg_final_kernel<<<n_entries, 32, 0, st>>>(all);
    SP_LAUNCH_CHECK("reg_final_kernel");
    return SP_OK;
}

extern "C" int sp_reg_eval(const double *P_dk, int d, int k, int reg, int degree, double *work, double *out,
                           sp_stream stream) {
    const sp_reg_entry e = {P_dk, reg, out};
    return sp_reg_eval_multi(&e, 1, d, k, degree, work, stream);
}
