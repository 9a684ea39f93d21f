// Regularizer cache kernel shared by pcd and pbcd.
#include "common.cuh"

namespace {
// ------------------------------------------------------------------ regularizer cache kernel
// compute_cache_pcd (squaredl12.py:42-45, omegati.py:62-80); block b computes the cache of table[b] in that entry's
// mode from its vector p (a component row of P, or the row norms of pbcd):
//   mode 0 (squaredl12): regstate[0] = sum_j |p_j|
//   mode 1 (omegati FM): regstate[t] = e_t(|p_1|..|p_d|), t = 0..degree  (truncated product of
//                        the polynomials 1 + |p_j| z; the reference folds them left to right,
//                        here each thread folds a contiguous chunk and the chunks are multiplied
//                        in a fixed tree -- all terms are >= 0, so this is well conditioned)
//   mode 2 (omegati all-subsets): regstate[0] = prod_j (1 + |p_j|)
constexpr int RC_THREADS = 1024;
__global__ void __launch_bounds__(RC_THREADS) reg_cache_kernel(const SpRegEntry *__restrict__ table, int degree,
                                                               int d) {
    const SpRegEntry ent = table[blockIdx.x];
    const int mode = ent.mode;
    const double *__restrict__ p = ent.p;
    double *regstate = ent.regstate;
    __shared__ double sh[RC_THREADS][SP_MAXDEG + 1];
    const int tid = threadIdx.x;
    const int m = mode == 1 ? degree : 0;
    double e[SP_MAXDEG + 1];
    for (int t = 0; t <= SP_MAXDEG; t++) e[t] = 0.0;
    e[0] = (mode == 0) ? 0.0 : 1.0;
    const int chunk = (d + RC_THREADS - 1) / RC_THREADS;
    const int lo = tid * chunk, hi = min(d, lo + chunk);
    // one loop per mode: with the mode read from the table, ptxas would not split a shared loop itself, and the
    // sum / product loops then keep one load in flight instead of sixteen
    if (mode == 0)
        for (int j = lo; j < hi; j++) e[0] += fabs(p[j]);
    else if (mode == 2)
        for (int j = lo; j < hi; j++) e[0] *= 1.0 + fabs(p[j]);
    else
        for (int j = lo; j < hi; j++) {
            const double av = fabs(p[j]);
            for (int t = m; t >= 1; t--) e[t] += e[t - 1] * av;
        }
    for (int t = 0; t <= SP_MAXDEG; t++) sh[tid][t] = e[t];
    __syncthreads();
    for (int off = 1; off < RC_THREADS; off <<= 1) {        // fixed tree, left operand first
        if ((tid & (2 * off - 1)) == 0) {
            double l[SP_MAXDEG + 1], r[SP_MAXDEG + 1], o[SP_MAXDEG + 1];
            for (int t = 0; t <= SP_MAXDEG; t++) { l[t] = sh[tid][t]; r[t] = sh[tid + off][t]; }
            if (mode == 0) o[0] = l[0] + r[0];
            else if (mode == 2) o[0] = l[0] * r[0];
            else
                for (int t = 0; t <= m; t++) {
                    double acc = 0.0;
                    for (int u = 0; u <= t; u++) acc += l[u] * r[t - u];
                    o[t] = acc;
                }
            for (int t = 0; t <= m; t++) sh[tid][t] = o[t];
        }
        __syncthreads();
    }
    if (tid == 0)
        for (int t = 0; t <= SP_MAXDEG; t++) regstate[t] = (t <= m) ? sh[0][t] : 0.0;
}

}  // namespace

int sp_launch_reg_cache_multi(const SpRegEntry *table, int n_tab, int degree, int d, cudaStream_t st) {
    if (degree != -1 && (degree < 1 || degree > SP_MAXDEG)) {
        sp_set_error("regularizer cache: degree %d unsupported", degree);
        return SP_ERR_UNSUPPORTED;
    }
    if (n_tab == 0) return SP_OK;
    sp_prof_begin(SP_PROF_REGCACHE, st);
    reg_cache_kernel<<<n_tab, RC_THREADS, 0, st>>>(table, degree, d);
    sp_prof_end(st);
    SP_LAUNCH_CHECK("reg_cache_kernel");
    return SP_OK;
}
