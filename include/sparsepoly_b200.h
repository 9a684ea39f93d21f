/*
 * sparsepoly_b200.h -- C ABI of the B200-native solver backend for sparsepoly.
 *
 * This is the drop-in boundary for ONE path of the reference: the per-epoch solver loops
 * (pcd / pbcd / psgd), the ANOVA / all-subsets kernels they are built on, the fused loss
 * derivatives and the regularizers' proximal operators.  In the reference that boundary is the
 * call from the Python fit drivers into numba @njit functions with numpy arrays mutated in
 * place (SURVEY.md section 8b); here it is Python -> ctypes -> these entry points with DEVICE
 * arrays mutated in place.  Each entry point cites the reference function it replaces.
 *
 * Conventions
 *   - every pointer is a CUDA device pointer unless its name ends in _host;
 *   - fp64 values, int32 indices / indptr (reference dataset.py:60-66);
 *   - `stream` is a cudaStream_t (0 = default stream); all calls are asynchronous;
 *   - return value: SP_OK (0) or an error code; sp_last_error() gives the message
 *     (thread-local).  Unsupported solver x regularizer x degree combinations return
 *     SP_ERR_UNSUPPORTED with the reference's wording where it has one;
 *   - calls sharing buffers must be issued on one stream; a handle-free API: all state lives
 *     in caller-owned device buffers (PyTorch tensors in the Python host layer).
 *   - loss ids : 0 squared, 1 logistic, 2 squared_hinge        (reference loss.py:13-71)
 *   - reg ids  : 0 l1, 1 l21, 2 squaredl12, 3 squaredl21, 4 omegati, 5 omegacs
 *                                                   (reference regularizer/__init__.py:8-15)
 *   - degree == -1 selects the all-subsets kernel (reference pcd_all.py:41, omegati.py:53).
 */
#ifndef SPARSEPOLY_B200_H
#define SPARSEPOLY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SP_ABI_VERSION 4
#define SP_MAX_HOT_FEATURES 16
#define SP_PBCD_ENT_PER_SLOT 3  /* pbcd window plan: hot nonzeros per window <= 3*slot_cap (pcd: 2*slot_cap) */
#define SP_WINDOW_MAX 256    /* most positions per window of the pipelined sweep */
#define SP_WPLAN_NO_SPECULATION 1   /* sp_wplan.flags: workers always wait for the write-backs they depend on;
                                       bits 8..15 (debug): a window speculates when <= 1/value of its
                                       coordinates start nonzero (0 = built-in default: <= 55 %) */

#define SP_PSGD_CHUNK 64      /* nonzeros per chunk of a long column in the planned psgd column pass */
#define SP_PSGD_SHORT 8       /* columns of at most this many nonzeros are summed by one group of lanes */
#define SP_PSGD_BAND_CAP 2048 /* band values per column and rank of the squared-l1,2 selection */
#define SP_MAX_RANKS 8        /* most ranks (GPUs of one NVSwitch domain) a psgd fit is sharded over */
#define SP_PSGD_CHANNELS 3    /* flag channels per rank: 0 step barriers, 1 exchanges inside the selection, 2 early pull */

typedef void *sp_stream;

enum { SP_STATUS_OK = 0, SP_STATUS_INVALID = 1, SP_STATUS_UNSUPPORTED = 2, SP_STATUS_CUDA = 3 };

/* Device-resident design matrix in both layouts (replaces CSRDataset / CSCDataset,
 * reference dataset.py:69-116).  Unused layouts may be NULL: psgd / predict need CSR,
 * pcd / pbcd need CSC (sweeps) and CSR (cache precompute).  Within a row / column the indices
 * must be strictly increasing. */
typedef struct sp_dataset {
    int32_t n_samples, n_features;
    int64_t nnz;
    const int32_t *csr_indptr, *csr_indices;
    const double *csr_data;
    const int32_t *csc_indptr, *csc_indices;
    const double *csc_data;
    /* optional (may be NULL / 0): dense features, used by sp_psgd_grad to pre-reduce their
     * gradient rows per warp instead of issuing one atomic per sample.  feat_hot[j] = slot
     * 0..n_hot_feat-1 or -1; hot_feat[slot] = j. */
    const int8_t *feat_hot;
    const int32_t *hot_feat;
    int32_t n_hot_feat;
} sp_dataset;

/* Coordinate-order plan for the sequential sweeps (built by sp_plan_partition + sp_plan_order).
 * n_cta = width of the thread-block cluster; samples are range-partitioned over its CTAs. */
typedef struct sp_plan {
    int32_t n_cta;            /* power of two, 1..16 */
    int32_t threads;          /* threads per CTA, multiple of 32, 32..256 */
    const int32_t *pos_ptr;   /* [d*(n_cta+1)] CSC offsets of the per-CTA slices, by position */
    const int32_t *flag_idx;  /* [nnz] CSC row index | 0x80000000 when the sample also occurs in
                                 the column visited at the previous position, | 0x40000000 when
                                 it occurs in the one before that */
    const int32_t *idx_feat;  /* [d] coordinate order (indices_feature in the reference) */
    const int32_t *pos_conf;  /* [d] 1 when the columns at positions t-1 and t share a sample */
    const struct sp_wplan *win; /* non-NULL: run sp_pcd_epoch / sp_cd_linear_epoch as the
                                 pipelined window sweep (the cluster fields above are ignored) */
} sp_plan;

/* Window plan of the pipelined sweep (built by sp_wplan_flag + sp_wplan_fill; wplan.cu).  The
 * coordinate order is cut into windows of `window` positions.  A nonzero is HOT when its sample
 * has another nonzero in a column visited within `horizon` windows; hot nonzeros are handled by
 * one engine CTA that keeps the window's hot sample records in shared memory slots, cold ones by
 * all other CTAs in bulk. */
typedef struct sp_wplan {
    int32_t window, horizon, n_windows, slot_cap;
    int32_t near, flags;      /* hot nonzeros whose slot was last touched <= near positions back are
                                 "late": evaluated by the engine's chain warp itself; flags: SP_WPLAN_* */
    const int32_t *cflag;     /* [nnz] CSC row index | 0x80000000 when the nonzero is hot */
    const int32_t *ht_ptr;    /* [d+1] offsets of the hot nonzeros of position t */
    const int32_t *ht_cls;    /* [d] per position: #late-only | #late+fwd << 8 | #fwd-only << 16 (the
                                 position's hot nonzeros are stored in that class order) */
    const int32_t *h_sd;      /* [n_hot] slot | (dep+1) << 16 | fwd << 29 | late << 30; dep = window-local
                                 position that last touched the slot, -1 = none */
    const double *h_x;        /* [n_hot] value */
    const int32_t *n_slots;   /* [n_windows] distinct hot samples */
    const int32_t *slot_row;  /* [n_windows*slot_cap] sample index of every slot */
    int32_t *sync;            /* [4*(n_windows+2)+2] scratch counters (zeroed by every sweep) */
    double *res;              /* [2*d] scratch: (update, new value) per position */
    double *base;             /* [2*d] scratch: cold partial sums (g, h) per position */
} sp_wplan;

int sp_abi_version(void);
const char *sp_last_error(void);
int sp_device_count(int *count_host);
/* make `device` current for this thread's subsequent calls (cudaSetDevice) */
int sp_set_device(int device);

/* Per-kernel-class CUDA-event timing (bench instrumentation).  Classes: 0 row DP kernels,
 * 1 regularizer caches, 2 pcd/linear sweeps, 3 pbcd sweeps, 4 psgd gradient, 5 psgd dense step,
 * 6 prox, 7 plan.  collect() synchronises and returns accumulated ms / launches since enable. */
int sp_profile_enable(int on);
int sp_profile_collect(double *ms_host /*[8]*/, long long *launches_host /*[8]*/);

/* ------------------------------------------------------------------ dataset / plan helpers */
/* out[j] = sum_i x_ij^2   (row_norms(X.T, squared=True), sparse_factorization_machines.py:409) */
int sp_col_norm_sq(const sp_dataset *ds, double *out, sp_stream stream);
/* col_part[j*(n_cta+1)+c]: CSC offset where CTA c's sample range starts in column j */
int sp_plan_partition(const sp_dataset *ds, int n_cta, int32_t *col_part, sp_stream stream);
/* position table + hazard flags for the order idx_feat (call again after every shuffle) */
int sp_plan_order(const sp_dataset *ds, int n_cta, const int32_t *col_part, const int32_t *idx_feat,
                  int32_t *pos_ptr, int32_t *flag_idx, int32_t *pos_conf, sp_stream stream);
/* Window plan, step 1: pos_scratch [d]; cflag [nnz] and hot_count [d] (hot nonzeros per position)
 * are written.  The caller turns hot_count into ht_ptr (exclusive prefix sum, d+1 entries). */
int sp_wplan_flag(const sp_dataset *ds, const int32_t *idx_feat, int window, int horizon,
                  int32_t *pos_scratch, int32_t *cflag, int32_t *hot_count, sp_stream stream);
/* Window plan, step 2: fills h_sd / h_x [ht_ptr[d]] (tmp_sd / tmp_x: scratch of the same size),
 * ht_cls [d], n_slots [n_windows], slot_row [n_windows*slot_cap]; *overflow is set to 1 when a window
 * needs more than slot_cap slots, more than ent_per_slot*slot_cap hot nonzeros, or a position has more than 32
 * chain-warp nonzeros (retry with a smaller window). */
int sp_wplan_fill(const sp_dataset *ds, const int32_t *idx_feat, int window, int slot_cap, int ent_per_slot, int near,
                  const int32_t *cflag, const int32_t *ht_ptr, int32_t *tmp_sd, double *tmp_x,
                  int32_t *h_sd, double *h_x, int32_t *ht_cls, int32_t *n_slots, int32_t *slot_row,
                  int32_t *overflow, sp_stream stream);
/* same for the pbcd window sweep (records = A[i,:,:] + {y_pred, y}); 0 when n_components > 32 (the
 * window engine handles k <= 32, wider models use the cluster sweep).  A pbcd window plan is
 * built with near = 0, window <= 64, res of 2*d*k doubles and base of sp_pbcd_wplan_base_doubles(). */
int sp_pbcd_wplan_slot_cap(int degree, int k);
/* doubles the `base` buffer of a pbcd window plan must hold (ring of cold partial sums) */
size_t sp_pbcd_wplan_base_doubles(void);
/* debug: cycle counters of the window sweep's roles (zeros unless the library was built with
 * -DSP_WPROF); out_host [16] */
int sp_wprof_read(unsigned long long *out_host);
/* zero-update speculation of the window sweep: out_host[0] = positions evaluated speculatively,
 * out_host[1] = speculations rejected (redone exactly), since the last call */
int sp_wspec_read(unsigned long long *out_host /*[2]*/);
/* debug: per-position timestamps of window 100 of the last sweep; out_host [SP_WINDOW_MAX*8] */
int sp_wtrace_read(long long *out_host);
/* slots (hot sample records) the engine CTA can hold in shared memory for records of this stride */
/* most hot-record slots per window the engine CTA can stage for this record stride (always even;
 * sp_wplan.slot_cap must be even and <= this) */
int sp_wplan_slot_cap(int rec_stride);
/* out[c*rows+r] = in[r*cols+c] */
int sp_transpose_f64(const double *in, double *out, int rows, int cols, sp_stream stream);
/* the same for `batch` (<= 65535) consecutive matrices in one launch: matrix b is in[b*rows*cols ...] -> out[b*rows*cols ...] */
int sp_transpose_f64_batch(const double *in, double *out, int batch, int rows, int cols, sp_stream stream);
/* doubles per sample record {y_pred, y, A^1..A^(m-1)} for a model of this top degree */
int sp_rec_stride(int degree);

/* ------------------------------------------------------------------------------ prediction */
/* out[i*out_stride] (+)= <w,x_i> + sum_s lams[s] * K(P[:,s], x_i)    (kernels.poly_predict,
 * reference kernels.py:140-153; K = ANOVA degree-m DP or all-subsets product).
 * P_dk is feature-major [d,k]; w may be NULL; accumulate != 0 adds to out. */
int sp_predict(const sp_dataset *ds, const double *P_dk, int k, const double *lams, int degree,
               const double *w, double *out, int out_stride, int accumulate, sp_stream stream);

/* Prediction of many models on one design matrix (decision_function_many; DESIGN.md 3.1).  One descriptor per model,
 * passed as a host array of at most SP_PREDICT_MAX_MODELS entries; the call is one launch over all models (the table
 * travels as a kernel parameter), and each model's rows are computed by the code sp_predict runs, so every model's
 * output is bit-identical to sp_predict with the same arguments.  sp_predict is the one-model case of this call.
 * k, degree, out_stride and accumulate hold for every model.  Models may share P_dk, lams and w, never out. */
#define SP_PREDICT_MAX_MODELS 256
typedef struct sp_predict_model {
    const double *P_dk;       /* [d,k] feature-major */
    const double *lams;       /* [k] */
    const double *w;          /* [d] or NULL (no linear term) */
    double *out;              /* out[i*out_stride] (+)= the model's output for sample i */
} sp_predict_model;
int sp_predict_multi(const sp_dataset *ds, const sp_predict_model *models, int n_models, int k, int degree,
                     int out_stride, int accumulate, sp_stream stream);

/* K[i*k+s] = K(P[:,s], x_i): the Gram matrix of kernels.anova_kernel (kernels.py:71-115) /
 * kernels.all_subsets_kernel (kernels.py:118-137, degree=-1). */
int sp_kernel_matrix(const sp_dataset *ds, const double *P_dk, int k, int degree, double *K,
                     sp_stream stream);

/* --------------------------------------------------------------------------- pcd / linear */
/* One pass of exact coordinate descent on w (cd_linear._cd_linear_epoch, cd_linear.py:8-33).
 * rec is the per-sample record array (y_pred at +0, y at +1); *viol accumulates sum |update|. */
int sp_cd_linear_epoch(const sp_dataset *ds, const sp_plan *plan, double *w,
                       const double *col_norm_sq, double alpha, int loss, double *rec,
                       int rec_stride, double *viol, sp_stream stream);

/* One pcd epoch over all k components of one order (pcd.pcd_epoch, pcd.py:71-137; degree=-1:
 * pcd_all.pcd_epoch, pcd_all.py:44-102).  P_kd is component-major [k,d] (the reference's
 * P_[order]); lams [k]; regstate >= 8 doubles of scratch; idx_comp_host = indices_component. */
int sp_pcd_epoch(const sp_dataset *ds, const sp_plan *plan, double *P_kd, int k, const double *lams,
                 int degree, double beta, double gamma, double eta, int reg, int loss, double *rec,
                 int rec_stride, double *regstate, double *viol, const int32_t *idx_comp_host,
                 sp_stream stream);

/* Many pcd models on one design matrix (fit_many; DESIGN.md 3.2).  One descriptor per model, passed as a
 * host array.  Every launch of a call covers all models, and each model's sweep is the code the single-model
 * call runs on that model's P, records and scratch, so its result is bit-identical to sp_pcd_epoch /
 * sp_cd_linear_epoch with a cluster plan of the same n_cta / threads.  Models may share a plan (the same
 * coordinate order), never P, rec, regstate or viol.  At most 65535 models per call. */
typedef struct sp_pcd_model {
    const int32_t *pos_ptr, *flag_idx, *idx_feat, *pos_conf;  /* the model's cluster plan (sp_plan fields,
                                                                 built for the call's n_cta) */
    double *P;                /* P_kd [k,d] of the order (sp_pcd_epoch_multi) or w [d] (sp_cd_linear_epoch_multi) */
    const double *lams;       /* [k] (unused by the linear sweep) */
    double ab;                /* beta (pcd) or alpha (linear) */
    double gamma, eta;        /* unused by the linear sweep */
    int32_t reg;              /* reg id: l1, squaredl12 or omegati (unused by the linear sweep) */
    double *rec;              /* [n*rec_stride] the model's sample records */
    double *regstate;         /* >= 8 doubles of scratch (unused by the linear sweep) */
    double *viol;             /* the model's running sum of |updates| */
    const int32_t *idx_comp_host; /* [k] the model's indices_component (unused by the linear sweep) */
} sp_pcd_model;

/* cd_linear._cd_linear_epoch (cd_linear.py:8-33) of every model: one launch. */
int sp_cd_linear_epoch_multi(const sp_dataset *ds, int n_cta, int threads, const double *col_norm_sq,
                             const sp_pcd_model *models, int n_models, int loss, int rec_stride, sp_stream stream);

/* pcd.pcd_epoch (pcd.py:71-137; degree=-1: pcd_all.pcd_epoch, pcd_all.py:44-102) of one order of every model.
 * Position ss of the component orders is one row-DP launch, one regularizer-cache launch (models other than
 * l1) and one sweep launch over all models; a model's dead components (the rule of sp_pcd_epoch) get no entry,
 * and a launch without entries is not issued.  One stream synchronisation per call (the dead-component scan). */
int sp_pcd_epoch_multi(const sp_dataset *ds, int n_cta, int threads, const sp_pcd_model *models, int n_models,
                       int k, int degree, int loss, int rec_stride, sp_stream stream);

/* ----------------------------------------------------------------------------------- pbcd */
/* One pbcd epoch (pbcd.pbcd_epoch, pbcd.py:82-148; degree=-1: pbcd_all.pbcd_epoch,
 * pbcd_all.py:68-132).  P_dk feature-major [d,k]; yrec [n,2] = {y_pred, y};
 * A [n,(m-1),k] (ANOVA) or [n,k] (all-subsets) scratch; reg_norms [d] and regstate [>=16]
 * regularizer scratch. */
int sp_pbcd_epoch(const sp_dataset *ds, const sp_plan *plan, double *P_dk, int k, const double *lams,
                  int degree, double beta, double gamma, double eta, int reg, int loss, double *yrec,
                  double *A, double *reg_norms, double *regstate, double *viol, sp_stream stream);

/* Many pbcd models on one design matrix (fit_many; DESIGN.md 3.3).  One descriptor per model, passed as a host
 * array.  One call runs one order of every model in at most four launches, each covering all models: the row DP,
 * the row norms and the regularizer caches (only if a model has squaredl21 or omegacs) and the block sweep, one
 * cluster of n_cta CTAs per model.  Each model's result is bit-identical to sp_pbcd_epoch with a cluster plan of
 * the same n_cta / threads.  Models may share a plan (the same feature order), never P, yrec, A, reg_norms,
 * regstate or viol.  At most 65535 models per call. */
typedef struct sp_pbcd_model {
    const int32_t *pos_ptr, *flag_idx, *idx_feat;  /* the model's cluster plan (sp_plan fields, built for the
                                                      call's n_cta) */
    double *P;                /* P_dk [d,k] of the order, feature-major */
    const double *lams;       /* [k] */
    double beta, gamma, eta;
    int32_t reg;              /* reg id: l1, l21, squaredl21 (degree 2 only) or omegacs */
    double *yrec;             /* [n,2] {y_pred, y} */
    double *A;                /* [n,(m-1),k] (ANOVA) or [n,k] (all-subsets) scratch */
    double *reg_norms;        /* [d] regularizer scratch */
    double *regstate;         /* >= 16 doubles of regularizer scratch */
    double *viol;             /* the model's running sum of |updates| */
} sp_pbcd_model;

/* pbcd.pbcd_epoch (pbcd.py:82-148; degree=-1: pbcd_all.pbcd_epoch, pbcd_all.py:68-132) of one order of every
 * model.  n_cta: power of two <= 16; threads: multiple of 32 <= 256; k <= 128. */
int sp_pbcd_epoch_multi(const sp_dataset *ds, int n_cta, int threads, const sp_pbcd_model *models, int n_models,
                        int k, int degree, int loss, sp_stream stream);

/* ----------------------------------------------------------------------------------- psgd */
/* (eta_P, eta_w) of psgd._get_eta (psgd.py:9-22); host-side scalar helper. */
int sp_get_eta(int learning_rate, double eta0, double alpha, double beta, double power_t,
               int64_t it, double *eta_P_host, double *eta_w_host);

/* The dense-gradient psgd path (every regularizer; the only one for l21 / squaredl21, and the
 * cross-check of the planned path below for l1 / squaredl12).
 * Minibatch gradient: samples idx_samples[b0..b1) (psgd._pred + _update_grads, psgd.py:47-91).
 * P_odk [n_orders,d,k]; grad_P same shape and grad_w [d] are accumulated into (fp64 atomics: the sum
 * order is not fixed); *loss_sum accumulates sum of losses at the pre-update parameters. */
int sp_psgd_grad(const sp_dataset *ds, const double *y, const double *P_odk, int n_orders, int k,
                 const double *w, const double *lams, int degree, int loss, int fit_linear,
                 const int32_t *idx_samples, int b0, int b1, double *grad_P, double *grad_w,
                 double *loss_sum, sp_stream stream);

/* SGD step + zeroing of the gradients (psgd._update_params without the prox, psgd.py:94-117,
 * :195-196):  P = (P - (eta_P/batch)*grad_P) / (1 + eta_P*beta), same for w with alpha. */
int sp_psgd_step(double *P_odk, double *grad_P, double *w, double *grad_w, int n_orders, int d, int k,
                 double eta_P, double eta_w, double alpha, double beta, int batch, int fit_linear,
                 sp_stream stream);

/* regularizer.prox on one order P_dk [d,k] (l1.py:50-51, l21.py:43-48, squaredl12.py:66-78,
 * squaredl21.py:63-74, regularizer/utils.py:26-70).  work: >= d + 8*k + 64 doubles. */
int sp_prox(double *P_dk, int d, int k, int reg, double strength, double *work, sp_stream stream);

/* doubles of scratch sp_prox / sp_psgd_epoch need for a [d,k] matrix */
size_t sp_prox_work_doubles(int d, int k);

/* Whole single-GPU psgd epoch = psgd.psgd_epoch (psgd.py:125-199) on the dense-gradient path: loops the
 * three calls above over the minibatches; *it_io_host is advanced once per parameter update. */
int sp_psgd_epoch(const sp_dataset *ds, const double *y, double *P_odk, int n_orders, int k, double *w,
                  const double *lams, int degree, double alpha, double beta, double gamma, int reg,
                  int loss, double *grad_P, double *grad_w, const int32_t *idx_samples,
                  int fit_linear, double eta0, int learning_rate, double power_t, int batch_size,
                  int64_t *it_io_host, double *loss_sum, double *work, sp_stream stream);


/* ------------------------------------------------------------------- planned psgd (l1 / squaredl12) */
/* "Batch CSC" plan of one sample order (built by the host layer with device sorts; psgd_plan.py): the
 * nonzeros of every minibatch regrouped by feature, samples ascending inside a feature -- the order in
 * which psgd._update_grads (psgd.py:60-91) adds them.  Minibatch m covers local positions
 * [m*batch_local, min((m+1)*batch_local, n_local)) of idx_samples.  Arrays named *_host live in host
 * memory, all others on the device.  Sharded plans (world > 1) order a minibatch's columns by
 * (owner = feature % world, feature) and carry the owner-side tables. */
typedef struct sp_psgd_plan {
    int32_t n_minibatches, batch_local, n_local;
    int32_t chunk, short_max;      /* must equal SP_PSGD_CHUNK / SP_PSGD_SHORT */
    const int64_t *mb_eptr_host;   /* [M+1] first nonzero of every minibatch */
    const int64_t *mb_uptr_host;   /* [M+1] first column (distinct feature) of every minibatch */
    const int64_t *mb_sgptr_host;  /* [M+1] first entry of sg_* */
    const int64_t *mb_shptr_host;  /* [M+1] first entry of sc_ptr / sc_u / sc_feat */
    const int64_t *mb_lcptr_host;  /* [M+1] first entry of lc_u / lc_e0 */
    const int64_t *mb_mlptr_host;  /* [M+1] first entry of ml_u / ml_c0 */
    const int32_t *e_pos;          /* [E] position of the sample inside its minibatch */
    const double *e_x;             /* [E] value */
    const int32_t *u_feat;         /* [U] feature id of every column */
    const int64_t *u_ptr;          /* [U+1] first nonzero of every column */
    const int32_t *sg_u, *sg_feat, *sg_pos; /* [N1] columns of ONE nonzero: column, feature, position of the sample ... */
    const double *sg_x;            /* [N1] ... and value */
    const int64_t *sc_ptr;         /* [Ns+1] columns of 2..short_max nonzeros: offsets into sc_pos / sc_x (their nonzeros,
                                      samples ascending, stored compactly) ... */
    const int32_t *sc_u, *sc_feat; /* [Ns] ... column and feature */
    const int32_t *sc_pos;         /* [Es] position of the sample inside its minibatch */
    const double *sc_x;            /* [Es] value */
    const int32_t *lc_u;           /* [Nc] chunks of the longer columns: column ... */
    const int32_t *lc_feat;        /* [Nc] ... its feature ... */
    const int32_t *lc_cnt;         /* [Nc] ... nonzeros in the chunk, | 0x40000000 when it is the column's only chunk ... */
    const int64_t *lc_e0;          /* [Nc] ... and first nonzero; a chunk ends after `chunk` nonzeros or with its column */
    const int32_t *ml_u;           /* [Nm] columns of more than one chunk ... */
    const int32_t *ml_c0;          /* [Nm] ... and the index of their first chunk inside the minibatch's chunk list */
    int64_t max_chunks;            /* most chunks in one minibatch (sizes part_g / part_w) */
    int64_t max_cols;              /* most columns in one minibatch (sizes the staging buffers) */
    /* sharded only */
    const int32_t *csr_slot;       /* [nnz] per CSR nonzero: index of its feature in its minibatch's columns */
    const int32_t *mb_owner_start_host; /* [M][world+1] first column of every owner inside the minibatch */
    const int64_t *mb_optr_host;   /* [M+1] first entry of own_q / own_src */
    const int32_t *own_q;          /* [O] rows (feature / world) of this rank touched by the GLOBAL minibatch */
    const int32_t *own_src;        /* [O][world] index of that row in the inbox region of every rank, or -1 */
} sp_psgd_plan;

/* State of a planned psgd fit: model, scratch and (sharded) peer pointers.  P / w hold RAW values in the
 * lazy frame  value = soft_threshold(raw, thr[column]) / C  (w: raw / Cw) between sp_psgd_plan_begin and
 * the materialising sp_psgd_plan_end; C, Cw, seq* are maintained by the library.  When sharded, P / w
 * are this rank's rows j % world == rank (d_rows = ceil(d / world)) and the peer_* pointers come from
 * sp_ipc_open (CUDA IPC, peer memory over NVLink). */
typedef struct sp_psgd_ctx {
    double *P, *w;                 /* [n_orders, d_rows, k], [d_rows] */
    const double *lams;            /* [k] */
    double *thr;                   /* [n_orders*k] raw-space thresholds */
    int32_t n_orders, k, d_rows, degree, reg, loss, fit_linear;
    int32_t world, rank;
    double *bufA, *bufdL;          /* [batch_local, arows*k], [batch_local]: per-sample tables of one minibatch */
    double *sample_loss;           /* [n_local] */
    double *part_g, *part_w;       /* [max_chunks, n_orders*k], [max_chunks] */
    double *work;                  /* sp_psgd_plan_work_doubles() */
    double *xwork;                 /* sp_psgd_plan_xwork_doubles(): statistics boxes (peer-visible when sharded) */
    double C, Cw;
    uint64_t seq, seq_generic;
    /* sharded only */
    double *stage, *stage_w;       /* [max_cols, n_orders, k], [max_cols] */
    double *inbox_g, *inbox_w;     /* [world, inbox_cap, n_orders*k], [world, inbox_cap] (peer-visible) */
    int64_t inbox_cap;
    int32_t *err;                  /* device flag: a cross-rank wait timed out */
    double *peer_P[SP_MAX_RANKS], *peer_w[SP_MAX_RANKS];
    double *peer_inbox_g[SP_MAX_RANKS], *peer_inbox_w[SP_MAX_RANKS];   /* region of THIS rank in rank r's inbox */
    double *peer_xwork[SP_MAX_RANKS];
    uint64_t *peer_flags[SP_MAX_RANKS];    /* [SP_PSGD_CHANNELS][SP_MAX_RANKS] per rank; [rank] is local */
    /* owned by the library (zero-initialised by the caller, released by sp_psgd_plan_release): the stream and
     * events of the early pull -- the next minibatch's rows are fetched from the owners while this minibatch's
     * selection runs -- and that channel's sequence number */
    uint64_t seq_pull;
    void *aux_stream, *aux_event[2];
} sp_psgd_ctx;

size_t sp_psgd_plan_work_doubles(int n_orders, int k);
size_t sp_psgd_plan_xwork_doubles(int n_orders, int k, int world);
/* start of a fit: thresholds, scales and the selection state are reset (P / w hold the model) */
int sp_psgd_plan_begin(sp_psgd_ctx *ctx, sp_stream stream);
/* minibatches [m_begin, m_end) of psgd.psgd_epoch (psgd.py:150-198): per minibatch the rows pass
 * (_pred, psgd.py:47-57), the column pass (_update_grads + the SGD step of _update_params,
 * psgd.py:60-117, on the touched rows only) and the prox (psgd.py:119-122) as a lazily applied column
 * threshold; *it_io_host advances once per minibatch.  After a minibatch that takes C or Cw out of
 * (1e-100, 1e100) the frame is folded into P / w (thr = 0, C = Cw = 1), so the scales never overflow. */
int sp_psgd_plan_run(sp_psgd_ctx *ctx, const sp_dataset *ds, const sp_psgd_plan *plan, const double *y,
                     const int32_t *idx_samples, double alpha, double beta, double gamma, double eta0,
                     int learning_rate, double power_t, int m_begin, int m_end, int64_t *it_io_host,
                     sp_stream stream);
/* end of an epoch: *loss_sum (device, may be NULL) += sum of the per-sample losses of positions
 * [0, n_local) in fixed order; materialize != 0 rewrites P / w as the model (thr = 0, C = Cw = 1). */
int sp_psgd_plan_end(sp_psgd_ctx *ctx, int n_local, double *loss_sum, int materialize, sp_stream stream);
/* the model the lazy frame represents, written to device buffers without changing ctx (training continues in the
 * same frame): P_out[o, s, j] = soft_threshold(P[o, j, s], thr[o*k+s]) / C in the component-major [n_orders, k, d]
 * layout of the estimators' P_, w_out = w / Cw (w when !fit_linear).  Bit-identical to the materialising
 * sp_psgd_plan_end followed by a transpose.  Single rank only (SP_ERR_UNSUPPORTED when world > 1). */
int sp_psgd_plan_read(const sp_psgd_ctx *ctx, double *P_out, double *w_out, sp_stream stream);
/* destroys the library-owned stream / events of ctx (idempotent) */
int sp_psgd_plan_release(sp_psgd_ctx *ctx);

/* diagnostics of the squared-l1,2 selection since sp_psgd_plan_begin (synchronises the stream): out_host[0] = prox
 * calls, [1] = solved from the band, [2] = needed generic passes, [3] = band half-width, [4] / [5] = mean / largest
 * band size per column at the last call */
int sp_psgd_plan_solver_stats(const sp_psgd_ctx *ctx, double *out_host /*[6]*/, sp_stream stream);

/* peer-visible device memory for the sharded path (cudaMalloc + CUDA IPC); handle64: 64 bytes */
int sp_shm_alloc(size_t bytes, void **out_host);
int sp_shm_free(void *p);
int sp_ipc_export(void *p, unsigned char *handle64_host);
int sp_ipc_open(const unsigned char *handle64_host, void **out_host);
int sp_ipc_close(void *p);
/* kind: 0 host->device, 1 device->host (synchronises the stream), 2 device->device */
int sp_memcpy(void *dst, const void *src, size_t bytes, int kind, sp_stream stream);

/* ------------------------------------------------------------------------------ objective */
/* The quantity the reference's update rules minimise but never evaluate
 * (sparse_factorization_machines.py:181-188, :265-272):
 *     sum_i loss(y_pred_i, y_i) + alpha/2 |w|^2 + beta/2 |P|^2 + gamma * Omega(P).
 * Three device reductions give its parts; each overwrites out[0] (device) and is deterministic.
 *
 * sp_loss_sum: sum_i loss(y_pred[i*pred_stride], y[i*y_stride])   (loss.py:19-20, :34-41, :61-65);
 *              the strides let it read the pcd sample records {y_pred, y, ...} in place.
 * sp_sqnorm  : sum_i v[i]^2.
 * work for both: sp_sum_work_doubles() doubles. */
int sp_loss_sum(const double *y_pred, int pred_stride, const double *y, int y_stride, int n, int loss,
                double *work, double *out, sp_stream stream);
int sp_sqnorm(const double *v, int64_t len, double *work, double *out, sp_stream stream);
size_t sp_sum_work_doubles(void);

/* Omega(P) of one order, P_dk feature-major [d,k] -- the regularizer classes' `eval`:
 *   l1         sum_js |p_js|                                  (l1.py:17-18, entrywise)
 *   l21        sum_j |p_j|_2                                  (l21.py:19-21)
 *   squaredl12 sum_s (sum_j |p_js|)^2                         (squaredl12.py:20-22)
 *   squaredl21 (sum_j |p_j|_2)^2                              (squaredl21.py:23-25)
 *   omegati    sum_s e_degree(|p_1s|..|p_ds|); degree=-1: sum_s prod_j (1+|p_js|)  (omegati.py:19-47)
 *   omegacs    e_degree(|p_1|_2..|p_d|_2);     degree=-1: prod_j (1+|p_j|_2)      (omegacs.py:22-39)
 * (e_m = m-th elementary symmetric polynomial).  degree is ignored by the first four.
 * work: sp_reg_eval_work_doubles(d, k) doubles. */
int sp_reg_eval(const double *P_dk, int d, int k, int reg, int degree, double *work, double *out,
                sp_stream stream);
size_t sp_reg_eval_work_doubles(int d, int k);

/* Many reductions of one length in one call (objective_many; DESIGN.md 3.5): host arrays of at most
 * SP_OBJECTIVE_MAX_ENTRIES entries, each launch covers all entries (the table travels as a kernel parameter), and
 * entry b's result is bit-identical to the single call on its arguments (the same blocks, partials and fixed tree),
 * which is the one-entry case of these.  Work buffers are per entry: n_entries x sp_sum_work_doubles() doubles for the
 * sums, n_entries x sp_reg_eval_work_doubles(d, k) for Omega; entry b uses the b-th slice.
 *   sp_loss_sum_multi: entry b: out[0] = sum_i loss_b(y_pred[i*pred_stride], y[i*y_stride]), i < n;
 *   sp_sqnorm_multi  : entry b: out[0] = sum_i v[i]^2, i < len;
 *   sp_reg_eval_multi: entry b: out[0] = Omega_reg(P_dk) of a [d,k] matrix at this degree; at most two partial
 *                      launches (column-fold and row-norm regularizers), one combine and one final launch. */
#define SP_OBJECTIVE_MAX_ENTRIES 256
typedef struct sp_loss_entry {
    const double *y_pred, *y;
    int32_t loss;             /* loss id */
    double *out;
} sp_loss_entry;
typedef struct sp_sqnorm_entry {
    const double *v;
    double *out;
} sp_sqnorm_entry;
typedef struct sp_reg_entry {
    const double *P_dk;       /* [d,k] feature-major */
    int32_t reg;              /* reg id */
    double *out;
} sp_reg_entry;
int sp_loss_sum_multi(const sp_loss_entry *entries, int n_entries, int pred_stride, int y_stride, int n,
                      double *work, sp_stream stream);
int sp_sqnorm_multi(const sp_sqnorm_entry *entries, int n_entries, int64_t len, double *work, sp_stream stream);
int sp_reg_eval_multi(const sp_reg_entry *entries, int n_entries, int d, int k, int degree, double *work,
                      sp_stream stream);

/* Device input (DESIGN.md 2): a design matrix that is already on the GPU, checked and converted there.  These are
 * the only entries whose input may be int32 OR int64 (indptr, indices) and fp32 OR fp64 (values).
 *
 * sp_csr_prepare: one pass over a CSR (indptr != NULL; `indptr_i64` / `indices_i64` / `values_f64` pick the types)
 * or a dense strided matrix (indptr == NULL: X[i, j] = values[i*stride_row + j*stride_col], every entry stored).
 * It fills report[SP_CSR_REPORT_LEN] (initialised by the call; "first" entries are the lowest offending row, or
 * INT64_MAX when there is none):
 *   [0] first row i with indptr[i+1] < indptr[i]     [1] indptr[0]       [2] indptr[n_rows] (dense: n_rows*n_cols)
 *   [3] first row with a column outside [0, n_cols)   [4] first row holding a NaN   [5] first row holding +-inf
 *   [6] number of rows whose columns are not strictly increasing      [7] the first of them
 * With out_indptr / out_indices / out_data (all or none) it also writes the int32 / fp64 CSR with n_dummy (<= 32)
 * columns of ones prepended to every row (columns 0..n_dummy-1; the others shift by n_dummy), in the input's order
 * within a row.  nnz is the length of indices / values; a corrupt indptr is reported, never read past nnz.
 *
 * sp_csr_sum_runs: canonicalisation after a stable sort of the keys row*n_cols+col of a CSR: for every run of equal
 * keys (head p: p == 0 or keys[p-1] != keys[p]), out_data[run_index[p]] = data[perm[p]] + data[perm[p+1]] + ...
 * summed left to right and out_indices[run_index[p]] = key % n_cols. */
#define SP_CSR_REPORT_LEN 8
#define SP_CSR_REPORT_DECREASING 0
#define SP_CSR_REPORT_INDPTR0 1
#define SP_CSR_REPORT_INDPTRN 2
#define SP_CSR_REPORT_RANGE 3
#define SP_CSR_REPORT_NAN 4
#define SP_CSR_REPORT_INF 5
#define SP_CSR_REPORT_N_UNSORTED 6
#define SP_CSR_REPORT_UNSORTED 7
int sp_csr_prepare(int64_t n_rows, int64_t n_cols, int64_t nnz, const void *indptr, int indptr_i64,
                   const void *indices, int indices_i64, const void *values, int values_f64, int64_t stride_row,
                   int64_t stride_col, int n_dummy, int32_t *out_indptr, int32_t *out_indices, double *out_data,
                   int64_t *report, sp_stream stream);
int sp_csr_sum_runs(int64_t nnz, const int64_t *keys, const int64_t *perm, const double *data,
                    const int64_t *run_index, int64_t n_cols, int32_t *out_indices, double *out_data,
                    sp_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* SPARSEPOLY_B200_H */
