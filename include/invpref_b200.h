/*
 * invpref_b200.h -- C ABI of the B200-native InvPref hot path (libinvpref_b200.so).
 *
 * The reference (AIflowerQ/InvPref_KDD_2022) has no FFI layer: its boundary is the Python
 * API of models.py / train.py, whose arithmetic is stock ATen.  This library replaces that
 * arithmetic for the train step and the EM environment re-assignment; every entry point
 * names the reference code it replaces (paths relative to the reference checkout).
 *
 * Conventions
 *  - All pointers are DEVICE pointers unless the name ends in _host.  The caller owns every
 *    buffer; the library allocates nothing persistent and frees nothing.
 *  - Tables are fp32, row-major, contiguous [rows, dim]; ids / envs are int64 (the reference
 *    uses LongTensor, train.py:708-713); scores / weights are fp32.
 *  - Every call is asynchronous on the given cudaStream_t (passed as void*) and never
 *    synchronises the device.  Return value: 0 = ok, negative = invpref_status.
 *  - There is no CPU fallback: a build without a usable GPU fails at launch with a CUDA error.
 */
#ifndef INVPREF_B200_H
#define INVPREF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define INVPREF_ABI_VERSION 2
#define INVPREF_MAX_ENVS 8      /* drivers use K = 2, 4, 5, 6 */
#define INVPREF_MAX_DIM 256     /* drivers use D = 30, 40; synthetic config D = 64 */
#define INVPREF_NUM_LOSSES 6    /* train.py:836-843: invariant, env_aware, envs, L2, L1, loss */

typedef enum {
    INVPREF_OK = 0,
    INVPREF_ERR_BAD_DIM = -1,        /* dim not in [1, INVPREF_MAX_DIM] or unsupported parity */
    INVPREF_ERR_BAD_ENVS = -2,       /* n_envs not in [1, INVPREF_MAX_ENVS] */
    INVPREF_ERR_BAD_ARG = -3,        /* null pointer / negative size / table too large */
    INVPREF_ERR_MISALIGNED = -4,     /* table base pointer not aligned for the vector width */
    INVPREF_ERR_WORKSPACE = -5,      /* workspace / plan buffer too small */
    INVPREF_ERR_CUDA = -6,           /* cudaGetLastError() != cudaSuccess after a launch */
    INVPREF_ERR_ID_RANGE = -7        /* (debug check) id outside its table */
} invpref_status;

/* models.py:415-446 / 273-305: model shape and variant flags. */
typedef struct {
    int64_t n_users;
    int64_t n_items;
    int32_t n_envs;          /* K */
    int32_t dim;             /* D = factor_num */
    int32_t implicit;        /* 0: InvPrefExplicit (MSE), 1: InvPrefImplicit (sigmoid + BCE) */
    int32_t reg_only_embed;  /* models.py:507-511 */
    int32_t reg_env_embed;   /* models.py:516-517 */
    int32_t _pad;
} invpref_desc;

/* The seven parameter tensors, in model.parameters() order (models.py:424-432). */
typedef struct {
    float* Uinv;  /* embed_user_invariant.weight  [n_users, D] */
    float* Iinv;  /* embed_item_invariant.weight  [n_items, D] */
    float* Uenv;  /* embed_user_env_aware.weight  [n_users, D] */
    float* Ienv;  /* embed_item_env_aware.weight  [n_items, D] */
    float* E;     /* embed_env.weight             [K, D] */
    float* W;     /* env_classifier.linear_map.weight [K, D] */
    float* b;     /* env_classifier.linear_map.bias   [K] */
} invpref_params;

/* torch.optim.Adam state (exp_avg, exp_avg_sq) for the same seven tensors (train.py:718). */
typedef struct {
    invpref_params m;
    invpref_params v;
    /* Optional LAZY dense Adam for the user tables (all three NULL/0 = plain dense mode).
     * torch.optim.Adam moves every row every step, also rows without a gradient (momentum).  In lazy mode a
     * user row that is not in the batch is left untouched in memory; user_last_step[r] remembers the step
     * it is updated to, and the skipped zero-gradient steps are replayed in registers -- with each step's
     * own bias corrections from `sched`, same arithmetic, same order, hence bit-identical -- when the row
     * is next touched by a batch, or by invpref_flush_users.  In this mode the user tables are updated IN
     * PLACE (params_out->Uinv/Uenv must alias params_in): the rows every reader of the step needs are
     * stashed in the workspace by the user pass.  Anything outside invpref_train_step that reads the user
     * tables (invpref_cluster, invpref_forward, predict, state_dict) needs invpref_flush_users first. */
    int32_t* user_last_step;   /* [n_users], zero-initialised */
    float* sched;              /* [sched_cap][2]: (lr/bc1, 1/sqrt(bc2)) of every step so far; entry t is
                                  written by the train step with hyper.step == t */
    int64_t sched_cap;
} invpref_adam;

/* One mini-batch = rows [s*B, (s+1)*B) of the training tensors (utils.py:12-19). */
typedef struct {
    const int64_t* users;
    const int64_t* items;
    const int64_t* envs;
    const float* scores;
    const float* weights;   /* sample_weights slice (train.py:956); may be NULL if both re-weights are off */
    int64_t B;
} invpref_batch;

/* The step-DEPENDENT scalars of one train step as a record in DEVICE memory (invpref_hyper.dyn).  Every other scalar
 * of invpref_hyper is baked into the kernel launches; these four change from step to step (Adam's bias corrections,
 * the alpha schedule of train.py:891-894, the step number of the lazy-Adam bookkeeping).  With hyper.dyn set the
 * kernels read them from the record instead, so a CUDA graph captured over the steps of one epoch (invpref_graph_*)
 * can be replayed for every later epoch after the caller has rewritten the records (one small H2D copy per epoch).
 * Fill the host copy with invpref_dyn_fill so that the arithmetic (double, as torch does) lives in one place. */
typedef struct {
    float step_size;      /* lr / (1 - beta1^step) */
    float inv_bc2_sqrt;   /* 1 / sqrt(1 - beta2^step) */
    float neg_alpha;      /* -alpha (functions.py:13-16) */
    int32_t step;         /* 1-based Adam step */
} invpref_dyn;

/* Row-sharded multi-GPU training, PUSH export of the partial item gradients (invpref_hyper.push, with
 * INVPREF_EXPORT_ITEM_GRADS): instead of writing row c of its partial item gradient into grads_out, the item pass
 * stores it straight into the staging buffer of the rank that OWNS the row, over NVLink (posted writes that overlap
 * the rest of the pass): table t (0 invariant, 1 env-aware) of cache row c goes to
 *     base[t * world + owner[c]] + index[c] * dim .
 * The owner then reduces from LOCAL memory (invpref_owner_adam_push).  All pointers are device pointers; `base` is a
 * DEVICE array of 2 * world pointers into the peers' mapped staging buffers. */
typedef struct {
    float* const* base;      /* device array [2 * world] */
    const int32_t* owner;    /* [cache rows] owner rank of every cache row */
    const int32_t* index;    /* [cache rows] row in the owner's staging buffer */
    int32_t world;
    int32_t _pad;
} invpref_push;

/* Loss coefficients (train.py:829-830), gradient-reversal alpha (functions.py:13-16) and
 * Adam settings.  bias corrections are derived from `step` in double, as torch does. */
typedef struct {
    double c_inv, c_ea, c_env, c_L2, c_L1;
    double alpha;
    double lr, beta1, beta2, eps;
    int64_t step;            /* 1-based Adam step of THIS update */
    int32_t use_class_rw;    /* train.py:814-815 */
    int32_t use_rec_rw;      /* train.py:817-819 */
    /* Data-parallel use (one process per GPU, the batch split across ranks): every 1/B factor of the
     * loss means and regularisers uses global_batch (0 = batch->B), so per-rank losses and gradients
     * are partial sums that add up to the single-GPU values. */
    int64_t global_batch;
    int32_t flags;           /* INVPREF_EXPORT_* | INVPREF_SKIP_PARAM_REG */
    int32_t _pad;
    const invpref_dyn* dyn;  /* DEVICE record overriding (lr, betas, step) -> step_size / inv_bc2_sqrt, alpha and step at
                                run time; NULL = use the fields above.  `step` above must still be an upper bound of
                                the steps the record will hold (it sizes the lazy-Adam schedule check). */
    const invpref_push* push; /* HOST pointer; NULL = exported item gradients go to grads_out */
} invpref_hyper;

/* invpref_hyper.flags.  An EXPORT flag makes invpref_train_step write the (partial) gradients of that
 * group of tensors into grads_out INSTEAD of applying Adam to them (rows without a gradient are not
 * written: zero the buffers first), so that the caller can reduce them across ranks and then call
 * invpref_adam_dense.  Tables of an exported group are not double-buffered (params_out may alias). */
#define INVPREF_EXPORT_USER_GRADS 1   /* Uinv, Uenv */
#define INVPREF_EXPORT_ITEM_GRADS 2   /* Iinv, Ienv */
#define INVPREF_EXPORT_SMALL_GRADS 4  /* E, W, b; loss_out then holds this rank's partial sums */
#define INVPREF_SKIP_PARAM_REG 8      /* leave out the classifier's own L1/L2 term (all ranks but one) */
#define INVPREF_DEFER_USER_SWEEP 16   /* skip the dense Adam sweep over user rows without a gradient: the
                                         caller runs invpref_user_sweep itself (e.g. on a second stream, so
                                         that it overlaps the NVLink exchange of the item gradients) */

const char* invpref_strerror(int status);

/* Host helper: the record invpref_hyper.dyn would hold for `hyper` (its lr, betas, step and alpha). */
int invpref_dyn_fill(const invpref_hyper* hyper, invpref_dyn* out_host);

/* ---- CUDA-graph capture of a sequence of library calls (train.py:881-910 runs 3-31 steps per epoch on the dataset
 * configs: launch latency and host overhead, not HBM, bound them) --------------------------------------------------
 * invpref_graph_begin puts `stream` (not the legacy default stream) into capture mode; every library call issued on
 * it until invpref_graph_end is recorded instead of executed.  invpref_graph_end instantiates the graph and returns an
 * opaque handle; invpref_graph_launch replays it on a stream; invpref_graph_destroy frees it.  The captured calls must
 * use invpref_hyper.dyn for whatever changes between replays; all buffers they name must stay alive and in place. */
int invpref_graph_begin(void* stream);
int invpref_graph_end(void* stream, void** out_graph);
int invpref_graph_launch(void* graph, void* stream);
int invpref_graph_destroy(void* graph);
/* Kernel launches recorded in the graph (what one invpref_graph_launch adds to invpref_launch_count). */
int64_t invpref_graph_launches(void* graph);
int invpref_abi_version(void);

/* ---- sizes -------------------------------------------------------------------------- */

/* Bytes of scratch a call on a batch of at most max_batch rows needs (plan building, train
 * step, backward).  The scratch holds nothing across calls. */
int invpref_workspace_bytes(const invpref_desc* desc, int64_t max_batch, size_t* out_bytes);

/* Bytes of one batch plan (both sort orders, see invpref_build_plan). */
int invpref_plan_bytes(const invpref_desc* desc, int64_t max_batch, size_t* out_bytes);

/* 1 if this shape runs the fused user pass (required by lazy Adam: invpref_adam.user_last_step), 0 if the
 * shape only has the unfused path (K * D too large for the per-CTA dE/dW slices), negative = invpref_status.
 * Callers that default to lazy Adam ask first and fall back to plain dense Adam. */
int invpref_upass_supported(const invpref_desc* desc);

/* ---- sort-segment plan ------------------------------------------------------------------
 * Replaces the duplicate handling of embedding_dense_backward (autograd of models.py:449-455):
 * a STABLE sort of the batch by user id and by item id, unique rows and segment offsets, the
 * split of long segments into fixed chunks, a bitmap of touched rows, one 32-byte descriptor per
 * segment (row, bounds, the indices of its first two interactions) and cost-balanced contiguous
 * segment ranges -- what the staged kernels need to request their data one step ahead.  The layout
 * is private to the library (opaque bytes, invpref_plan_bytes).  A plan depends only on (users,
 * items) of the batch, which utils.mini_batch keeps fixed across epochs, so a trainer builds it
 * once per batch and reuses it; it only touches the sort scratch of `ws`, which a train step that
 * is GIVEN a plan never uses, so the next batch's plan may be built on another stream meanwhile. */
int invpref_build_plan(const invpref_desc* desc, const int64_t* users, const int64_t* items, int64_t B,
                       void* plan, size_t plan_bytes, void* ws, size_t ws_bytes, void* stream);

/* Id validation.  The reference raises IndexError (CPU) / a device-side assert (CUDA) on an id outside its
 * table (nn.Embedding, models.py:449-455).  invpref_build_plan clamps such ids so that no kernel reads out of
 * bounds and records the fact in the plan; invpref_plan_status reads that record back: it SYNCHRONISES the
 * stream (the only entry point besides invpref_profile_read that does) and returns INVPREF_ERR_ID_RANGE if any
 * user or item id of the batch was outside its table.  Call it once after building a cached plan. */
int invpref_plan_status(const invpref_desc* desc, const void* plan, int64_t B, void* stream);

/* Asynchronous validation for the entry points that take raw ids without a plan (invpref_forward,
 * invpref_predict, invpref_cluster): ORs into the device word *flag (int32, caller-zeroed) bit 0 if a user id,
 * bit 1 if an item id, bit 2 if an env id of [0, B) is outside [0, n_users) / [0, n_items) / [0, n_envs).
 * Any of the three id pointers may be NULL. */
int invpref_check_ids(const invpref_desc* desc, const int64_t* users, const int64_t* items, const int64_t* envs,
                      int64_t B, int32_t* flag, void* stream);

/* Stand-alone segment builder with int64 outputs, for callers/tests that want the raw result:
 * perm is bit-equal to torch.sort(ids, stable=True).indices; seg_row[0..n_seg) are the unique
 * ids ascending; seg_off[0..n_seg] the offsets into perm.  n_seg is a device int64. */
int invpref_build_segments(const int64_t* ids, int64_t B, int64_t n_rows, int64_t* perm, int64_t* seg_row,
                           int64_t* seg_off, int64_t* n_seg, void* ws, size_t ws_bytes, void* stream);

/* ---- forward ------------------------------------------------------------------------------
 * models.py:448-467 (explicit) / 307-326 (implicit), incl. the classifier models.py:206-209.
 * Any of s_inv / s_env / logp may be NULL.  logp is [B, K]. */
int invpref_forward(const invpref_desc* desc, const invpref_params* params, const int64_t* users,
                    const int64_t* items, const int64_t* envs, int64_t B, float* s_inv, float* s_env,
                    float* logp, void* stream);

/* models.py:534-539: explicit predict = invariant score only (envs not needed). */
int invpref_predict(const invpref_desc* desc, const invpref_params* params, const int64_t* users,
                    const int64_t* items, int64_t B, float* score, void* stream);

/* Autograd backward of invpref_forward (what loss.backward() does through models.py:448-467 and
 * functions.py:13-16): given upstream gradients of s_inv, s_env, logp (any may be NULL) it
 * ACCUMULATES (+=) dense gradients into `grads` (same layout as params).  Deterministic. */
int invpref_backward(const invpref_desc* desc, const invpref_params* params, const invpref_batch* batch,
                     double alpha, const float* g_s_inv, const float* g_s_env, const float* g_logp,
                     const void* plan, invpref_params* grads, void* ws, size_t ws_bytes, void* stream);

/* ---- fused train step -------------------------------------------------------------------------
 * train.py:771-844 in one call: forward, the five loss terms, closed-form backward (SURVEY.md
 * §3.4), dense torch.optim.Adam update of all seven tensors.  The four embedding tables are
 * double-buffered: rows are read from params_in and the updated rows written to params_out
 * (params_out->{Uinv,Iinv,Uenv,Ienv} must not alias params_in; E/W/b may alias and are updated
 * last).  The caller swaps the two sets after the call.  Adam state is updated in place.
 * loss_out: 6 device floats in the order of train.py:836-843.
 * If `grads_out` is non-NULL the dense gradients are ALSO written there (testing aid; moves
 * extra bytes).  plan may be NULL: the step then builds a plan in the workspace first. */
int invpref_train_step(const invpref_desc* desc, const invpref_params* params_in, invpref_params* params_out,
                       invpref_adam* adam, const invpref_batch* batch, const invpref_hyper* hyper,
                       const void* plan, float* loss_out, invpref_params* grads_out, void* ws, size_t ws_bytes,
                       void* stream);

/* ---- EM environment re-assignment ---------------------------------------------------------------
 * train.py:846-879 for a whole slice at once: each sample's loss under all K environments,
 * optional tie-break perturbation eps_table[perm_idx[n]] (train.py:868-873; eps_table is the fp32
 * [K!, K] table of train.py:763-769, perm_idx in [0, K!) the host-drawn np.random.randint, NULL =
 * cluster_use_random_sort off), first-min argmin.
 * new_envs: int64 [B].  hist (int64[K], nullable) and diff (int64, nullable; counts
 * new != old_envs, train.py:933-934) are ACCUMULATED into; zero them first. */
int invpref_cluster(const invpref_desc* desc, const invpref_params* params, const int64_t* users,
                    const int64_t* items, const float* scores, const int64_t* perm_idx, const float* eps_table,
                    const int64_t* old_envs, int64_t B, int64_t* new_envs, int64_t* hist, int64_t* diff,
                    void* stream);

/* The same re-assignment over a USER-SORTED view of the whole dataset (train.py:912-936 walks the dataset once per
 * call; users and items never change, so the view is built once): perm[k] = original position of the k-th sample in
 * stable user order, users_sorted / items_sorted / scores_sorted the sorted copies (int32 ids).  perm_idx, old_envs,
 * new_envs, hist and diff are as for invpref_cluster, in ORIGINAL order.  Results are identical to invpref_cluster;
 * consecutive samples share their user, whose two rows then come out of L2 instead of HBM: at N / U samples per user
 * the DRAM bytes per sample drop from 16 D + 44 towards 8 D + 130. */
int invpref_cluster_sorted(const invpref_desc* desc, const invpref_params* params, const int32_t* perm,
                           const int32_t* users_sorted, const int32_t* items_sorted, const float* scores_sorted,
                           const int64_t* perm_idx, const float* eps_table, const int64_t* old_envs, int64_t N,
                           int64_t* new_envs, int64_t* hist, int64_t* diff, void* stream);

/* train.py:945-957: class_weights[k] = min(cnt_k + 1, N - 1) / N (double -> fp32) from a finished
 * histogram, and sample_weights[n] = class_weights[envs[n]]. */
int invpref_stat_envs(const int64_t* envs, int64_t N, int32_t n_envs, const int64_t* hist, float* class_weights,
                      float* sample_weights, void* stream);

/* Histogram of envs (train.py:949), accumulated into hist (int64[K]). */
int invpref_env_hist(const int64_t* envs, int64_t N, int32_t n_envs, int64_t* hist, void* stream);

/* ---- building blocks of the multi-GPU paths (no reference counterpart: the reference is single-GPU) ----
 * Dense torch.optim.Adam on one flat fp32 tensor with a materialised gradient (after a cross-rank
 * reduction): theta, m, v updated in place.  Uses lr/betas/eps/step of `hyper`. */
int invpref_adam_dense(float* theta, float* m, float* v, const float* grad, int64_t n, const invpref_hyper* hyper,
                       void* stream);

/* Lazy mode (invpref_adam.user_last_step != NULL): bring every user row up to step hyper->step (the last
 * completed train step), in place. */
int invpref_flush_users(const invpref_desc* desc, invpref_params* params, invpref_adam* adam,
                        const invpref_hyper* hyper, void* stream);

/* The deferred part of invpref_train_step (INVPREF_DEFER_USER_SWEEP): dense Adam (zero gradient) on every
 * user row that has no segment in `plan` (built for a batch of B interactions), reading params_in and writing
 * params_out / the Adam state.  Must use the same step / lr / betas / eps as the train step it completes. */
int invpref_user_sweep(const invpref_desc* desc, const invpref_params* params_in, invpref_params* params_out,
                       invpref_adam* adam, const invpref_hyper* hyper, const void* plan, int64_t B, void* stream);

/* out[j, :] = table[rows[j], :] for j < n (row-sharded tables: rows a peer asked for). */
int invpref_gather_rows(const float* table, const int64_t* rows, int64_t n, int32_t dim, float* out, void* stream);

/* table[rows[j], :] += src[j, :] for j < n.  rows must be unique within one call (no atomics); callers
 * apply peers one after the other in rank order, which fixes the summation order. */
int invpref_scatter_add_rows(const float* src, const int64_t* rows, int64_t n, int32_t dim, float* table,
                             void* stream);

/* ---- implicit evaluator helpers (evaluate.py:94-135; per-user item lists as CSR over user ids:
 * off int64 [n_users + 1], items int64 [nnz], ascending and unique within a user) ---------------------
 * invpref_mask_scores: for r < b: rating[r, items(users[r])] = value (add == 0: the train-positive mask,
 * evaluate.py:98) or += value (add != 0: the item-pool highlight, evaluate.py:110).  rating: fp32 [b, n_items]. */
int invpref_mask_scores(float* rating, int64_t b, int64_t n_items, const int64_t* users, const int64_t* off,
                        const int64_t* items, float value, int32_t add, void* stream);

/* invpref_hits_from_csr: hits[r, j] = 1 if top[r, j] is in items(users[r]) else 0 (evaluate.py:11-19 get_label);
 * n_list[r] (nullable) = length of that list (the per-user ground-truth count of recall / IDCG). */
int invpref_hits_from_csr(const int64_t* top, int64_t b, int32_t k, const int64_t* users, const int64_t* off,
                          const int64_t* items, uint8_t* hits, int64_t* n_list, void* stream);

/* invpref_eval_topk: the whole of ImplicitTestManager.evaluate_batch's device work (evaluate.py:88-135) for one
 * batch of b test users in ONE kernel, without materialising the [b, n_items] rating matrix:
 *   rating[r, i] = predict(users[r])[i]   (models.py:393-407: sigmoid(<Uinv[u], Iinv[i]>); explicit model: no sigmoid)
 *   rating[r, mask items of users[r]] = -1024 (evaluate.py:98);  rating[r, pool items] += 1024 (evaluate.py:110)
 *   top_items[r, :] = the k items of largest rating, descending (torch.topk, evaluate.py:113; ties, which torch
 *   leaves unspecified, go to the lower item id);  hits[r, j] = top_items[r, j] in ground truth (evaluate.py:11-19);
 *   n_gt[r] = size of the user's ground-truth list.
 * Lists are CSR over user ids as for invpref_mask_scores (ascending unique items per user); mask / pool / gt may be
 * NULL (no masking / no pool / no hit look-up: hits and n_gt must then be NULL).  1 <= k <= 256, k <= n_items.
 * top_scores (nullable): the adjusted ratings of the selected items. */
int invpref_eval_topk(const invpref_desc* desc, const invpref_params* params, const int64_t* users, int64_t b,
                      const int64_t* mask_off, const int64_t* mask_items, const int64_t* pool_off,
                      const int64_t* pool_items, const int64_t* gt_off, const int64_t* gt_items, int32_t k,
                      int64_t* top_items, float* top_scores, uint8_t* hits, int64_t* n_gt, void* stream);

/* ---- the same exchange over peer memory (NVLink loads; no collective on the data path) -------------
 * `tables` / `grads`: HOST arrays of 2 * world device pointers, [t * world + rank] = base of item table t
 * (0 invariant, 1 env-aware) / of the partial-gradient cache t of rank `rank`, the caller's own rank
 * included; the peers' buffers must be mapped into this process (CUDA IPC / VMM, e.g. torch symmetric
 * memory).  The caller orders producers and consumers across ranks with a barrier.
 *
 * invpref_fetch_rows_p2p: out_t[c, :] = tables[t * world + owner[c]][rows[c], :] for c < n, t = 0, 1
 * (replaces invpref_gather_rows on the owners + an all-to-all of rows). */
int invpref_fetch_rows_p2p(const float* const* tables, int32_t world, const int32_t* owner, const int64_t* rows,
                           int64_t n, int32_t dim, float* out_inv, float* out_env, void* stream);

/* invpref_owner_adam_p2p: for every row j < n_rows of the caller's item shard and t = 0, 1:
 * g = sum over ranks p = 0..world-1 (in this order) of grads[t * world + p][pos[p * n_rows + j], :]
 * (pos < 0: rank p has no partial for row j), then one dense torch.optim.Adam step on theta/m/v with g --
 * the same order and arithmetic as zero-fill + invpref_scatter_add_rows per rank + invpref_adam_dense, in one
 * kernel reading the partials where the ranks' item passes wrote them. */
int invpref_owner_adam_p2p(float* theta_inv, float* theta_env, float* m_inv, float* m_env, float* v_inv, float* v_env,
                           int64_t n_rows, int32_t dim, int32_t world, const float* const* grads, const int32_t* pos,
                           const invpref_hyper* hyper, void* stream);

/* invpref_owner_adam_push: the push counterpart of invpref_owner_adam_p2p, reading LOCAL memory and writing peers.
 * For every row j < n_rows of the caller's item shard and t = 0, 1:
 *   g = sum over ranks p = 0..world-1 (in this order) of stage_t[spos[p * n_rows + j], :]   (spos < 0: no partial)
 *   one dense torch.optim.Adam step on theta/m/v with g  (same order and arithmetic as invpref_owner_adam_p2p), then
 *   for every rank p with npos[p * n_rows + j] >= 0: caches[t * world + p][npos[p * n_rows + j], :] = updated row
 * i.e. the updated row is pushed into the slot it has in rank p's row cache for the NEXT batch (posted NVLink
 * writes; replaces invpref_fetch_rows_p2p).  stage_*: the caller's own staging buffers, filled by the ranks' item
 * passes (invpref_push).  caches: HOST array of 2 * world device pointers; npos / caches may be NULL (last batch). */
int invpref_owner_adam_push(float* theta_inv, float* theta_env, float* m_inv, float* m_env, float* v_inv, float* v_env,
                            int64_t n_rows, int32_t dim, int32_t world, const float* stage_inv, const float* stage_env,
                            const int32_t* spos, float* const* caches, const int32_t* npos,
                            const invpref_hyper* hyper, void* stream);

/* invpref_peer_allreduce: in-place SUM all-reduce of buf[0..n) over the ranks + a rank-wide barrier, over peer memory
 * (two small kernels, no NCCL call: the sharded step of parallel.py needs two such points per step, train.py has no
 * counterpart -- the reference is single-GPU).  peer_slots / peer_flags: HOST arrays of `world` device pointers to
 * every rank's slot array (2 * world * n_max floats) and flag array (world uint32, zero-initialised before the first
 * call on any rank), the caller's own included, mapped into this process.  counter: device uint32 (zero-initialised),
 * private to the rank, advanced by one per call -- every rank must make the same sequence of calls.  The sum runs
 * in rank order on every rank (replicas stay bit-identical).  On return (stream order) everything EVERY rank had
 * enqueued before its call is complete and visible, peer-memory stores included.  n = 0: barrier only.
 * A peer that does not arrive within a few seconds sets bit 0 of *status (device int32) instead of hanging. */
int invpref_peer_allreduce(float* buf, int32_t n, int32_t n_max, int32_t world, int32_t rank, float* const* peer_slots,
                           uint32_t* const* peer_flags, uint32_t* counter, int32_t* status, void* stream);

/* ---- numpy's legacy global stream (np.random.randint, MT19937) continued on the device ----------------------------
 * The reference draws its initial environments (train.py:711) and its tie-break rows (train.py:870-871, one randint per
 * cluster batch; consecutive calls concatenate) from numpy's global RandomState.  These calls produce exactly those
 * draws on the device and the generator state numpy would be left in, so that a caller can hand the state back to
 * numpy (np.random.set_state) and stay on the reference's stream.
 *
 * invpref_mt_jump_bytes: bytes of the jump table (GF(2) matrices of T^(8 * 2^i), T = one twist of the 624-word key,
 * 13 matrices of 49.8 MB) and of the scratch one invpref_mt_randint call needs.  Either pointer may be NULL. */
int invpref_mt_jump_bytes(size_t* jump_bytes, size_t* ws_bytes);

/* Builds the jump table into a caller buffer of at least jump_bytes (once per device; ~15 GF(2) matrix squarings). */
int invpref_mt_build_jumps(void* jumps, size_t jump_bytes, void* stream);

/* out[0..n) = np.random.randint(0, high, n) (int64, ready as perm_idx of invpref_cluster) drawn from the MT19937 state
 * (key_in: the 624 key words on the device, pos_in: numpy's pos, 0..624 -- a fresh np.random.seed leaves 624), and
 * key_out (624 words) / *pos_out (device int32) = the state after the call, as np.random.get_state() would report it.
 * numpy's method for 1 <= high <= 2^32: one tempered word w per attempt, accept w & mask if <= high - 1 (mask =
 * 2^bitlen(high - 1) - 1); high == 1 returns zeros and consumes nothing.  INVPREF_ERR_BAD_ARG for high < 1 or
 * high > 2^32 (numpy's 64-bit path), n < 0 or pos_in outside [0, 624].  key_out must not overlap key_in. */
int invpref_mt_randint(const uint32_t* key_in, int32_t pos_in, int64_t high, int64_t n, int64_t* out,
                       uint32_t* key_out, int32_t* pos_out, const void* jumps, void* ws, size_t ws_bytes, void* stream);

/* Number of kernels the library has launched in this process (bench.py's gpu_launches). */
int64_t invpref_launch_count(void);

/* ---- per-phase device timing (bench.py's roofline) ----------------------------------------------
 * invpref_profile_enable(n > 0): the next n calls of invpref_train_step record CUDA events between
 * their kernels on the call's stream (no synchronisation); n = 0 disables and frees the events.
 * invpref_profile_read(step, out_ms_host): after the caller has synchronised the stream, elapsed
 * milliseconds of each phase of recorded step `step` (0-based), INVPREF_NUM_PHASES floats in the
 * order: plan build, forward (empty on the fused path), user chunks, user rows (fused user pass:
 * forward + user-side reduce + Adam), item chunks, item rows, item sweep, user sweep, tail.  invpref_profile_steps(): number of steps recorded since the last enable. */
#define INVPREF_NUM_PHASES 9
int invpref_profile_enable(int max_steps);
int invpref_profile_steps(void);
int invpref_profile_read(int step, float* out_ms_host);

#ifdef __cplusplus
}
#endif
#endif /* INVPREF_B200_H */
