// Internal launcher interface between api.cu and the kernel translation units.
#pragma once

#include "common.cuh"

namespace invpref {

// ---- fwd.cu ----------------------------------------------------------------------------------
struct FwdTrainArgs {
    const float *Uinv, *Iinv, *Uenv, *Ienv, *E, *W, *b;
    const int64_t *users, *items, *envs;
    const float *scores, *weights;
    int64_t B;
    int D, K, GS;
    int implicit, reg_env_embed, use_class_rw, use_rec_rw;
    float c_inv, c_ea, c_env, neg_alpha, invB;
    float* gpack;      // [B, GS]: g_z1, g_z2, env (int bits), -alpha * g_logits[K]
    float* partials;   // [gridDim.x, P]
    int P;
    // generic autograd backward (invpref_backward): upstream grads instead of the built-in losses
    const float *up_s_inv, *up_s_env, *up_logp;
    int generic;
    const invpref_dyn* dyn;   // optional device record overriding neg_alpha
};

struct FwdOnlyArgs {
    const float *Uinv, *Iinv, *Uenv, *Ienv, *E, *W, *b;
    const int64_t *users, *items, *envs;
    int64_t B;
    int D, K, implicit;
    float *s_inv, *s_env, *logp;
};

int fwd_train_grid(int64_t B);
int launch_fwd_train(const Geometry& g, const FwdTrainArgs& a, int grid, cudaStream_t stream);
int launch_fwd_only(const Geometry& g, const FwdOnlyArgs& a, cudaStream_t stream);
int launch_predict(const Geometry& g, const float* Uinv, const float* Iinv, const int64_t* users, const int64_t* items,
                   int64_t B, float* score, cudaStream_t stream);

// ---- bwd.cu ----------------------------------------------------------------------------------
enum { EPI_ADAM = 0, EPI_ACCUM = 1, EPI_EXPORT = 2 };

// One side (user tables or item tables) of the segmented backward.
struct BwdSideArgs {
    const float *own_inv_in, *own_env_in;     // this side's tables, values BEFORE the step
    float *own_inv_out, *own_env_out;         // where the updated rows go (double buffer)
    float *m_inv, *m_env, *v_inv, *v_env;     // Adam state, updated in place
    const float *partner_inv, *partner_env;   // the other side's tables (BEFORE the step)
    float *grad_inv, *grad_env;               // optional dense gradient output / accumulation target
    PlanSide plan;
    float* chunk_part;                        // [max_chunks, 2, D]
    const float* gpack;
    const float *E, *W;
    int D, K, GS;
    float reg2, reg1;                         // 2*c_L2/(B*D*2), c_L1/(B*D*2)
    AdamScalars adam;
    // lazy user-row Adam (null = dense): see invpref_adam in the header
    int32_t* last_step;                       // [rows of this side] step each row is updated to
    const float2* sched;                      // [step] (lr/bc1, 1/sqrt(bc2))
    int step;                                 // Adam step of this call
    float* stash;                             // user pass: OUT [n_seg, 2, D] caught-up rows before this step;
                                              // item pass: partner rows are read from here via plan.pseg
    const invpref_dyn* dyn;                   // optional device record overriding adam.step_size / inv_bc2_sqrt, step
                                              // (and UserPassArgs.neg_alpha): CUDA-graph replay
    // EPI_EXPORT to peer memory (invpref_push): row r of the partial gradient goes to
    // push_base[t * push_world + push_owner[r]] + push_index[r] * D instead of grad_inv / grad_env
    float* const* push_base;
    const int32_t* push_owner;
    const int32_t* push_index;
    int push_world;
};

int launch_bwd_chunks(const Geometry& g, const BwdSideArgs& a, cudaStream_t stream);
int launch_bwd_rows(const Geometry& g, const BwdSideArgs& a, int epi, cudaStream_t stream);
int launch_sweep(const Geometry& g, const BwdSideArgs& a, cudaStream_t stream);
int launch_flush(const Geometry& g, const BwdSideArgs& a, cudaStream_t stream);     // lazy rows -> step a.step
int launch_sched_write(float2* sched, int step, const AdamScalars& s, const invpref_dyn* dyn, cudaStream_t stream);

// ---- upass.cu: fused forward + user-side backward + Adam ---------------------------------------------
constexpr int UPASS_CHUNK_CTAS = 148;  // CTAs of the long-user-segment kernel (idle on C5, busy on the dataset configs)

struct UserPassArgs {
    BwdSideArgs side;        // own = user tables, partner = item tables, plan = user side
    const float* b;
    const int64_t* envs;
    const float *scores, *weights;
    int implicit, use_class_rw, use_rec_rw;
    float c_inv, c_ea, c_env, neg_alpha, invB;
    float* gpack_out;        // [B, GS], written for the item pass
    float* partials;         // [rows grid + UPASS_CHUNK_CTAS, P]
    int P;
};

bool upass_supported(const Geometry& g);
int upass_rows_grid(const Geometry& g, int64_t max_seg);
int launch_upass_chunks(const Geometry& g, const UserPassArgs& a, int cta_offset, cudaStream_t stream);
int launch_upass_rows(const Geometry& g, const UserPassArgs& a, int epi, int grid, cudaStream_t stream);

struct TailArgs {
    const float* partials;
    int n_partials, P;
    int64_t B;
    int D, K;
    int reg_only_embed, reg_env_embed;
    float c_inv, c_ea, c_env, c_L2, c_L1;
    const float *E_in, *W_in, *b_in;
    float *E_out, *W_out, *b_out;
    float *mE, *mW, *mb, *vE, *vW, *vb;
    float *gE, *gW, *gb;      // optional grads out (EPI_ADAM) / accumulation target (EPI_ACCUM)
    float* loss_out;          // [6]
    AdamScalars adam;
    int epi;
    const invpref_dyn* dyn;
};

int launch_tail(const TailArgs& a, cudaStream_t stream);

// ---- cluster.cu ------------------------------------------------------------------------------
struct ClusterArgs {
    const float *Uinv, *Iinv, *Uenv, *Ienv, *E;
    const int64_t *users, *items;
    const float* scores;
    const int64_t* perm_idx;
    const float* eps_table;
    const int64_t* old_envs;
    int64_t B;
    int D, K, implicit;
    int64_t* new_envs;
    unsigned long long *hist, *diff;
    // user-sorted view (perm != nullptr): sample k of the view is original sample perm[k]; users32 / items32 /
    // scores are the sorted copies, perm_idx / old_envs / new_envs stay in original order
    const int32_t *perm, *users32, *items32;
};

int launch_cluster(const Geometry& g, const ClusterArgs& a, cudaStream_t stream);
int launch_env_hist(const int64_t* envs, int64_t N, int K, unsigned long long* hist, cudaStream_t stream);
int launch_stat_envs(const int64_t* envs, int64_t N, int K, const int64_t* hist, float* class_weights,
                     float* sample_weights, cudaStream_t stream);

// ---- dist.cu ---------------------------------------------------------------------------------
int launch_adam_dense(float* theta, float* m, float* v, const float* grad, int64_t n, const AdamScalars& s,
                      const invpref_dyn* dyn, cudaStream_t stream);
int launch_gather_rows(const float* table, const int64_t* rows, int64_t n, int dim, float* out, cudaStream_t stream);
int launch_scatter_add_rows(const float* src, const int64_t* rows, int64_t n, int dim, float* table,
                            cudaStream_t stream);

// peer-memory variants (pointer arrays are HOST arrays of 2 * world device pointers: [t * world + rank])
int launch_fetch_rows_p2p(const float* const* tables_host, int world, const int32_t* owner, const int64_t* rows,
                          int64_t n, int dim, float* out0, float* out1, cudaStream_t stream);
int launch_owner_adam_push(float* th0, float* th1, float* m0, float* m1, float* v0, float* v1, int64_t n_rows, int dim,
                           int world, const float* stage0, const float* stage1, const int32_t* spos,
                           float* const* caches_host, const int32_t* npos, const AdamScalars& s,
                           const invpref_dyn* dyn, cudaStream_t stream);

int launch_peer_allreduce(float* buf, int n, int n_max, int world, int rank, float* const* slots_host,
                          uint32_t* const* flags_host, uint32_t* ctr, int32_t* status, cudaStream_t stream);

// ---- eval.cu ---------------------------------------------------------------------------------
int launch_mask_scores(float* rating, int64_t b, int64_t n_items, const int64_t* users, const int64_t* off,
                       const int64_t* items, float value, int add, cudaStream_t stream);
int launch_hits_from_csr(const int64_t* top, int64_t b, int k, const int64_t* users, const int64_t* off,
                         const int64_t* items, uint8_t* hits, int64_t* n_list, cudaStream_t stream);
// the evaluator (eval.cu): one CTA per user below 2048 items, else launch_topk_stream in EVAL mode
int launch_eval_topk(const float* Uinv, const float* Iinv, int64_t n_items, int D, int implicit, const int64_t* users,
                     int64_t b, const int64_t* mask_off, const int64_t* mask_items, const int64_t* pool_off,
                     const int64_t* pool_items, const int64_t* gt_off, const int64_t* gt_items, int k,
                     int64_t* top_items, float* top_scores, uint8_t* hits, int64_t* n_gt, cudaStream_t stream);
// streaming top-k (eval.cu) of the b query rows Q[qids[r]] over the n_rows rows of the catalogue table X: score =
// <query row, catalogue row> (sigmoid of it if implicit); lists are CSR over query ids.
// exclude == 0 -> list 0 = mask (-1024), list 1 = pool (+1024), hits / n_gt from gt;
// exclude == 1 -> list 0 = catalogue rows that are never candidates, no list 1, trailing slots (item -1, score -inf).
// inv_norm != NULL -> cosine (Q == X, qids index X, inv_norm [n_rows] from launch_row_inv_norm), no sigmoid, catalogue
// row qids[r] never a candidate of query r; pass exclude == 1 and no lists.
int launch_topk_stream(const float* Q, const int64_t* qids, int64_t b, const float* X, int64_t n_rows, int D,
                       int implicit, const float* inv_norm, const int64_t* list0_off, const int64_t* list0_items,
                       const int64_t* list1_off, const int64_t* list1_items, int exclude, const int64_t* gt_off,
                       const int64_t* gt_items, int k, int64_t* top_items, float* top_scores, uint8_t* hits,
                       int64_t* n_gt, cudaStream_t stream);
// inv_norm[i] = 1 / sqrtf(sum_d x[i, d]^2) for the n rows of x [n, D] (row_inv_norm_kernel: order and edge cases)
int launch_row_inv_norm(const float* x, int64_t n, int D, float* inv_norm, cudaStream_t stream);

// ---- foldin.cu -------------------------------------------------------------------------------
// fold-in of the b histories (off [b + 1], ids, scores) against the catalogue table V [n_cat, D]: fp32 rows out [b, D]
// and Newton step counts iters [b] (nullable); the definition is invpref_fold_in_users' in the header
int fold_in_max_dim();
int launch_fold_in(const float* V, int64_t n_cat, int D, int implicit, const int64_t* off, const int64_t* ids,
                   const float* scores, int64_t b, double l2, int max_iter, float* out, int32_t* iters,
                   cudaStream_t stream);

// ---- plan.cu ---------------------------------------------------------------------------------
int build_plan_side(const int64_t* ids, const int64_t* other_ids, int64_t other_rows, const int32_t* other_seg_of,
                    PlanSide p, char* tmp, size_t tmp_bytes, cudaStream_t stream);
int launch_check_ids(const int64_t* users, const int64_t* items, const int64_t* envs, int64_t B, int64_t n_users,
                     int64_t n_items, int64_t n_envs, int32_t* flag, cudaStream_t stream);
int build_segments_i64(const int64_t* ids, int64_t B, int64_t rows, int64_t* perm, int64_t* seg_row, int64_t* seg_off,
                       int64_t* n_seg, char* ws, size_t ws_bytes, cudaStream_t stream);

}  // namespace invpref
