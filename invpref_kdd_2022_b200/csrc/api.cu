// extern "C" entry points of libinvpref_b200.so (see include/invpref_b200.h).
#include <math.h>

#include "common.cuh"
#include "kernels.h"

#include <vector>

namespace invpref {
long long g_launch_count = 0;

namespace {

// per-phase CUDA events of the profiled train steps (invpref_profile_*)
constexpr int NEV = INVPREF_NUM_PHASES + 1;
std::vector<cudaEvent_t> g_prof_events;
int g_prof_max = 0, g_prof_n = 0;

struct PhaseMark {
    cudaEvent_t* ev;
    cudaStream_t st;
    int idx;
    PhaseMark(cudaStream_t s) : ev(nullptr), st(s), idx(0) {
        if (g_prof_n < g_prof_max) ev = &g_prof_events[(size_t)g_prof_n * NEV];
    }
    void mark() {
        if (ev && idx < NEV) cudaEventRecord(ev[idx++], st);
    }
    void done() {
        if (ev) ++g_prof_n;
    }
};

inline bool aligned_for(const void* p, int vec) { return ((uintptr_t)p % (size_t)(vec * 4)) == 0; }

int check_tables(const Geometry& g, const invpref_params* p) {
    if (!p || !p->Uinv || !p->Iinv || !p->Uenv || !p->Ienv || !p->E || !p->W || !p->b) return INVPREF_ERR_BAD_ARG;
    if (!aligned_for(p->Uinv, g.VEC) || !aligned_for(p->Iinv, g.VEC) || !aligned_for(p->Uenv, g.VEC) ||
        !aligned_for(p->Ienv, g.VEC))
        return INVPREF_ERR_MISALIGNED;
    return INVPREF_OK;
}

AdamScalars make_adam(const invpref_hyper* h) {
    // torch/optim/adam.py (_single_tensor_adam): python-float bias corrections from the int step
    AdamScalars s;
    const double bc1 = 1.0 - pow(h->beta1, (double)h->step);
    const double bc2 = 1.0 - pow(h->beta2, (double)h->step);
    s.one_minus_b1 = (float)(1.0 - h->beta1);
    s.b2 = (float)h->beta2;
    s.one_minus_b2 = (float)(1.0 - h->beta2);
    s.step_size = (float)(h->lr / bc1);
    s.bc2_sqrt = (float)sqrt(bc2);
    s.inv_bc2_sqrt = (float)(1.0 / sqrt(bc2));
    s.eps = (float)h->eps;
    return s;
}

void carve_plan(const invpref_desc* d, int64_t B, char* plan, PlanSide* pu, PlanSide* pi) {
    int64_t Bp = B > 0 ? B : 1;
    *pu = carve_plan_side(plan, Bp, d->n_users);
    *pi = carve_plan_side(plan + plan_side_bytes(Bp, d->n_users), Bp, d->n_items);
    pu->B = B;
    pi->B = B;
}

int build_plan_impl(const invpref_desc* d, const int64_t* users, const int64_t* items, int64_t B, char* plan,
                    char* tmp, size_t tmp_bytes, cudaStream_t st) {
    PlanSide pu, pi;
    carve_plan(d, B, plan, &pu, &pi);
    // user side first; the item side then also records, per sorted interaction, the USER segment of its partner row
    // (pseg: where the item pass finds that row in the stash) -- the user side's pseg has no reader and stays unwritten
    int rc = build_plan_side(users, items, d->n_items, nullptr, pu, tmp, tmp_bytes, st);
    if (rc != INVPREF_OK) return rc;
    return build_plan_side(items, users, d->n_users, pu.seg_of, pi, tmp, tmp_bytes, st);
}

}  // namespace
}  // namespace invpref

using namespace invpref;

extern "C" {

const char* invpref_strerror(int status) {
    switch (status) {
        case INVPREF_OK: return "ok";
        case INVPREF_ERR_BAD_DIM: return "unsupported embedding dimension";
        case INVPREF_ERR_BAD_ENVS: return "unsupported number of environments";
        case INVPREF_ERR_BAD_ARG: return "bad argument (null pointer, negative size or table too large)";
        case INVPREF_ERR_MISALIGNED: return "table pointer not aligned for the vector width of this dimension";
        case INVPREF_ERR_WORKSPACE: return "workspace or plan buffer too small";
        case INVPREF_ERR_CUDA: return "CUDA error at kernel launch";
        case INVPREF_ERR_ID_RANGE: return "id outside its table";
        default: return "unknown status";
    }
}

int invpref_abi_version(void) { return INVPREF_ABI_VERSION; }

int64_t invpref_launch_count(void) { return (int64_t)g_launch_count; }

int invpref_dyn_fill(const invpref_hyper* hyper, invpref_dyn* out_host) {
    if (!hyper || !out_host || hyper->step < 1) return INVPREF_ERR_BAD_ARG;
    const AdamScalars s = make_adam(hyper);
    out_host->step_size = s.step_size;
    out_host->inv_bc2_sqrt = s.inv_bc2_sqrt;
    out_host->neg_alpha = (float)(-hyper->alpha);
    out_host->step = (int32_t)hyper->step;
    return INVPREF_OK;
}

// ---- CUDA-graph capture / replay of a sequence of library calls ----
struct GraphHandle {
    cudaGraphExec_t exec;
    long long launches;
};
static long long g_capture_launch0 = -1;

int invpref_graph_begin(void* stream) {
    if (stream == nullptr || g_capture_launch0 >= 0) return INVPREF_ERR_BAD_ARG;   // not the legacy stream; not nested
    if (cudaStreamBeginCapture((cudaStream_t)stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) {
        cudaGetLastError();
        return INVPREF_ERR_CUDA;
    }
    g_capture_launch0 = g_launch_count;
    return INVPREF_OK;
}

int invpref_graph_end(void* stream, void** out_graph) {
    if (g_capture_launch0 < 0 || !out_graph) return INVPREF_ERR_BAD_ARG;
    const long long n = g_launch_count - g_capture_launch0;
    g_launch_count = g_capture_launch0;       // recorded, not executed: they count when the graph is launched
    g_capture_launch0 = -1;
    cudaGraph_t graph = nullptr;
    if (cudaStreamEndCapture((cudaStream_t)stream, &graph) != cudaSuccess || graph == nullptr) {
        cudaGetLastError();
        return INVPREF_ERR_CUDA;
    }
    cudaGraphExec_t exec = nullptr;
    const cudaError_t rc = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (rc != cudaSuccess) {
        cudaGetLastError();
        return INVPREF_ERR_CUDA;
    }
    *out_graph = new GraphHandle{exec, n};
    return INVPREF_OK;
}

int invpref_graph_launch(void* graph, void* stream) {
    if (!graph) return INVPREF_ERR_BAD_ARG;
    GraphHandle* h = (GraphHandle*)graph;
    if (cudaGraphLaunch(h->exec, (cudaStream_t)stream) != cudaSuccess) {
        cudaGetLastError();
        return INVPREF_ERR_CUDA;
    }
    g_launch_count += h->launches;
    return INVPREF_OK;
}

int invpref_graph_destroy(void* graph) {
    if (!graph) return INVPREF_OK;
    GraphHandle* h = (GraphHandle*)graph;
    cudaGraphExecDestroy(h->exec);
    delete h;
    return INVPREF_OK;
}

int64_t invpref_graph_launches(void* graph) { return graph ? (int64_t)((GraphHandle*)graph)->launches : 0; }

int invpref_profile_enable(int max_steps) {
    for (cudaEvent_t e : g_prof_events) cudaEventDestroy(e);
    g_prof_events.clear();
    g_prof_max = 0;
    g_prof_n = 0;
    if (max_steps <= 0) return INVPREF_OK;
    if (max_steps > 4096) return INVPREF_ERR_BAD_ARG;
    g_prof_events.resize((size_t)max_steps * NEV);
    for (auto& e : g_prof_events)
        if (cudaEventCreate(&e) != cudaSuccess) return INVPREF_ERR_CUDA;
    g_prof_max = max_steps;
    return INVPREF_OK;
}

int invpref_profile_steps(void) { return g_prof_n; }

int invpref_profile_read(int step, float* out_ms_host) {
    if (step < 0 || step >= g_prof_n || !out_ms_host) return INVPREF_ERR_BAD_ARG;
    cudaEvent_t* ev = &g_prof_events[(size_t)step * NEV];
    for (int i = 0; i < INVPREF_NUM_PHASES; ++i)
        if (cudaEventElapsedTime(&out_ms_host[i], ev[i], ev[i + 1]) != cudaSuccess) return INVPREF_ERR_CUDA;
    return INVPREF_OK;
}

int invpref_workspace_bytes(const invpref_desc* desc, int64_t max_batch, size_t* out_bytes) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if (max_batch < 0 || max_batch > 0x7fffffffLL || !out_bytes) return INVPREF_ERR_BAD_ARG;
    *out_bytes = workspace_bytes_impl(desc, g, max_batch, nullptr, nullptr);
    return INVPREF_OK;
}

int invpref_plan_bytes(const invpref_desc* desc, int64_t max_batch, size_t* out_bytes) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if (max_batch < 0 || max_batch > 0x7fffffffLL || !out_bytes) return INVPREF_ERR_BAD_ARG;
    int64_t Bp = max_batch > 0 ? max_batch : 1;
    *out_bytes = plan_side_bytes(Bp, desc->n_users) + plan_side_bytes(Bp, desc->n_items);
    return INVPREF_OK;
}

int invpref_build_plan(const invpref_desc* desc, const int64_t* users, const int64_t* items, int64_t B, void* plan,
                       size_t plan_bytes, void* ws, size_t ws_bytes, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if (B < 0 || B > 0x7fffffffLL || !plan || !ws || (B > 0 && (!users || !items))) return INVPREF_ERR_BAD_ARG;
    size_t need = 0;
    invpref_plan_bytes(desc, B, &need);
    if (plan_bytes < need) return INVPREF_ERR_WORKSPACE;
    Workspace w;
    if (ws_bytes < workspace_bytes_impl(desc, g, B, &w, (char*)ws)) return INVPREF_ERR_WORKSPACE;
    return build_plan_impl(desc, users, items, B, (char*)plan, w.sort_tmp, w.sort_tmp_bytes, (cudaStream_t)stream);
}

int invpref_upass_supported(const invpref_desc* desc) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    return upass_supported(g) ? 1 : 0;
}

int invpref_plan_status(const invpref_desc* desc, const void* plan, int64_t B, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if (!plan || B < 0 || B > 0x7fffffffLL) return INVPREF_ERR_BAD_ARG;
    PlanSide pu, pi;
    carve_plan(desc, B, (char*)plan, &pu, &pi);
    int32_t cu[4] = {0, 0, 0, 0}, ci[4] = {0, 0, 0, 0};
    cudaStream_t st = (cudaStream_t)stream;
    if (cudaMemcpyAsync(cu, pu.counters, sizeof(cu), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaMemcpyAsync(ci, pi.counters, sizeof(ci), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess)
        return INVPREF_ERR_CUDA;
    return (cu[2] || ci[2]) ? INVPREF_ERR_ID_RANGE : INVPREF_OK;
}

int invpref_check_ids(const invpref_desc* desc, const int64_t* users, const int64_t* items, const int64_t* envs,
                      int64_t B, int32_t* flag, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if (B < 0 || !flag) return INVPREF_ERR_BAD_ARG;
    if (B == 0 || (!users && !items && !envs)) return INVPREF_OK;
    return launch_check_ids(users, items, envs, B, desc->n_users, desc->n_items, desc->n_envs, flag,
                            (cudaStream_t)stream);
}

int invpref_build_segments(const int64_t* ids, int64_t B, int64_t n_rows, int64_t* perm, int64_t* seg_row,
                           int64_t* seg_off, int64_t* n_seg, void* ws, size_t ws_bytes, void* stream) {
    if (B < 0 || B > 0x7fffffffLL || n_rows < 1 || n_rows > 0x7fffffffLL || !ws || !seg_off || !n_seg ||
        (B > 0 && (!ids || !perm || !seg_row)))
        return INVPREF_ERR_BAD_ARG;
    return build_segments_i64(ids, B, n_rows, perm, seg_row, seg_off, n_seg, (char*)ws, ws_bytes, (cudaStream_t)stream);
}

int invpref_forward(const invpref_desc* desc, const invpref_params* params, const int64_t* users, const int64_t* items,
                    const int64_t* envs, int64_t B, float* s_inv, float* s_env, float* logp, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if ((rc = check_tables(g, params)) != INVPREF_OK) return rc;
    if (B < 0 || (B > 0 && (!users || !items || !envs))) return INVPREF_ERR_BAD_ARG;
    if (B == 0) return INVPREF_OK;
    FwdOnlyArgs a;
    a.Uinv = params->Uinv; a.Iinv = params->Iinv; a.Uenv = params->Uenv; a.Ienv = params->Ienv;
    a.E = params->E; a.W = params->W; a.b = params->b;
    a.users = users; a.items = items; a.envs = envs; a.B = B;
    a.D = g.D; a.K = g.K; a.implicit = desc->implicit;
    a.s_inv = s_inv; a.s_env = s_env; a.logp = logp;
    return launch_fwd_only(g, a, (cudaStream_t)stream);
}

int invpref_predict(const invpref_desc* desc, const invpref_params* params, const int64_t* users, const int64_t* items,
                    int64_t B, float* score, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if ((rc = check_tables(g, params)) != INVPREF_OK) return rc;
    if (B < 0 || (B > 0 && (!users || !items || !score))) return INVPREF_ERR_BAD_ARG;
    if (B == 0) return INVPREF_OK;
    return launch_predict(g, params->Uinv, params->Iinv, users, items, B, score, (cudaStream_t)stream);
}

static void fill_side(BwdSideArgs* s, const Geometry& g, const float* gpack, const float* E, const float* W) {
    s->gpack = gpack; s->E = E; s->W = W; s->D = g.D; s->K = g.K; s->GS = g.GS;
}

int invpref_train_step(const invpref_desc* desc, const invpref_params* pin, invpref_params* pout, invpref_adam* adam,
                       const invpref_batch* batch, const invpref_hyper* hyper, const void* plan, float* loss_out,
                       invpref_params* grads_out, void* ws, size_t ws_bytes, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if ((rc = check_tables(g, pin)) != INVPREF_OK) return rc;
    if ((rc = check_tables(g, pout)) != INVPREF_OK) return rc;
    if (!adam || !batch || !hyper || !ws) return INVPREF_ERR_BAD_ARG;
    if ((rc = check_tables(g, &adam->m)) != INVPREF_OK) return rc;
    if ((rc = check_tables(g, &adam->v)) != INVPREF_OK) return rc;
    if (grads_out && (rc = check_tables(g, grads_out)) != INVPREF_OK) return rc;
    const int64_t B = batch->B;
    if (B < 1 || B > 0x7fffffffLL || !batch->users || !batch->items || !batch->envs || !batch->scores)
        return INVPREF_ERR_BAD_ARG;
    if ((hyper->use_class_rw || hyper->use_rec_rw) && !batch->weights) return INVPREF_ERR_BAD_ARG;
    const bool exp_u = hyper->flags & INVPREF_EXPORT_USER_GRADS, exp_i = hyper->flags & INVPREF_EXPORT_ITEM_GRADS;
    const bool exp_s = hyper->flags & INVPREF_EXPORT_SMALL_GRADS;
    if ((exp_u || exp_i || exp_s) && !grads_out) return INVPREF_ERR_BAD_ARG;
    const invpref_push* push = hyper->push;
    if (push && (!exp_i || !push->base || !push->owner || !push->index || push->world < 1 || push->world > 16))
        return INVPREF_ERR_BAD_ARG;
    const bool lazy = adam->user_last_step != nullptr;
    if (lazy) {
        // lazy user rows: fused pass only, in place, Adam (not export), schedule table with room for this step
        if (exp_u || !adam->sched || hyper->step >= adam->sched_cap || !upass_supported(g) ||
            pin->Uinv != pout->Uinv || pin->Uenv != pout->Uenv || (hyper->flags & INVPREF_DEFER_USER_SWEEP))
            return INVPREF_ERR_BAD_ARG;
    }
    if ((!exp_u && !lazy && (pin->Uinv == pout->Uinv || pin->Uenv == pout->Uenv)) ||
        (!exp_i && (pin->Iinv == pout->Iinv || pin->Ienv == pout->Ienv)))
        return INVPREF_ERR_BAD_ARG;   // tables that Adam updates in this call are double-buffered
    if (hyper->step < 1 || hyper->global_batch < 0) return INVPREF_ERR_BAD_ARG;
    // grads_out: with EXPORT flags only the exported groups are written; without any, all (testing aid)
    const bool any_exp = exp_u || exp_i || exp_s;
    const bool wr_u = grads_out && (exp_u || !any_exp), wr_i = grads_out && (exp_i || !any_exp);
    const bool wr_s = grads_out && (exp_s || !any_exp);
    const int64_t Bg = hyper->global_batch > 0 ? hyper->global_batch : B;   // every 1/B factor uses this
    Workspace w;
    if (ws_bytes < workspace_bytes_impl(desc, g, B, &w, (char*)ws)) return INVPREF_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    PhaseMark pm(st);
    pm.mark();

    const char* plan_base = (const char*)plan;
    if (plan_base == nullptr) {
        rc = build_plan_impl(desc, batch->users, batch->items, B, w.plan, w.sort_tmp, w.sort_tmp_bytes, st);
        if (rc != INVPREF_OK) return rc;
        plan_base = w.plan;
    }
    PlanSide pu, pi;
    carve_plan(desc, B, (char*)plan_base, &pu, &pi);
    pm.mark();

    // (3)+(4) arguments of the segmented backward feeding Adam (or exporting partial gradients), per side
    const AdamScalars as = make_adam(hyper);
    const double bd2 = (double)Bg * g.D * 2.0;
    BwdSideArgs su, si;
    fill_side(&su, g, w.gpack, pin->E, pin->W);
    su.own_inv_in = pin->Uinv; su.own_env_in = pin->Uenv; su.own_inv_out = pout->Uinv; su.own_env_out = pout->Uenv;
    su.m_inv = adam->m.Uinv; su.m_env = adam->m.Uenv; su.v_inv = adam->v.Uinv; su.v_env = adam->v.Uenv;
    su.partner_inv = pin->Iinv; su.partner_env = pin->Ienv;
    su.grad_inv = wr_u ? grads_out->Uinv : nullptr; su.grad_env = wr_u ? grads_out->Uenv : nullptr;
    su.plan = pu; su.chunk_part = w.chunk_part_u;
    su.reg2 = (float)(2.0 * hyper->c_L2 / bd2); su.reg1 = (float)(hyper->c_L1 / bd2); su.adam = as;
    fill_side(&si, g, w.gpack, pin->E, pin->W);
    si.own_inv_in = pin->Iinv; si.own_env_in = pin->Ienv; si.own_inv_out = pout->Iinv; si.own_env_out = pout->Ienv;
    si.m_inv = adam->m.Iinv; si.m_env = adam->m.Ienv; si.v_inv = adam->v.Iinv; si.v_env = adam->v.Ienv;
    si.partner_inv = pin->Uinv; si.partner_env = pin->Uenv;
    si.grad_inv = wr_i ? grads_out->Iinv : nullptr; si.grad_env = wr_i ? grads_out->Ienv : nullptr;
    si.plan = pi; si.chunk_part = w.chunk_part_i;
    si.reg2 = su.reg2; si.reg1 = su.reg1; si.adam = as;
    su.last_step = nullptr; su.sched = nullptr; su.step = (int)hyper->step; su.stash = nullptr; su.dyn = hyper->dyn;
    si.last_step = nullptr; si.sched = nullptr; si.step = (int)hyper->step; si.stash = nullptr; si.dyn = hyper->dyn;
    su.push_base = nullptr; su.push_owner = nullptr; su.push_index = nullptr; su.push_world = 0;
    si.push_base = push ? push->base : nullptr; si.push_owner = push ? push->owner : nullptr;
    si.push_index = push ? push->index : nullptr; si.push_world = push ? push->world : 0;
    if (lazy) {
        su.last_step = adam->user_last_step; su.sched = (const float2*)adam->sched; su.stash = w.stash;
        si.stash = w.stash;     // the item pass reads the user rows of this step from the stash
        if ((rc = launch_sched_write((float2*)adam->sched, (int)hyper->step, as, hyper->dyn, st)) != INVPREF_OK) return rc;
    }

    const int P = fwd_partial_floats(g);
    int n_partials;
    if (upass_supported(g)) {
        // (1)+(2)+(3u)+(4u) fused USER PASS: forward, losses, user-side segment reduce, Adam on user rows
        UserPassArgs up;
        up.side = su;
        up.b = pin->b; up.envs = batch->envs; up.scores = batch->scores; up.weights = batch->weights;
        up.implicit = desc->implicit; up.use_class_rw = hyper->use_class_rw; up.use_rec_rw = hyper->use_rec_rw;
        up.c_inv = (float)hyper->c_inv; up.c_ea = (float)hyper->c_ea; up.c_env = (float)hyper->c_env;
        up.neg_alpha = (float)(-hyper->alpha); up.invB = 1.f / (float)Bg;
        up.gpack_out = w.gpack; up.partials = w.partials; up.P = P;
        const int ugrid = upass_rows_grid(g, pu.max_seg);
        n_partials = ugrid + UPASS_CHUNK_CTAS;
        pm.mark();   // "forward" phase is empty on this path
        if ((rc = launch_upass_chunks(g, up, ugrid, st)) != INVPREF_OK) return rc;
        pm.mark();
        if ((rc = launch_upass_rows(g, up, exp_u ? EPI_EXPORT : EPI_ADAM, ugrid, st)) != INVPREF_OK) return rc;
        pm.mark();
    } else {
        // (1)+(2) forward, losses, per-interaction gradients, dW/db/dE partials; then the user side
        FwdTrainArgs f;
        f.Uinv = pin->Uinv; f.Iinv = pin->Iinv; f.Uenv = pin->Uenv; f.Ienv = pin->Ienv;
        f.E = pin->E; f.W = pin->W; f.b = pin->b;
        f.users = batch->users; f.items = batch->items; f.envs = batch->envs;
        f.scores = batch->scores; f.weights = batch->weights; f.B = B;
        f.D = g.D; f.K = g.K; f.GS = g.GS;
        f.implicit = desc->implicit; f.reg_env_embed = desc->reg_env_embed;
        f.use_class_rw = hyper->use_class_rw; f.use_rec_rw = hyper->use_rec_rw;
        f.c_inv = (float)hyper->c_inv; f.c_ea = (float)hyper->c_ea; f.c_env = (float)hyper->c_env;
        f.neg_alpha = (float)(-hyper->alpha); f.invB = 1.f / (float)Bg;
        f.gpack = w.gpack; f.partials = w.partials; f.P = P;
        f.up_s_inv = f.up_s_env = f.up_logp = nullptr; f.generic = 0; f.dyn = hyper->dyn;
        n_partials = fwd_train_grid(B);
        if ((rc = launch_fwd_train(g, f, n_partials, st)) != INVPREF_OK) return rc;
        pm.mark();
        if ((rc = launch_bwd_chunks(g, su, st)) != INVPREF_OK) return rc;
        pm.mark();
        if ((rc = launch_bwd_rows(g, su, exp_u ? EPI_EXPORT : EPI_ADAM, st)) != INVPREF_OK) return rc;
        pm.mark();
    }
    // item pass: reads the g-pack and the OLD user rows
    if ((rc = launch_bwd_chunks(g, si, st)) != INVPREF_OK) return rc;
    pm.mark();
    if ((rc = launch_bwd_rows(g, si, exp_i ? EPI_EXPORT : EPI_ADAM, st)) != INVPREF_OK) return rc;
    pm.mark();
    if (!exp_i && (rc = launch_sweep(g, si, st)) != INVPREF_OK) return rc;
    pm.mark();
    if (!exp_u && !lazy && !(hyper->flags & INVPREF_DEFER_USER_SWEEP) && (rc = launch_sweep(g, su, st)) != INVPREF_OK)
        return rc;
    pm.mark();

    // losses, E / W / b gradients and their Adam update (or export)
    TailArgs t;
    t.partials = w.partials; t.n_partials = n_partials; t.P = P; t.B = Bg; t.D = g.D; t.K = g.K;
    t.reg_only_embed = desc->reg_only_embed || (hyper->flags & INVPREF_SKIP_PARAM_REG);
    t.reg_env_embed = desc->reg_env_embed;
    t.c_inv = (float)hyper->c_inv; t.c_ea = (float)hyper->c_ea; t.c_env = (float)hyper->c_env;
    t.c_L2 = (float)hyper->c_L2; t.c_L1 = (float)hyper->c_L1;
    t.E_in = pin->E; t.W_in = pin->W; t.b_in = pin->b;
    t.E_out = pout->E; t.W_out = pout->W; t.b_out = pout->b;
    t.mE = adam->m.E; t.mW = adam->m.W; t.mb = adam->m.b; t.vE = adam->v.E; t.vW = adam->v.W; t.vb = adam->v.b;
    t.gE = wr_s ? grads_out->E : nullptr; t.gW = wr_s ? grads_out->W : nullptr;
    t.gb = wr_s ? grads_out->b : nullptr;
    t.loss_out = loss_out; t.adam = as; t.epi = exp_s ? EPI_EXPORT : EPI_ADAM; t.dyn = hyper->dyn;
    rc = launch_tail(t, st);
    pm.mark();
    pm.done();
    return rc;
}

int invpref_flush_users(const invpref_desc* desc, invpref_params* params, invpref_adam* adam,
                        const invpref_hyper* hyper, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if ((rc = check_tables(g, params)) != INVPREF_OK) return rc;
    if (!adam || !hyper || !adam->user_last_step || !adam->sched || hyper->step < 0 || hyper->step >= adam->sched_cap)
        return INVPREF_ERR_BAD_ARG;
    if (hyper->step == 0) return INVPREF_OK;
    BwdSideArgs su = {};
    su.own_inv_in = params->Uinv; su.own_env_in = params->Uenv;
    su.own_inv_out = params->Uinv; su.own_env_out = params->Uenv;
    su.m_inv = adam->m.Uinv; su.m_env = adam->m.Uenv; su.v_inv = adam->v.Uinv; su.v_env = adam->v.Uenv;
    su.plan.rows = desc->n_users; su.D = g.D; su.K = g.K; su.GS = g.GS;
    invpref_hyper h1 = *hyper;
    if (h1.step < 1) h1.step = 1;
    su.adam = make_adam(&h1);
    su.last_step = adam->user_last_step; su.sched = (const float2*)adam->sched; su.step = (int)hyper->step;
    su.dyn = hyper->dyn;
    return launch_flush(g, su, (cudaStream_t)stream);
}

int invpref_user_sweep(const invpref_desc* desc, const invpref_params* pin, invpref_params* pout, invpref_adam* adam,
                       const invpref_hyper* hyper, const void* plan, int64_t B, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if ((rc = check_tables(g, pin)) != INVPREF_OK) return rc;
    if ((rc = check_tables(g, pout)) != INVPREF_OK) return rc;
    if (!adam || !hyper || !plan || B < 0 || hyper->step < 1) return INVPREF_ERR_BAD_ARG;
    if (pin->Uinv == pout->Uinv || pin->Uenv == pout->Uenv) return INVPREF_ERR_BAD_ARG;
    PlanSide pu, pi;
    carve_plan(desc, B, (char*)plan, &pu, &pi);
    BwdSideArgs su = {};
    su.own_inv_in = pin->Uinv; su.own_env_in = pin->Uenv; su.own_inv_out = pout->Uinv; su.own_env_out = pout->Uenv;
    su.m_inv = adam->m.Uinv; su.m_env = adam->m.Uenv; su.v_inv = adam->v.Uinv; su.v_env = adam->v.Uenv;
    su.plan = pu; su.D = g.D; su.K = g.K; su.GS = g.GS; su.adam = make_adam(hyper); su.dyn = hyper->dyn;
    return launch_sweep(g, su, (cudaStream_t)stream);
}

int invpref_adam_dense(float* theta, float* m, float* v, const float* grad, int64_t n, const invpref_hyper* hyper,
                       void* stream) {
    if (!theta || !m || !v || !grad || !hyper || n < 0 || hyper->step < 1) return INVPREF_ERR_BAD_ARG;
    if (n == 0) return INVPREF_OK;
    return launch_adam_dense(theta, m, v, grad, n, make_adam(hyper), hyper->dyn, (cudaStream_t)stream);
}

int invpref_gather_rows(const float* table, const int64_t* rows, int64_t n, int32_t dim, float* out, void* stream) {
    if (n < 0 || dim < 1 || (n > 0 && (!table || !rows || !out))) return INVPREF_ERR_BAD_ARG;
    if (n == 0) return INVPREF_OK;
    return launch_gather_rows(table, rows, n, dim, out, (cudaStream_t)stream);
}

int invpref_scatter_add_rows(const float* src, const int64_t* rows, int64_t n, int32_t dim, float* table,
                             void* stream) {
    if (n < 0 || dim < 1 || (n > 0 && (!table || !rows || !src))) return INVPREF_ERR_BAD_ARG;
    if (n == 0) return INVPREF_OK;
    return launch_scatter_add_rows(src, rows, n, dim, table, (cudaStream_t)stream);
}

int invpref_mask_scores(float* rating, int64_t b, int64_t n_items, const int64_t* users, const int64_t* off,
                        const int64_t* items, float value, int32_t add, void* stream) {
    if (b < 0 || n_items < 1 || (b > 0 && (!rating || !users || !off))) return INVPREF_ERR_BAD_ARG;
    if (b == 0 || !items) return INVPREF_OK;     // items == NULL: every list is empty
    return launch_mask_scores(rating, b, n_items, users, off, items, value, add, (cudaStream_t)stream);
}

int invpref_hits_from_csr(const int64_t* top, int64_t b, int32_t k, const int64_t* users, const int64_t* off,
                          const int64_t* items, uint8_t* hits, int64_t* n_list, void* stream) {
    if (b < 0 || k < 1 || (b > 0 && (!top || !users || !off || !items || !hits))) return INVPREF_ERR_BAD_ARG;
    if (b == 0) return INVPREF_OK;
    return launch_hits_from_csr(top, b, k, users, off, items, hits, n_list, (cudaStream_t)stream);
}

int invpref_eval_topk(const invpref_desc* desc, const invpref_params* params, const int64_t* users, int64_t b,
                      const int64_t* mask_off, const int64_t* mask_items, const int64_t* pool_off,
                      const int64_t* pool_items, const int64_t* gt_off, const int64_t* gt_items, int32_t k,
                      int64_t* top_items, float* top_scores, uint8_t* hits, int64_t* n_gt, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if (!params || !params->Uinv || !params->Iinv) return INVPREF_ERR_BAD_ARG;
    if (b < 0 || k < 1 || k > 256 || k > desc->n_items || (b > 0 && (!users || !top_items))) return INVPREF_ERR_BAD_ARG;
    if ((mask_off && !mask_items) || (pool_off && !pool_items) || (gt_off && !gt_items)) return INVPREF_ERR_BAD_ARG;
    if ((hits || n_gt) && !gt_off) return INVPREF_ERR_BAD_ARG;
    if (b == 0) return INVPREF_OK;
    return launch_eval_topk(params->Uinv, params->Iinv, desc->n_items, g.D, desc->implicit, users, b, mask_off,
                            mask_items, pool_off, pool_items, gt_off, gt_items, k, top_items, top_scores, hits, n_gt,
                            (cudaStream_t)stream);
}

int invpref_recommend(const invpref_desc* desc, const invpref_params* params, const int64_t* users, int64_t b,
                      const int64_t* excl_off, const int64_t* excl_items, int32_t k, int64_t* top_items,
                      float* top_scores, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if (!params || !params->Uinv || !params->Iinv) return INVPREF_ERR_BAD_ARG;
    if (b < 0 || k < 1 || k > 256 || k > desc->n_items || (b > 0 && (!users || !top_items || !top_scores)))
        return INVPREF_ERR_BAD_ARG;
    if (excl_off && !excl_items) return INVPREF_ERR_BAD_ARG;
    if (b == 0) return INVPREF_OK;
    return launch_topk_stream(params->Uinv, users, b, params->Iinv, desc->n_items, g.D, desc->implicit, nullptr,
                              excl_off, excl_items, nullptr, nullptr, 1, nullptr, nullptr, k, top_items, top_scores,
                              nullptr, nullptr, (cudaStream_t)stream);
}

int invpref_similar_items(const invpref_desc* desc, const invpref_params* params, const int64_t* items, int64_t b,
                          int32_t k, float* inv_norm, int64_t* top_items, float* top_scores, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if (!params || !params->Iinv) return INVPREF_ERR_BAD_ARG;
    if (b < 0 || k < 1 || k > 256 || k > desc->n_items || (b > 0 && (!items || !inv_norm || !top_items || !top_scores)))
        return INVPREF_ERR_BAD_ARG;
    if (b == 0) return INVPREF_OK;
    cudaStream_t st = (cudaStream_t)stream;
    if ((rc = launch_row_inv_norm(params->Iinv, desc->n_items, g.D, inv_norm, st)) != INVPREF_OK) return rc;
    return launch_topk_stream(params->Iinv, items, b, params->Iinv, desc->n_items, g.D, 0, inv_norm, nullptr,
                              nullptr, nullptr, nullptr, 1, nullptr, nullptr, k, top_items, top_scores, nullptr,
                              nullptr, st);
}

int invpref_top_users(const invpref_desc* desc, const invpref_params* params, const int64_t* items, int64_t b,
                      const int64_t* excl_off, const int64_t* excl_users, int32_t k, int64_t* top_users,
                      float* top_scores, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if (!params || !params->Uinv || !params->Iinv) return INVPREF_ERR_BAD_ARG;
    if (b < 0 || k < 1 || k > 256 || k > desc->n_users || (b > 0 && (!items || !top_users || !top_scores)))
        return INVPREF_ERR_BAD_ARG;
    if (excl_off && !excl_users) return INVPREF_ERR_BAD_ARG;
    if (b == 0) return INVPREF_OK;
    return launch_topk_stream(params->Iinv, items, b, params->Uinv, desc->n_users, g.D, desc->implicit, nullptr,
                              excl_off, excl_users, nullptr, nullptr, 1, nullptr, nullptr, k, top_users, top_scores,
                              nullptr, nullptr, (cudaStream_t)stream);
}

static int fold_in(const invpref_desc* desc, const float* V, int64_t n_cat, const int64_t* off, const int64_t* ids,
                   const float* scores, int64_t b, double l2, int32_t max_iter, float* rows, int32_t* iters,
                   void* stream) {
    if (!desc) return INVPREF_ERR_BAD_ARG;
    if (desc->dim < 1 || desc->dim > fold_in_max_dim()) return INVPREF_ERR_BAD_DIM;
    if (desc->n_users < 1 || desc->n_items < 1 || !V) return INVPREF_ERR_BAD_ARG;
    if (!(l2 > 0.0) || !isfinite(l2) || max_iter < 1 || b < 0) return INVPREF_ERR_BAD_ARG;
    if (b > 0 && (!off || !ids || !scores || !rows)) return INVPREF_ERR_BAD_ARG;
    if (b == 0) return INVPREF_OK;
    return launch_fold_in(V, n_cat, desc->dim, desc->implicit, off, ids, scores, b, l2, max_iter, rows, iters,
                          (cudaStream_t)stream);
}

int invpref_fold_in_users(const invpref_desc* desc, const invpref_params* params, const int64_t* off,
                          const int64_t* items, const float* scores, int64_t b, double l2, int32_t max_iter,
                          float* rows, int32_t* iters, void* stream) {
    if (!desc || !params) return INVPREF_ERR_BAD_ARG;
    return fold_in(desc, params->Iinv, desc->n_items, off, items, scores, b, l2, max_iter, rows, iters, stream);
}

int invpref_fold_in_items(const invpref_desc* desc, const invpref_params* params, const int64_t* off,
                          const int64_t* users, const float* scores, int64_t b, double l2, int32_t max_iter,
                          float* rows, int32_t* iters, void* stream) {
    if (!desc || !params) return INVPREF_ERR_BAD_ARG;
    return fold_in(desc, params->Uinv, desc->n_users, off, users, scores, b, l2, max_iter, rows, iters, stream);
}

int invpref_recommend_rows(const invpref_desc* desc, const invpref_params* params, const float* rows,
                           const int64_t* row_ids, int64_t b, const int64_t* excl_off, const int64_t* excl_items,
                           int32_t k, int64_t* top_items, float* top_scores, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if (!params || !params->Iinv) return INVPREF_ERR_BAD_ARG;
    if (b < 0 || k < 1 || k > 256 || k > desc->n_items ||
        (b > 0 && (!rows || !row_ids || !top_items || !top_scores)))
        return INVPREF_ERR_BAD_ARG;
    if (excl_off && !excl_items) return INVPREF_ERR_BAD_ARG;
    if (b == 0) return INVPREF_OK;
    return launch_topk_stream(rows, row_ids, b, params->Iinv, desc->n_items, g.D, desc->implicit, nullptr, excl_off,
                              excl_items, nullptr, nullptr, 1, nullptr, nullptr, k, top_items, top_scores, nullptr,
                              nullptr, (cudaStream_t)stream);
}

int invpref_top_users_rows(const invpref_desc* desc, const invpref_params* params, const float* rows,
                           const int64_t* row_ids, int64_t b, const int64_t* excl_off, const int64_t* excl_users,
                           int32_t k, int64_t* top_users, float* top_scores, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if (!params || !params->Uinv) return INVPREF_ERR_BAD_ARG;
    if (b < 0 || k < 1 || k > 256 || k > desc->n_users ||
        (b > 0 && (!rows || !row_ids || !top_users || !top_scores)))
        return INVPREF_ERR_BAD_ARG;
    if (excl_off && !excl_users) return INVPREF_ERR_BAD_ARG;
    if (b == 0) return INVPREF_OK;
    return launch_topk_stream(rows, row_ids, b, params->Uinv, desc->n_users, g.D, desc->implicit, nullptr, excl_off,
                              excl_users, nullptr, nullptr, 1, nullptr, nullptr, k, top_users, top_scores, nullptr,
                              nullptr, (cudaStream_t)stream);
}

int invpref_fetch_rows_p2p(const float* const* tables, int32_t world, const int32_t* owner, const int64_t* rows,
                           int64_t n, int32_t dim, float* out_inv, float* out_env, void* stream) {
    if (n < 0 || dim < 1 || !tables || (n > 0 && (!owner || !rows || !out_inv || !out_env))) return INVPREF_ERR_BAD_ARG;
    for (int i = 0; i < 2 * world && world >= 1 && world <= 16; ++i)
        if (!tables[i]) return INVPREF_ERR_BAD_ARG;
    if (n == 0) return INVPREF_OK;
    return launch_fetch_rows_p2p(tables, world, owner, rows, n, dim, out_inv, out_env, (cudaStream_t)stream);
}

int invpref_owner_adam_push(float* theta_inv, float* theta_env, float* m_inv, float* m_env, float* v_inv, float* v_env,
                            int64_t n_rows, int32_t dim, int32_t world, const float* stage_inv, const float* stage_env,
                            const int32_t* spos, float* const* caches, const int32_t* npos,
                            const invpref_hyper* hyper, void* stream) {
    if (n_rows < 0 || dim < 1 || world < 1 || world > 16 || !hyper || hyper->step < 1) return INVPREF_ERR_BAD_ARG;
    if (n_rows > 0 && (!theta_inv || !theta_env || !m_inv || !m_env || !v_inv || !v_env || !spos || !stage_inv ||
                       !stage_env))
        return INVPREF_ERR_BAD_ARG;
    if ((caches == nullptr) != (npos == nullptr)) return INVPREF_ERR_BAD_ARG;
    for (int i = 0; caches && i < 2 * world; ++i)
        if (!caches[i]) return INVPREF_ERR_BAD_ARG;
    if (n_rows == 0) return INVPREF_OK;
    return launch_owner_adam_push(theta_inv, theta_env, m_inv, m_env, v_inv, v_env, n_rows, dim, world, stage_inv,
                                  stage_env, spos, caches, npos, make_adam(hyper), hyper->dyn, (cudaStream_t)stream);
}

int invpref_peer_allreduce(float* buf, int32_t n, int32_t n_max, int32_t world, int32_t rank, float* const* peer_slots,
                           uint32_t* const* peer_flags, uint32_t* counter, int32_t* status, void* stream) {
    if (world < 1 || world > 16 || rank < 0 || rank >= world || n < 0 || n > n_max || !peer_slots || !peer_flags ||
        !counter || !status || (n > 0 && !buf))
        return INVPREF_ERR_BAD_ARG;
    for (int p = 0; p < world; ++p)
        if (!peer_flags[p] || (n_max > 0 && !peer_slots[p])) return INVPREF_ERR_BAD_ARG;
    return launch_peer_allreduce(buf, n, n_max, world, rank, peer_slots, peer_flags, counter, status,
                                 (cudaStream_t)stream);
}

int invpref_backward(const invpref_desc* desc, const invpref_params* params, const invpref_batch* batch, double alpha,
                     const float* g_s_inv, const float* g_s_env, const float* g_logp, const void* plan,
                     invpref_params* grads, void* ws, size_t ws_bytes, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if ((rc = check_tables(g, params)) != INVPREF_OK) return rc;
    if ((rc = check_tables(g, grads)) != INVPREF_OK) return rc;
    if (!batch || !ws) return INVPREF_ERR_BAD_ARG;
    const int64_t B = batch->B;
    if (B < 0 || B > 0x7fffffffLL) return INVPREF_ERR_BAD_ARG;
    if (B == 0) return INVPREF_OK;
    if (!batch->users || !batch->items || !batch->envs) return INVPREF_ERR_BAD_ARG;
    Workspace w;
    if (ws_bytes < workspace_bytes_impl(desc, g, B, &w, (char*)ws)) return INVPREF_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const char* plan_base = (const char*)plan;
    if (plan_base == nullptr) {
        rc = build_plan_impl(desc, batch->users, batch->items, B, w.plan, w.sort_tmp, w.sort_tmp_bytes, st);
        if (rc != INVPREF_OK) return rc;
        plan_base = w.plan;
    }
    PlanSide pu, pi;
    carve_plan(desc, B, (char*)plan_base, &pu, &pi);

    FwdTrainArgs f;
    f.Uinv = params->Uinv; f.Iinv = params->Iinv; f.Uenv = params->Uenv; f.Ienv = params->Ienv;
    f.E = params->E; f.W = params->W; f.b = params->b;
    f.users = batch->users; f.items = batch->items; f.envs = batch->envs;
    f.scores = nullptr; f.weights = nullptr; f.B = B;
    f.D = g.D; f.K = g.K; f.GS = g.GS;
    f.implicit = desc->implicit; f.reg_env_embed = 0; f.use_class_rw = 0; f.use_rec_rw = 0;
    f.c_inv = f.c_ea = f.c_env = 0.f; f.neg_alpha = (float)(-alpha); f.invB = 0.f;
    f.gpack = w.gpack; f.partials = w.partials; f.P = fwd_partial_floats(g);
    f.up_s_inv = g_s_inv; f.up_s_env = g_s_env; f.up_logp = g_logp; f.generic = 1; f.dyn = nullptr;
    const int fgrid = fwd_train_grid(B);
    if ((rc = launch_fwd_train(g, f, fgrid, st)) != INVPREF_OK) return rc;

    AdamScalars as = {};
    BwdSideArgs su = {}, si = {};
    fill_side(&su, g, w.gpack, params->E, params->W);
    su.partner_inv = params->Iinv; su.partner_env = params->Ienv;
    su.grad_inv = grads->Uinv; su.grad_env = grads->Uenv; su.plan = pu; su.chunk_part = w.chunk_part_u; su.adam = as;
    fill_side(&si, g, w.gpack, params->E, params->W);
    si.partner_inv = params->Uinv; si.partner_env = params->Uenv;
    si.grad_inv = grads->Iinv; si.grad_env = grads->Ienv; si.plan = pi; si.chunk_part = w.chunk_part_i; si.adam = as;
    if ((rc = launch_bwd_chunks(g, si, st)) != INVPREF_OK) return rc;
    if ((rc = launch_bwd_chunks(g, su, st)) != INVPREF_OK) return rc;
    if ((rc = launch_bwd_rows(g, si, EPI_ACCUM, st)) != INVPREF_OK) return rc;
    if ((rc = launch_bwd_rows(g, su, EPI_ACCUM, st)) != INVPREF_OK) return rc;

    TailArgs t = {};
    t.partials = w.partials; t.n_partials = fgrid; t.P = f.P; t.B = B; t.D = g.D; t.K = g.K;
    t.gE = grads->E; t.gW = grads->W; t.gb = grads->b; t.epi = EPI_ACCUM;
    return launch_tail(t, st);
}

int invpref_cluster(const invpref_desc* desc, const invpref_params* params, const int64_t* users, const int64_t* items,
                    const float* scores, const int64_t* perm_idx, const float* eps_table, const int64_t* old_envs,
                    int64_t B, int64_t* new_envs, int64_t* hist, int64_t* diff, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if ((rc = check_tables(g, params)) != INVPREF_OK) return rc;
    if (B < 0 || (B > 0 && (!users || !items || !scores || !new_envs))) return INVPREF_ERR_BAD_ARG;
    if (perm_idx && !eps_table) return INVPREF_ERR_BAD_ARG;
    if (diff && !old_envs) return INVPREF_ERR_BAD_ARG;
    if (B == 0) return INVPREF_OK;
    ClusterArgs a;
    a.Uinv = params->Uinv; a.Iinv = params->Iinv; a.Uenv = params->Uenv; a.Ienv = params->Ienv; a.E = params->E;
    a.users = users; a.items = items; a.scores = scores; a.perm_idx = perm_idx; a.eps_table = eps_table;
    a.old_envs = old_envs; a.B = B; a.D = g.D; a.K = g.K; a.implicit = desc->implicit;
    a.new_envs = new_envs; a.hist = (unsigned long long*)hist; a.diff = (unsigned long long*)diff;
    a.perm = nullptr; a.users32 = nullptr; a.items32 = nullptr;
    return launch_cluster(g, a, (cudaStream_t)stream);
}

int invpref_cluster_sorted(const invpref_desc* desc, const invpref_params* params, const int32_t* perm,
                           const int32_t* users_sorted, const int32_t* items_sorted, const float* scores_sorted,
                           const int64_t* perm_idx, const float* eps_table, const int64_t* old_envs, int64_t N,
                           int64_t* new_envs, int64_t* hist, int64_t* diff, void* stream) {
    Geometry g;
    int rc = make_geometry(desc, &g);
    if (rc != INVPREF_OK) return rc;
    if ((rc = check_tables(g, params)) != INVPREF_OK) return rc;
    if (N < 0 || N > 0x7fffffffLL || (N > 0 && (!perm || !users_sorted || !items_sorted || !scores_sorted || !new_envs)))
        return INVPREF_ERR_BAD_ARG;
    if (perm_idx && !eps_table) return INVPREF_ERR_BAD_ARG;
    if (diff && !old_envs) return INVPREF_ERR_BAD_ARG;
    if (N == 0) return INVPREF_OK;
    ClusterArgs a;
    a.Uinv = params->Uinv; a.Iinv = params->Iinv; a.Uenv = params->Uenv; a.Ienv = params->Ienv; a.E = params->E;
    a.users = nullptr; a.items = nullptr; a.scores = scores_sorted; a.perm_idx = perm_idx; a.eps_table = eps_table;
    a.old_envs = old_envs; a.B = N; a.D = g.D; a.K = g.K; a.implicit = desc->implicit;
    a.new_envs = new_envs; a.hist = (unsigned long long*)hist; a.diff = (unsigned long long*)diff;
    a.perm = perm; a.users32 = users_sorted; a.items32 = items_sorted;
    return launch_cluster(g, a, (cudaStream_t)stream);
}

int invpref_stat_envs(const int64_t* envs, int64_t N, int32_t n_envs, const int64_t* hist, float* class_weights,
                      float* sample_weights, void* stream) {
    if (n_envs < 1 || n_envs > INVPREF_MAX_ENVS) return INVPREF_ERR_BAD_ENVS;
    if (N < 1 || !hist || (sample_weights && !envs)) return INVPREF_ERR_BAD_ARG;
    return launch_stat_envs(envs, N, n_envs, hist, class_weights, sample_weights, (cudaStream_t)stream);
}

int invpref_env_hist(const int64_t* envs, int64_t N, int32_t n_envs, int64_t* hist, void* stream) {
    if (n_envs < 1 || n_envs > INVPREF_MAX_ENVS) return INVPREF_ERR_BAD_ENVS;
    if (N < 0 || !hist || (N > 0 && !envs)) return INVPREF_ERR_BAD_ARG;
    if (N == 0) return INVPREF_OK;
    return launch_env_hist(envs, N, n_envs, (unsigned long long*)hist, (cudaStream_t)stream);
}

}  // extern "C"
