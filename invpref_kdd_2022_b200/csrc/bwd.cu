// Deterministic segmented backward + fused dense Adam.
//
// Replaces, for the four embedding tables, ATen's embedding_dense_backward (zero-fill + index_add,
// 13x per step in the reference: autograd of models.py:449-455 and of the re-gathers in
// models.py:469-532), the norm backward (2x / sign(x)) and torch.optim.Adam.step (train.py:832-834).
//
//  bwd_chunks_kernel : pre-reduces CHUNK-sized pieces of long segments (hot items) into partials.
//  bwd_rows_kernel   : one 16-lane group per touched row: sums its segment (or its chunk partials) in
//                      the fixed sorted order -- no atomics -- adds the L1/L2 term of the row, and
//                      applies Adam in registers; the gradient table is never materialised.
//  sweep_kernel      : dense Adam for every row WITHOUT a segment (g = 0: momentum still moves it),
//                      a pure stream over theta, m, v.
//  tail_kernel       : fixed-order sum of the forward kernel's per-CTA partials -> the six loss
//                      scalars (train.py:836-843), gradients of E / W / b and their Adam update.
#include "common.cuh"
#include "kernels.h"

namespace invpref {

namespace {

// Sum over sorted positions [beg, end) of this side's per-interaction gradient contributions:
//   acc_inv += (g_z1 + sum_k (-alpha g_logits[k]) W[k, d]) * partner_inv[d]      (g_p (.) partner)
//   acc_env += g_z2 * partner_env[d] * E[e, d]
template <int VEC, int NV, bool STASH>
__device__ __forceinline__ void accumulate_range(const BwdSideArgs& a, const float* __restrict__ sE,
                                                 const float* __restrict__ sW, int beg, int end, int lane,
                                                 float* acc_inv, float* acc_env) {
    const int D = a.D, K = a.K, GS = a.GS;
    const int32_t* __restrict__ perm = a.plan.perm;
    // lazy mode: the partner (user) rows of this step were stashed, caught up, by the user pass, indexed by
    // the user's segment: row 2*seg = invariant, 2*seg+1 = env-aware
    const int32_t* __restrict__ partner = STASH ? a.plan.pseg : a.plan.partner;
    const float* __restrict__ pinv = STASH ? a.stash : a.partner_inv;
    const float* __restrict__ penv = STASH ? a.stash + D : a.partner_env;
    constexpr int pmul = STASH ? 2 : 1;
    // software pipeline: the partner rows / g-pack of interaction k+PF are requested into L2 now; their
    // indices were loaded one iteration earlier, so the (in-order) warp never waits for them
    constexpr int PF = 4;
    int pid_q = 0, n_q = 0;
    if (beg + PF < end) { pid_q = partner[beg + PF]; n_q = perm[beg + PF]; }
    for (int k = beg; k < end; ++k) {
        if (k + PF < end) {
            prefetch_row(pinv, pid_q * pmul, D, lane);
            prefetch_row(penv, pid_q * pmul, D, lane);
            if (lane == 8) prefetch_l2(a.gpack + (int64_t)n_q * GS);
        }
        if (k + 1 + PF < end) { pid_q = partner[k + 1 + PF]; n_q = perm[k + 1 + PF]; }
        const int n = perm[k];
        const int pid = partner[k];
        const float4* gp = reinterpret_cast<const float4*>(a.gpack + (int64_t)n * GS);
        float g[12];
        float4 q0 = gp[0], q1 = gp[1];
        g[0] = q0.x; g[1] = q0.y; g[2] = q0.z; g[3] = q0.w;
        g[4] = q1.x; g[5] = q1.y; g[6] = q1.z; g[7] = q1.w;
        if (GS > 8) {
            float4 q2 = gp[2];
            g[8] = q2.x; g[9] = q2.y; g[10] = q2.z; g[11] = q2.w;
        } else {
            g[8] = g[9] = g[10] = g[11] = 0.f;
        }
        Row<VEC, NV> pc, pe;
        load_row<VEC, NV>(pc, pinv, pid * pmul, D, lane);
        load_row<VEC, NV>(pe, penv, pid * pmul, D, lane);
        const float g_z1 = g[0], g_z2 = g[1];
        const int e = __float_as_int(g[2]);
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int d0 = dim_of<VEC>(lane, j);
            if (d0 < D) {
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    const int x = j * VEC + v;
                    float gpd = g_z1;
#pragma unroll
                    for (int kk = 0; kk < INVPREF_MAX_ENVS; ++kk)
                        if (kk < K) gpd += g[3 + kk] * sW[kk * D + d0 + v];
                    acc_inv[x] += gpd * pc.x[x];
                    acc_env[x] += g_z2 * pe.x[x] * sE[e * D + d0 + v];
                }
            }
        }
    }
}

__device__ __forceinline__ void stage_EW(const BwdSideArgs& a, float* sE, float* sW) {
    for (int t = threadIdx.x; t < a.K * a.D; t += blockDim.x) {
        sE[t] = a.E[t];
        sW[t] = a.W[t];
    }
    __syncthreads();
}

// Epilogue of one row: its own L1/L2 term (models.py:469-497, every occurrence counts), then Adam in
// registers / gradient export / accumulation into a dense gradient.
template <int VEC, int NV, int EPI>
__device__ __forceinline__ void finish_row(const BwdSideArgs& a, int64_t row, float cnt, Row<VEC, NV>& th_i,
                                           Row<VEC, NV>& th_e, Row<VEC, NV>& m_i, Row<VEC, NV>& m_e,
                                           Row<VEC, NV>& v_i, Row<VEC, NV>& v_e, Row<VEC, NV>& gi, Row<VEC, NV>& ge,
                                           int lane, int D) {
    const AdamScalars adam = with_dyn(a.adam, a.dyn);   // read where it is used: no register held over the segment
    if (EPI == EPI_ADAM || EPI == EPI_EXPORT) {
#pragma unroll
        for (int x = 0; x < NV * VEC; ++x) {
            gi.x[x] += cnt * (a.reg2 * th_i.x[x] + mul_sign(a.reg1, th_i.x[x]));
            ge.x[x] += cnt * (a.reg2 * th_e.x[x] + mul_sign(a.reg1, th_e.x[x]));
        }
        if (EPI == EPI_EXPORT && a.push_base != nullptr) {
            // straight into the owner's staging buffer over NVLink (posted writes)
            const int o = a.push_owner[row];
            const int64_t idx = a.push_index[row];
            store_row<VEC, NV>(gi, a.push_base[o], idx, D, lane);
            store_row<VEC, NV>(ge, a.push_base[a.push_world + o], idx, D, lane);
        } else if (a.grad_inv != nullptr) {
            store_row<VEC, NV>(gi, a.grad_inv, row, D, lane);
            store_row<VEC, NV>(ge, a.grad_env, row, D, lane);
        }
    }
    if (EPI == EPI_ADAM) {
#pragma unroll
        for (int x = 0; x < NV * VEC; ++x) {
            adam_update(th_i.x[x], m_i.x[x], v_i.x[x], gi.x[x], adam);
            adam_update(th_e.x[x], m_e.x[x], v_e.x[x], ge.x[x], adam);
        }
        store_row<VEC, NV>(th_i, a.own_inv_out, row, D, lane);
        store_row<VEC, NV>(th_e, a.own_env_out, row, D, lane);
        store_row<VEC, NV, true>(m_i, a.m_inv, row, D, lane);
        store_row<VEC, NV, true>(m_e, a.m_env, row, D, lane);
        store_row<VEC, NV, true>(v_i, a.v_inv, row, D, lane);
        store_row<VEC, NV, true>(v_e, a.v_env, row, D, lane);
    } else if (EPI == EPI_ACCUM) {
        Row<VEC, NV> oi, oe;
        load_row<VEC, NV>(oi, a.grad_inv, row, D, lane);
        load_row<VEC, NV>(oe, a.grad_env, row, D, lane);
#pragma unroll
        for (int x = 0; x < NV * VEC; ++x) { oi.x[x] += gi.x[x]; oe.x[x] += ge.x[x]; }
        store_row<VEC, NV>(oi, a.grad_inv, row, D, lane);
        store_row<VEC, NV>(oe, a.grad_env, row, D, lane);
    }
}

template <int VEC, int NV, bool STASH>
__global__ void __launch_bounds__(BLOCK, 3) bwd_chunks_kernel(BwdSideArgs a) {
    extern __shared__ float smem[];
    float* sE = smem;
    float* sW = smem + a.K * a.D;
    stage_EW(a, sE, sW);
    const int lane = threadIdx.x & (GROUP - 1);
    const int n_chunks = a.plan.counters[1];
    const int ngroups = gridDim.x * GROUPS_PER_BLOCK;
    for (int c = blockIdx.x * GROUPS_PER_BLOCK + (threadIdx.x >> 4); c < n_chunks; c += ngroups) {
        const int4 desc = reinterpret_cast<const int4*>(a.plan.chunk_desc)[c];
        Row<VEC, NV> ai, ae;
#pragma unroll
        for (int x = 0; x < NV * VEC; ++x) { ai.x[x] = 0.f; ae.x[x] = 0.f; }
        accumulate_range<VEC, NV, STASH>(a, sE, sW, desc.y, desc.z, lane, ai.x, ae.x);
        store_row<VEC, NV>(ai, a.chunk_part, (int64_t)c * 2, a.D, lane);
        store_row<VEC, NV>(ae, a.chunk_part, (int64_t)c * 2 + 1, a.D, lane);
    }
}

template <int VEC, int NV, int EPI, bool STASH>
__global__ void __launch_bounds__(BLOCK, 3) bwd_rows_kernel(BwdSideArgs a) {
    extern __shared__ float smem[];
    float* sE = smem;
    float* sW = smem + a.K * a.D;
    stage_EW(a, sE, sW);
    const int D = a.D;
    const int lane = threadIdx.x & (GROUP - 1);
    const int n_seg = a.plan.counters[0];
    const int ngroups = gridDim.x * GROUPS_PER_BLOCK;
    for (int s = blockIdx.x * GROUPS_PER_BLOCK + (threadIdx.x >> 4); s < n_seg; s += ngroups) {
        const int64_t row = a.plan.seg_row[s];
        const int beg = a.plan.seg_off[s], end = a.plan.seg_off[s + 1];
        const int c0 = a.plan.seg_chunk[s], c1 = a.plan.seg_chunk[s + 1];
        Row<VEC, NV> th_i, th_e, m_i, m_e, v_i, v_e;
        if (EPI == EPI_ADAM || EPI == EPI_EXPORT) {
            load_row<VEC, NV>(th_i, a.own_inv_in, row, D, lane);
            load_row<VEC, NV>(th_e, a.own_env_in, row, D, lane);
        }
        if (EPI == EPI_ADAM) {
            load_row<VEC, NV, true>(m_i, a.m_inv, row, D, lane);
            load_row<VEC, NV, true>(m_e, a.m_env, row, D, lane);
            load_row<VEC, NV, true>(v_i, a.v_inv, row, D, lane);
            load_row<VEC, NV, true>(v_e, a.v_env, row, D, lane);
        }
        Row<VEC, NV> gi, ge;
#pragma unroll
        for (int x = 0; x < NV * VEC; ++x) { gi.x[x] = 0.f; ge.x[x] = 0.f; }
        if (c1 > c0) {
            for (int c = c0; c < c1; ++c) {
                Row<VEC, NV> pi, pe;
                load_row<VEC, NV>(pi, a.chunk_part, (int64_t)c * 2, D, lane);
                load_row<VEC, NV>(pe, a.chunk_part, (int64_t)c * 2 + 1, D, lane);
#pragma unroll
                for (int x = 0; x < NV * VEC; ++x) { gi.x[x] += pi.x[x]; ge.x[x] += pe.x[x]; }
            }
        } else {
            accumulate_range<VEC, NV, STASH>(a, sE, sW, beg, end, lane, gi.x, ge.x);
        }
        finish_row<VEC, NV, EPI>(a, row, (float)(end - beg), th_i, th_e, m_i, m_e, v_i, v_e, gi, ge, lane, D);
    }
}

constexpr int RING = 4;   // interactions in flight per group (ring kernels); deeper rings measured slower (DESIGN.md §3)

// One interaction of the ring kernels: its g-pack (shared by the group) and the two partner-row slices this
// lane staged, accumulated exactly as accumulate_range does.
template <int VEC, int NV, int KX>
__device__ __forceinline__ void ring_consume(const float* __restrict__ gslot, const float* __restrict__ ring,
                                             int rslot, const float* __restrict__ sE, const float* __restrict__ sW,
                                             int D, int K, int GS, int lane, Row<VEC, NV>& gi, Row<VEC, NV>& ge) {
    float gq[12];
    {
        const float4* gp = reinterpret_cast<const float4*>(gslot);
        const float4 q0 = gp[0], q1 = gp[1];
        gq[0] = q0.x; gq[1] = q0.y; gq[2] = q0.z; gq[3] = q0.w;
        gq[4] = q1.x; gq[5] = q1.y; gq[6] = q1.z; gq[7] = q1.w;
        if (GS > 8) {
            const float4 q2 = gp[2];
            gq[8] = q2.x; gq[9] = q2.y; gq[10] = q2.z; gq[11] = q2.w;
        } else {
            gq[8] = gq[9] = gq[10] = gq[11] = 0.f;
        }
    }
    Row<VEC, NV> pc, pe;
    read_staged_row<VEC, NV>(pc, ring, rslot * 2 + 0, D, lane);
    read_staged_row<VEC, NV>(pe, ring, rslot * 2 + 1, D, lane);
    const float g_z1 = gq[0], g_z2 = gq[1];
    const int e = __float_as_int(gq[2]);
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int d0 = dim_of<VEC>(lane, j);
        if (d0 < D) {
            float ee[VEC], gpd[VEC];
            ldv<VEC>(sE + e * D + d0, ee);
#pragma unroll
            for (int v = 0; v < VEC; ++v) gpd[v] = g_z1;
#pragma unroll
            for (int kk = 0; kk < (KX ? KX : INVPREF_MAX_ENVS); ++kk) {
                if (kk < K) {
                    float wk[VEC];
                    ldv<VEC>(sW + kk * D + d0, wk);
#pragma unroll
                    for (int v = 0; v < VEC; ++v) gpd[v] += gq[3 + kk] * wk[v];
                }
            }
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                const int x = j * VEC + v;
                gi.x[x] += gpd[v] * pc.x[x];
                ge.x[x] += g_z2 * pe.x[x] * ee[v];
            }
        }
    }
}

// Ring version of bwd_chunks_kernel: a group walks its chunks (c = g, g + G, ...) with the producer RING-1
// interactions ahead, across chunk boundaries.  Chunks are spread over the CTAs first (a few hundred chunks of
// a few hundred sequential interactions each: the critical path of the item pass).
template <int VEC, int NV, bool STASH, int KX, int DX = GROUP * VEC * NV>
__global__ void __launch_bounds__(BLOCK, 3) bwd_chunks_ring_kernel(BwdSideArgs a) {
    extern __shared__ __align__(128) float smem[];
    const int D = KX ? DX : a.D, K = KX ? KX : a.K, GS = KX ? (KX <= 5 ? 8 : 12) : a.GS, KD = K * D;
    float* sE = smem;
    float* sW = smem + KD;
    float* sG = smem + ((2 * KD + 3) & ~3);
    float* ring = smem + ring_align_up(((2 * KD + 3) & ~3) + GROUPS_PER_BLOCK * (RING + 1) * 12);
    stage_EW(a, sE, sW);
    const int lane = threadIdx.x & (GROUP - 1);
    const unsigned gmask = group_mask();
    float* myG = sG + (threadIdx.x >> 4) * (RING + 1) * 12;
    const int n_chunks = a.plan.counters[1];
    const int4* __restrict__ chunk_desc = reinterpret_cast<const int4*>(a.plan.chunk_desc);
    const int32_t* __restrict__ perm = a.plan.perm;
    const int32_t* __restrict__ partner = STASH ? a.plan.pseg : a.plan.partner;
    const float* __restrict__ pinv = STASH ? a.stash : a.partner_inv;
    const float* __restrict__ penv = STASH ? a.stash + D : a.partner_env;
    constexpr int pmul = STASH ? 2 : 1;
    const int G = gridDim.x * GROUPS_PER_BLOCK;
    const int g = blockIdx.x + gridDim.x * (threadIdx.x >> 4);

    // producer: chunk pc, position pk in [.., pend); the next chunk's bounds are loaded one chunk ahead
    int pc = g, pk = 0, pend = 0, nk = 0, nend = 0, n_q = 0, pid_q = 0;
    auto p_enter = [&]() {
        pk = nk; pend = nend;
        if (pc + G < n_chunks) { const int4 d = chunk_desc[pc + G]; nk = d.y; nend = d.z; }
    };
    if (pc < n_chunks) {
        const int4 d = chunk_desc[pc];
        nk = d.y; nend = d.z;
        p_enter();
        n_q = perm[pk]; pid_q = partner[pk];
    }
    int wslot = 0, wgs = 0;
    auto produce = [&]() {
        if (pc < n_chunks) {
            stage_row_async<VEC, NV>(ring, wslot * 2 + 0, pinv, (int64_t)pid_q * pmul, D, lane);
            stage_row_async<VEC, NV>(ring, wslot * 2 + 1, penv, (int64_t)pid_q * pmul, D, lane);
            if (lane * 4 < GS) cp_async<16>(smem_addr(myG + wgs * 12 + lane * 4), a.gpack + (int64_t)n_q * GS + lane * 4);
            if (++pk == pend) { pc += G; if (pc < n_chunks) p_enter(); }
            if (pc < n_chunks) { n_q = perm[pk]; pid_q = partner[pk]; }
        }
        cp_async_commit();
        if (++wslot == RING) wslot = 0;
        if (++wgs == RING + 1) wgs = 0;
    };
#pragma unroll
    for (int q = 0; q < RING - 1; ++q) produce();

    int rslot = 0, rgs = 0;
    for (int c = g; c < n_chunks; c += G) {
        const int4 desc = chunk_desc[c];
        Row<VEC, NV> gi, ge;
#pragma unroll
        for (int x = 0; x < NV * VEC; ++x) { gi.x[x] = 0.f; ge.x[x] = 0.f; }
        for (int k = desc.y; k < desc.z; ++k) {
            produce();
            cp_async_wait<RING - 1>();
            __syncwarp(gmask);
            ring_consume<VEC, NV, KX>(myG + rgs * 12, ring, rslot, sE, sW, D, K, GS, lane, gi, ge);
            if (++rslot == RING) rslot = 0;
            if (++rgs == RING + 1) rgs = 0;
        }
        store_row<VEC, NV>(gi, a.chunk_part, (int64_t)c * 2, D, lane);
        store_row<VEC, NV>(ge, a.chunk_part, (int64_t)c * 2 + 1, D, lane);
    }
    cp_async_wait<0>();
}

// ---------------------------------------------------------------------------------------------------------
// Ring rows kernel (row slices of <= 16 bytes per lane, i.e. D <= 64; Adam / export epilogues).
//
// ncu on bwd_rows_kernel (round 1): 47 % of the warp samples wait on the long scoreboard -- perm/partner ->
// g-pack + two partner rows per interaction, L2 prefetch or not.  Here
//  * the plan cuts the segments into cost-balanced CONTIGUOUS ranges (plan.cu: write_chunks_ranges_kernel); a group
//    takes ranges g, g + G, ...: inside a range the sorted positions it walks are contiguous across segment
//    boundaries, and the strided assignment averages out what the cost model misses (a first version with ONE
//    range per group ran 1.5x longer on its slowest SM than on average);
//  * a producer cursor runs RING-1 interactions ahead of the consumer -- across segment and range boundaries
//    -- and copies the partner rows (each lane its own slice) and the g-pack of every interaction global ->
//    shared with cp.async: no register is held while the data is in flight;
//  * per segment the arithmetic is accumulate_range's / finish_row's, value for value and in the same order.
// KX > 0: D = DX (64, or 40 = the drivers' factor_num) and K = KX are compile-time constants (bounds guards fold away,
// row offsets are shifts and adds); KX = 0: any D, K.
template <int VEC, int NV, int EPI, bool STASH, int KX, int DX = GROUP * VEC * NV>
__global__ void __launch_bounds__(BLOCK, 3) bwd_rows_ring_kernel(BwdSideArgs a, int long_len) {
    extern __shared__ __align__(128) float smem[];
    const int D = KX ? DX : a.D, K = KX ? KX : a.K, GS = KX ? (KX <= 5 ? 8 : 12) : a.GS, KD = K * D;
    float* sE = smem;
    float* sW = smem + KD;
    float* sG = smem + ((2 * KD + 3) & ~3);                    // [groups][RING + 1][12] g-packs
    float* ring = smem + ring_align_up(((2 * KD + 3) & ~3) + GROUPS_PER_BLOCK * (RING + 1) * 12);   // [RING][2 rows][NV][BLOCK][VEC]
    stage_EW(a, sE, sW);
    const int lane = threadIdx.x & (GROUP - 1);
    const unsigned gmask = group_mask();
    float* myG = sG + (threadIdx.x >> 4) * (RING + 1) * 12;
    const int n_seg = a.plan.counters[0];
    const int NR = a.plan.counters[3];
    const int32_t* __restrict__ range_start = a.plan.range_start;
    const int32_t* __restrict__ seg_off = a.plan.seg_off;
    const int32_t* __restrict__ seg_row = a.plan.seg_row;
    const int32_t* __restrict__ perm = a.plan.perm;
    const int32_t* __restrict__ partner = STASH ? a.plan.pseg : a.plan.partner;
    const float* __restrict__ pinv = STASH ? a.stash : a.partner_inv;
    const float* __restrict__ penv = STASH ? a.stash + D : a.partner_env;
    constexpr int pmul = STASH ? 2 : 1;
    const int G = gridDim.x * GROUPS_PER_BLOCK;
    const int g = blockIdx.x * GROUPS_PER_BLOCK + (threadIdx.x >> 4);

    // ---- hot rows (more than HOT_CHUNKS chunk partials): one CTA per row.  Group q sums the q-th contiguous slice
    //      of the row's partials in chunk order (two row pairs in flight), the 16 slice sums meet in shared memory and
    //      group 0 adds them in slice order and finishes the row: a fixed two-level order, no atomics.  The ring
    //      below skips these rows.  (The ring's shared memory is free until the first produce().)
    {
        const int n_hot = a.plan.counters[4];
        const int grp = threadIdx.x >> 4;
        float* sHot = ring;                                   // [16 groups][2 rows][16 lanes][NV * VEC]
        for (int h = blockIdx.x; h < n_hot; h += gridDim.x) {
            const int cs = a.plan.hot_list[h];
            const int c0 = a.plan.seg_chunk[cs], c1 = a.plan.seg_chunk[cs + 1];
            const int per = (c1 - c0 + GROUPS_PER_BLOCK - 1) / GROUPS_PER_BLOCK;
            const int cb = c0 + grp * per, ce = (cb + per < c1) ? cb + per : c1;
            Row<VEC, NV> gi, ge;
#pragma unroll
            for (int x = 0; x < NV * VEC; ++x) { gi.x[x] = 0.f; ge.x[x] = 0.f; }
            for (int c = cb; c < ce; c += 2) {
                Row<VEC, NV> pi[2], pe[2];
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    if (c + q < ce) {
                        load_row<VEC, NV>(pi[q], a.chunk_part, (int64_t)(c + q) * 2, D, lane);
                        load_row<VEC, NV>(pe[q], a.chunk_part, (int64_t)(c + q) * 2 + 1, D, lane);
                    }
                }
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    if (c + q < ce) {
#pragma unroll
                        for (int x = 0; x < NV * VEC; ++x) { gi.x[x] += pi[q].x[x]; ge.x[x] += pe[q].x[x]; }
                    }
                }
            }
            float* mine = sHot + ((size_t)(grp * 2) * GROUP + lane) * (NV * VEC);
#pragma unroll
            for (int x = 0; x < NV * VEC; ++x) {
                mine[x] = gi.x[x];
                mine[GROUP * NV * VEC + x] = ge.x[x];
            }
            __syncthreads();
            if (grp == 0) {
#pragma unroll
                for (int x = 0; x < NV * VEC; ++x) { gi.x[x] = 0.f; ge.x[x] = 0.f; }
                for (int q = 0; q < GROUPS_PER_BLOCK; ++q) {
                    const float* sl = sHot + ((size_t)(q * 2) * GROUP + lane) * (NV * VEC);
#pragma unroll
                    for (int x = 0; x < NV * VEC; ++x) { gi.x[x] += sl[x]; ge.x[x] += sl[GROUP * NV * VEC + x]; }
                }
                const int64_t row = seg_row[cs];
                Row<VEC, NV> th_i, th_e, m_i, m_e, v_i, v_e;
                load_row<VEC, NV>(th_i, a.own_inv_in, row, D, lane);
                load_row<VEC, NV>(th_e, a.own_env_in, row, D, lane);
                if (EPI == EPI_ADAM) {
                    load_row<VEC, NV, true>(m_i, a.m_inv, row, D, lane);
                    load_row<VEC, NV, true>(m_e, a.m_env, row, D, lane);
                    load_row<VEC, NV, true>(v_i, a.v_inv, row, D, lane);
                    load_row<VEC, NV, true>(v_e, a.v_env, row, D, lane);
                }
                finish_row<VEC, NV, EPI>(a, row, (float)(seg_off[cs + 1] - seg_off[cs]), th_i, th_e, m_i, m_e, v_i, v_e,
                                         gi, ge, lane, D);
            }
            __syncthreads();
        }
    }

    // ---- producer cursor: the next interaction to request.  (pr, ps, pk): range, segment, sorted position;
    //      pr >= NR: exhausted.  Long segments (pre-reduced by the chunks kernel) are skipped.
    int pr = g, ps = 0, psb = 0, pk = 0, pend = 0, pend_nx = 0, nsa = 0, nsb = 0, n_q = 0, pid_q = 0;
    auto p_enter_range = [&]() {   // bounds of range pr were loaded one range ago (nsa, nsb)
        ps = nsa; psb = nsb;
        if (pr + G < NR) { nsa = range_start[pr + G]; nsb = range_start[pr + G + 1]; }
        if (ps < psb) {
            pk = seg_off[ps]; pend = seg_off[ps + 1];
            pend_nx = (ps + 2 <= n_seg) ? seg_off[ps + 2] : 0;
        }
    };
    auto p_next_seg = [&]() {
        ++ps; pk = pend; pend = pend_nx;
        pend_nx = (ps + 2 <= n_seg) ? seg_off[ps + 2] : 0;
    };
    auto p_seek = [&]() {          // settle on a short segment, or run out of ranges
        while (pr < NR) {
            if (ps >= psb) { pr += G; if (pr < NR) p_enter_range(); continue; }
            if (pend - pk > long_len) { p_next_seg(); continue; }
            break;
        }
    };
    if (pr < NR) {
        nsa = range_start[pr]; nsb = range_start[pr + 1];
        p_enter_range();
        p_seek();
        if (pr < NR) { n_q = perm[pk]; pid_q = partner[pk]; }
    }
    int wslot = 0, wgs = 0;        // ring slot / g-pack slot the producer fills next
    auto produce = [&]() {
        if (pr < NR) {
            stage_row_async<VEC, NV>(ring, wslot * 2 + 0, pinv, (int64_t)pid_q * pmul, D, lane);
            stage_row_async<VEC, NV>(ring, wslot * 2 + 1, penv, (int64_t)pid_q * pmul, D, lane);
            if (lane * 4 < GS) cp_async<16>(smem_addr(myG + wgs * 12 + lane * 4), a.gpack + (int64_t)n_q * GS + lane * 4);
            if (++pk == pend) { p_next_seg(); p_seek(); }
            if (pr < NR) { n_q = perm[pk]; pid_q = partner[pk]; }
        }
        cp_async_commit();
        if (++wslot == RING) wslot = 0;
        if (++wgs == RING + 1) wgs = 0;
    };
#pragma unroll
    for (int q = 0; q < RING - 1; ++q) produce();

    // ---- consumer: the same ranges, segment by segment ----
    auto request_own = [&](int64_t row_) {     // theta / m / v rows of one item row -> the six slots behind the ring
        stage_row_async<VEC, NV>(ring, RING * 2 + 0, a.own_inv_in, row_, D, lane);
        stage_row_async<VEC, NV>(ring, RING * 2 + 1, a.own_env_in, row_, D, lane);
        if (EPI == EPI_ADAM) {
            stage_row_async<VEC, NV>(ring, RING * 2 + 2, a.m_inv, row_, D, lane);
            stage_row_async<VEC, NV>(ring, RING * 2 + 3, a.m_env, row_, D, lane);
            stage_row_async<VEC, NV>(ring, RING * 2 + 4, a.v_inv, row_, D, lane);
            stage_row_async<VEC, NV>(ring, RING * 2 + 5, a.v_env, row_, D, lane);
        }
    };
    int rslot = 0, rgs = 0;
    int csa_n = 0, csb_n = 0;      // bounds of the consumer's next range
    if (g < NR) { csa_n = range_start[g]; csb_n = range_start[g + 1]; }
    for (int r = g; r < NR; r += G) {
        const int sa = csa_n, sb = csb_n;
        if (r + G < NR) { csa_n = range_start[r + G]; csb_n = range_start[r + G + 1]; }
        if (sa >= sb) continue;
        int cend = seg_off[sa], cend_nx = seg_off[sa + 1], row_nx = seg_row[sa];
        for (int cs = sa; cs < sb; ++cs) {
            const int beg = cend, end = cend_nx;
            const int64_t row = row_nx;
            cend = cend_nx;
            cend_nx = (cs + 2 <= n_seg) ? seg_off[cs + 2] : 0;
            if (cs + 1 < n_seg) row_nx = seg_row[cs + 1];
            int c0 = 0, c1 = 0;
            if (end - beg > long_len) {
                c0 = a.plan.seg_chunk[cs]; c1 = a.plan.seg_chunk[cs + 1];
                if (c1 - c0 > HOT_CHUNKS) continue;           // reduced by a whole CTA above
            }
            Row<VEC, NV> th_i, th_e, m_i, m_e, v_i, v_e;
            // own rows: global -> shared now (slots behind the ring; each lane its own slice), read after the loop.
            // The copies join the cp.async group of the next commit (the first produce() below).  Register loads
            // issued here instead would carry their scoreboard wait on the interaction loop's first branch, where
            // ncu found 37 % of the kernel's warp samples (DESIGN.md §3).
            request_own(row);
            Row<VEC, NV> gi, ge;
#pragma unroll
            for (int x = 0; x < NV * VEC; ++x) { gi.x[x] = 0.f; ge.x[x] = 0.f; }
            if (end - beg > long_len) {
                for (int c = c0; c < c1; ++c) {
                    Row<VEC, NV> pi, pe;
                    load_row<VEC, NV>(pi, a.chunk_part, (int64_t)c * 2, D, lane);
                    load_row<VEC, NV>(pe, a.chunk_part, (int64_t)c * 2 + 1, D, lane);
#pragma unroll
                    for (int x = 0; x < NV * VEC; ++x) { gi.x[x] += pi.x[x]; ge.x[x] += pe.x[x]; }
                }
                cp_async_commit();       // no produce() on this path: the own rows get a group of their own
                cp_async_wait<0>();
            } else {
                for (int k = beg; k < end; ++k) {
                    produce();
                    cp_async_wait<RING - 1>();
                    __syncwarp(gmask);   // the g-pack was copied by lanes 0..2 of this group
                    ring_consume<VEC, NV, KX>(myG + rgs * 12, ring, rslot, sE, sW, D, K, GS, lane, gi, ge);
                    if (++rslot == RING) rslot = 0;
                    if (++rgs == RING + 1) rgs = 0;
                }
                // The own rows travel in the group of the segment's FIRST produce(); len - 1 groups were committed after
                // it.  A loop of RING or more interactions has waited for it already (wait<RING - 1> after its last
                // produce); a shorter one allows exactly the younger groups to stay pending.
                {
                    const int len = end - beg;
                    if (len == 1) cp_async_wait<0>();
                    else if (len == 2) cp_async_wait<1>();
                    else if (len == 3) cp_async_wait<2>();
                    else if (len < RING) cp_async_wait<0>();      // any other loop shorter than the ring: wait for all
                }
            }
            read_staged_row<VEC, NV>(th_i, ring, RING * 2 + 0, D, lane);
            read_staged_row<VEC, NV>(th_e, ring, RING * 2 + 1, D, lane);
            if (EPI == EPI_ADAM) {
                read_staged_row<VEC, NV>(m_i, ring, RING * 2 + 2, D, lane);
                read_staged_row<VEC, NV>(m_e, ring, RING * 2 + 3, D, lane);
                read_staged_row<VEC, NV>(v_i, ring, RING * 2 + 4, D, lane);
                read_staged_row<VEC, NV>(v_e, ring, RING * 2 + 5, D, lane);
            }
            finish_row<VEC, NV, EPI>(a, row, (float)(end - beg), th_i, th_e, m_i, m_e, v_i, v_e, gi, ge, lane, D);
        }
    }
    cp_async_wait<0>();
}

// Dense Adam over the rows that received no gradient this step.
template <int VEC, int NV>
__global__ void __launch_bounds__(BLOCK) sweep_kernel(BwdSideArgs a) {
    const int D = a.D;
    const int lane = threadIdx.x & (GROUP - 1);
    const int64_t rows = a.plan.rows;
    const int64_t ngroups = (int64_t)gridDim.x * GROUPS_PER_BLOCK;
    const uint32_t* __restrict__ touched = a.plan.touched;
    const AdamScalars adam = with_dyn(a.adam, a.dyn);
    for (int64_t row = (int64_t)blockIdx.x * GROUPS_PER_BLOCK + (threadIdx.x >> 4); row < rows; row += ngroups) {
        if ((touched[row >> 5] >> (row & 31)) & 1u) continue;
        Row<VEC, NV> th_i, th_e, m_i, m_e, v_i, v_e;
        load_row<VEC, NV, true>(th_i, a.own_inv_in, row, D, lane);
        load_row<VEC, NV, true>(th_e, a.own_env_in, row, D, lane);
        load_row<VEC, NV, true>(m_i, a.m_inv, row, D, lane);
        load_row<VEC, NV, true>(m_e, a.m_env, row, D, lane);
        load_row<VEC, NV, true>(v_i, a.v_inv, row, D, lane);
        load_row<VEC, NV, true>(v_e, a.v_env, row, D, lane);
#pragma unroll
        for (int x = 0; x < NV * VEC; ++x) {
            adam_zero_step(th_i.x[x], m_i.x[x], v_i.x[x], adam, adam.step_size, adam.inv_bc2_sqrt);
            adam_zero_step(th_e.x[x], m_e.x[x], v_e.x[x], adam, adam.step_size, adam.inv_bc2_sqrt);
        }
        store_row<VEC, NV, true>(th_i, a.own_inv_out, row, D, lane);
        store_row<VEC, NV, true>(th_e, a.own_env_out, row, D, lane);
        store_row<VEC, NV, true>(m_i, a.m_inv, row, D, lane);
        store_row<VEC, NV, true>(m_e, a.m_env, row, D, lane);
        store_row<VEC, NV, true>(v_i, a.v_inv, row, D, lane);
        store_row<VEC, NV, true>(v_e, a.v_env, row, D, lane);
        if (a.grad_inv != nullptr) {
            Row<VEC, NV> z;
#pragma unroll
            for (int x = 0; x < NV * VEC; ++x) z.x[x] = 0.f;
            store_row<VEC, NV>(z, a.grad_inv, row, D, lane);
            store_row<VEC, NV>(z, a.grad_env, row, D, lane);
        }
    }
}

// Lazy mode: bring every row of this side that is behind up to step a.step (dense zero-gradient Adam steps
// replayed in registers with each step's own bias corrections), in place.  Run before anything outside the
// train step reads the table (EM re-assignment, evaluation, state_dict) -- or never, in dense mode.
template <int VEC, int NV>
__global__ void __launch_bounds__(BLOCK) flush_kernel(BwdSideArgs a) {
    const int D = a.D;
    const int lane = threadIdx.x & (GROUP - 1);
    const int64_t rows = a.plan.rows;
    const int64_t ngroups = (int64_t)gridDim.x * GROUPS_PER_BLOCK;
    const int step = a.dyn ? a.dyn->step : a.step;
    for (int64_t row = (int64_t)blockIdx.x * GROUPS_PER_BLOCK + (threadIdx.x >> 4); row < rows; row += ngroups) {
        const int last = a.last_step[row];
        if (last >= step) continue;
        Row<VEC, NV> th_i, th_e, m_i, m_e, v_i, v_e;
        load_row<VEC, NV, true>(th_i, a.own_inv_in, row, D, lane);
        load_row<VEC, NV, true>(th_e, a.own_env_in, row, D, lane);
        load_row<VEC, NV, true>(m_i, a.m_inv, row, D, lane);
        load_row<VEC, NV, true>(m_e, a.m_env, row, D, lane);
        load_row<VEC, NV, true>(v_i, a.v_inv, row, D, lane);
        load_row<VEC, NV, true>(v_e, a.v_env, row, D, lane);
        for (int j = last + 1; j <= step; ++j) {
            const float2 sc = a.sched[j];
#pragma unroll
            for (int x = 0; x < NV * VEC; ++x) {
                adam_zero_step(th_i.x[x], m_i.x[x], v_i.x[x], a.adam, sc.x, sc.y);
                adam_zero_step(th_e.x[x], m_e.x[x], v_e.x[x], a.adam, sc.x, sc.y);
            }
        }
        store_row<VEC, NV, true>(th_i, a.own_inv_out, row, D, lane);
        store_row<VEC, NV, true>(th_e, a.own_env_out, row, D, lane);
        store_row<VEC, NV, true>(m_i, a.m_inv, row, D, lane);
        store_row<VEC, NV, true>(m_e, a.m_env, row, D, lane);
        store_row<VEC, NV, true>(v_i, a.v_inv, row, D, lane);
        store_row<VEC, NV, true>(v_e, a.v_env, row, D, lane);
        if (lane == 0) a.last_step[row] = step;
    }
}

__global__ void sched_write_kernel(float2* sched, int step, float step_size, float inv_bc2_sqrt,
                                   const invpref_dyn* dyn) {
    if (dyn != nullptr) sched[dyn->step] = make_float2(dyn->step_size, dyn->inv_bc2_sqrt);
    else sched[step] = make_float2(step_size, inv_bc2_sqrt);
}

constexpr int TAIL_THREADS = 256;     // threads that run the epilogue
constexpr int TAIL_SLICES = 4;        // the column sums over the per-CTA partials are cut into this many row slices,
                                      // one per group of TAIL_THREADS threads (the sum was 30-40 us of a 0.38 ms step
                                      // on the dataset-scale configs with one slice)
constexpr int P_DB = 8, P_CNT = 16, P_DW = 24;

__device__ __forceinline__ double block_sum_double(double v, double* sbuf) {
    __syncthreads();
    if (threadIdx.x < TAIL_THREADS) sbuf[threadIdx.x] = v;
    __syncthreads();
    for (int s = TAIL_THREADS / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) sbuf[threadIdx.x] += sbuf[threadIdx.x + s];
        __syncthreads();
    }
    return sbuf[0];
}

__global__ void __launch_bounds__(TAIL_THREADS * TAIL_SLICES) tail_kernel(TailArgs a) {
    extern __shared__ double stot[];          // [P] totals, [TAIL_THREADS] scratch, [TAIL_SLICES][P] slice sums
    double* sbuf = stot + a.P;
    double* sslice = sbuf + TAIL_THREADS;
    const int K = a.K, D = a.D, KD = a.K * a.D;
    {
        // fixed-order column sums: slice q = rows [q * per, (q+1) * per) of the per-CTA partials, four interleaved
        // accumulators per thread (fixed assignment => deterministic), then the slices in order
        const int q = threadIdx.x / TAIL_THREADS, t = threadIdx.x % TAIL_THREADS;
        const int per = (a.n_partials + TAIL_SLICES - 1) / TAIL_SLICES;
        const int b0 = q * per, b1 = (b0 + per < a.n_partials) ? b0 + per : a.n_partials;
        for (int idx = t; idx < a.P; idx += TAIL_THREADS) {
            double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
            int b = b0;
            for (; b + 3 < b1; b += 4) {
                s0 += (double)a.partials[(int64_t)b * a.P + idx];
                s1 += (double)a.partials[(int64_t)(b + 1) * a.P + idx];
                s2 += (double)a.partials[(int64_t)(b + 2) * a.P + idx];
                s3 += (double)a.partials[(int64_t)(b + 3) * a.P + idx];
            }
            for (; b < b1; ++b) s0 += (double)a.partials[(int64_t)b * a.P + idx];
            sslice[q * a.P + idx] = (s0 + s1) + (s2 + s3);
        }
        __syncthreads();
        if (threadIdx.x < TAIL_THREADS) {
            for (int idx = t; idx < a.P; idx += TAIL_THREADS) {
                double s = 0.0;
#pragma unroll
                for (int qq = 0; qq < TAIL_SLICES; ++qq) s += sslice[qq * a.P + idx];
                stot[idx] = s;
            }
        }
    }
    // the epilogue below runs on the first TAIL_THREADS threads; the others only take part in the barriers
    const int tid = threadIdx.x < TAIL_THREADS ? (int)threadIdx.x : (1 << 30);
    __syncthreads();
    const double Bf = (double)a.B, Df = (double)D;
    const AdamScalars adam = with_dyn(a.adam, a.dyn);
    if (a.epi == EPI_ADAM || a.epi == EPI_EXPORT) {
        const bool do_adam = a.epi == EPI_ADAM;
        // classifier norms (models.py:210-217), only when it is regularised
        double w2 = 0.0, w1 = 0.0, b2 = 0.0, b1 = 0.0;
        if (!a.reg_only_embed) {
            for (int idx = tid; idx < KD; idx += TAIL_THREADS) {
                double x = a.W_in[idx];
                w2 += x * x; w1 += fabs(x);
            }
            if (tid < K) { double x = a.b_in[tid]; b2 = x * x; b1 = fabs(x); }
            w2 = block_sum_double(w2, sbuf);
            w1 = block_sum_double(w1, sbuf);
            b2 = block_sum_double(b2, sbuf);
            b1 = block_sum_double(b1, sbuf);
        }
        // env-embedding norms over the gathered rows (models.py:499-504) = sum_k count_k * |E_k|
        double e2 = 0.0, e1 = 0.0;
        if (a.reg_env_embed) {
            for (int idx = tid; idx < KD; idx += TAIL_THREADS) {
                const double x = a.E_in[idx], c = stot[P_CNT + idx / D];
                e2 += c * x * x; e1 += c * fabs(x);
            }
            e2 = block_sum_double(e2, sbuf);
            e1 = block_sum_double(e1, sbuf);
        }
        if (tid == 0 && a.loss_out != nullptr) {
            const float inv_loss = (float)(stot[0] / Bf);
            const float ea_loss = (float)(stot[1] / Bf);
            const float envs_loss = (float)(stot[2] / Bf);
            double L2 = stot[3] / (Bf * Df * 2.0), L1 = stot[4] / (Bf * Df * 2.0);
            if (!a.reg_only_embed) {
                L2 += w2 / (Df * K) + b2 / K;
                L1 += w1 / (Df * K) + b1 / K;
            }
            if (a.reg_env_embed) {
                L2 += e2 / (Bf * Df);
                L1 += e1 / (Bf * Df);
            }
            const float L2f = (float)L2, L1f = (float)L1;
            a.loss_out[0] = inv_loss;
            a.loss_out[1] = ea_loss;
            a.loss_out[2] = envs_loss;
            a.loss_out[3] = L2f;
            a.loss_out[4] = L1f;
            a.loss_out[5] = inv_loss * a.c_inv + ea_loss * a.c_ea + envs_loss * a.c_env + L2f * a.c_L2 + L1f * a.c_L1;
        }
        const float rW2 = 2.f * a.c_L2 / (float)(Df * K), rW1 = a.c_L1 / (float)(Df * K);
        const float rb2 = 2.f * a.c_L2 / (float)K, rb1 = a.c_L1 / (float)K;
        const float rE2 = (float)(2.0 * a.c_L2 / (Bf * Df)), rE1 = (float)(a.c_L1 / (Bf * Df));
        for (int idx = tid; idx < KD; idx += TAIL_THREADS) {
            const int k = idx / D;
            float w = a.W_in[idx], e = a.E_in[idx];
            float gW = (float)stot[P_DW + idx];
            float gE = (float)stot[P_DW + KD + idx];
            if (!a.reg_only_embed) gW += rW2 * w + rW1 * signf_(w);
            if (a.reg_env_embed) gE += (float)stot[P_CNT + k] * (rE2 * e + rE1 * signf_(e));
            if (a.gW) { a.gW[idx] = gW; a.gE[idx] = gE; }
            if (do_adam) {
                float m = a.mW[idx], v = a.vW[idx];
                adam_update(w, m, v, gW, adam);
                a.W_out[idx] = w; a.mW[idx] = m; a.vW[idx] = v;
                m = a.mE[idx]; v = a.vE[idx];
                adam_update(e, m, v, gE, adam);
                a.E_out[idx] = e; a.mE[idx] = m; a.vE[idx] = v;
            }
        }
        if (tid < K) {
            float bb = a.b_in[tid];
            float gb = (float)stot[P_DB + tid];
            if (!a.reg_only_embed) gb += rb2 * bb + rb1 * signf_(bb);
            if (a.gb) a.gb[tid] = gb;
            if (do_adam) {
                float m = a.mb[tid], v = a.vb[tid];
                adam_update(bb, m, v, gb, adam);
                a.b_out[tid] = bb; a.mb[tid] = m; a.vb[tid] = v;
            }
        }
    } else {
        for (int idx = tid; idx < KD; idx += TAIL_THREADS) {
            a.gW[idx] += (float)stot[P_DW + idx];
            a.gE[idx] += (float)stot[P_DW + KD + idx];
        }
        if (tid < K) a.gb[tid] += (float)stot[P_DB + tid];
    }
}

inline int grid_groups(int64_t n, int max_blocks) {
    int64_t need = (n + GROUPS_PER_BLOCK - 1) / GROUPS_PER_BLOCK;
    if (need < 1) need = 1;
    return (int)(need < max_blocks ? need : max_blocks);
}

}  // namespace

static size_t ring_smem(const Geometry& g) {   // E, W, g-pack slots, the ring of partner rows + six own-row slots
    return ((size_t)ring_align_up(((2 * g.K * g.D + 3) & ~3) + GROUPS_PER_BLOCK * (RING + 1) * 12) +
            (size_t)(RING * 2 + 6) * g.NV * g.VEC * BLOCK) * sizeof(float);
}

int launch_bwd_chunks(const Geometry& g, const BwdSideArgs& a, cudaStream_t stream) {
    const bool stash = a.stash != nullptr;
    if (g.NV * g.VEC <= 4) {
        const size_t smem = ring_smem(g);
        // chunk c goes to CTA c % grid: one CTA per SM first, up to three
        int64_t need = a.plan.max_chunks;
        const int grid = (int)(need < 1 ? 1 : (need < 148 * 3 ? need : 148 * 3));
#define LAUNCH(KERNEL)                                                                                           \
    do {                                                                                                         \
        INVPREF_SET_SMEM_ONCE(KERNEL, smem);                                                                     \
        KERNEL<<<grid, BLOCK, smem, stream>>>(a);                                                                \
    } while (0)
#define CALL_D(V, N, KX_, DX_)                                                                                   \
    do {                                                                                                         \
        if (stash) LAUNCH((bwd_chunks_ring_kernel<V, N, true, KX_, DX_>));                                       \
        else LAUNCH((bwd_chunks_ring_kernel<V, N, false, KX_, DX_>));                                            \
    } while (0)
#define CALL(V, N, KX_) CALL_D(V, N, KX_, GROUP * V * N)
        if (g.VEC == 4 && g.D == 40 && g.K == 2) { CALL_D(4, 1, 2, 40); }
        else if (g.VEC == 4 && g.D == 40 && g.K == 6) { CALL_D(4, 1, 6, 40); }
        else if (g.VEC == 4 && g.D == 40 && g.K == 5) { CALL_D(4, 1, 5, 40); }
        else if (g.VEC == 4 && g.D == GROUP * 4 && g.K == 2) { CALL(4, 1, 2); }
        else if (g.VEC == 4 && g.D == GROUP * 4 && g.K == 4) { CALL(4, 1, 4); }
        else if (g.VEC == 4 && g.D == GROUP * 4 && g.K == 6) { CALL(4, 1, 6); }
        else if (g.VEC == 4) { CALL(4, 1, 0); }
        else if (g.VEC == 2 && g.NV == 1) { CALL(2, 1, 0); }
        else if (g.VEC == 2) { CALL(2, 2, 0); }
        else { CALL(1, 4, 0); }
#undef CALL
#undef CALL_D
#undef LAUNCH
        count_launch();
        return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
    }
    // wider row slices: VEC = 4 with NV = 2 or 4
    size_t smem = (size_t)2 * g.K * g.D * sizeof(float);
    int grid = grid_groups(a.plan.max_chunks, 148 * 8);
#define CALL(V, N)                                                                                               \
    do {                                                                                                         \
        if (stash) bwd_chunks_kernel<V, N, true><<<grid, BLOCK, smem, stream>>>(a);                              \
        else bwd_chunks_kernel<V, N, false><<<grid, BLOCK, smem, stream>>>(a);                                   \
    } while (0)
    if (g.NV == 2) CALL(4, 2);
    else CALL(4, 4);
#undef CALL
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

static bool use_ring(const Geometry& g, int epi) {
    return g.NV * g.VEC <= 4 && (epi == EPI_ADAM || epi == EPI_EXPORT);
}

int launch_bwd_rows(const Geometry& g, const BwdSideArgs& a, int epi, cudaStream_t stream) {
    const bool stash = a.stash != nullptr;
    if (use_ring(g, epi)) {
        const size_t smem = ring_smem(g);
        const int grid = grid_groups(a.plan.max_seg, 148 * 3);   // three CTAs per SM are resident: one wave
        const int long_len = 2 * chunk_for(a.plan.B);
#define LAUNCH(KERNEL)                                                                                           \
    do {                                                                                                         \
        INVPREF_SET_SMEM_ONCE(KERNEL, smem);                                                                     \
        KERNEL<<<grid, BLOCK, smem, stream>>>(a, long_len);                                                      \
    } while (0)
#define CALL_D(V, N, KX_, DX_)                                                                                   \
    do {                                                                                                         \
        if (epi == EPI_ADAM && stash) LAUNCH((bwd_rows_ring_kernel<V, N, EPI_ADAM, true, KX_, DX_>));            \
        else if (epi == EPI_ADAM) LAUNCH((bwd_rows_ring_kernel<V, N, EPI_ADAM, false, KX_, DX_>));               \
        else if (stash) LAUNCH((bwd_rows_ring_kernel<V, N, EPI_EXPORT, true, KX_, DX_>));                        \
        else LAUNCH((bwd_rows_ring_kernel<V, N, EPI_EXPORT, false, KX_, DX_>));                                  \
    } while (0)
#define CALL(V, N, KX_) CALL_D(V, N, KX_, GROUP * V * N)
        if (g.VEC == 4 && g.D == 40 && g.K == 2) { CALL_D(4, 1, 2, 40); }          // exact: D = 40 (MovieLens / MIND)
        else if (g.VEC == 4 && g.D == 40 && g.K == 6) { CALL_D(4, 1, 6, 40); }
        else if (g.VEC == 4 && g.D == 40 && g.K == 5) { CALL_D(4, 1, 5, 40); }
        else if (g.VEC == 4 && g.D == GROUP * 4 && g.K == 2) { CALL(4, 1, 2); }    // exact: D = 64, K = KT
        else if (g.VEC == 4 && g.D == GROUP * 4 && g.K == 4) { CALL(4, 1, 4); }
        else if (g.VEC == 4 && g.D == GROUP * 4 && g.K == 6) { CALL(4, 1, 6); }
        else if (g.VEC == 4) { CALL(4, 1, 0); }
        else if (g.VEC == 2 && g.NV == 1) { CALL(2, 1, 0); }
        else if (g.VEC == 2) { CALL(2, 2, 0); }
        else { CALL(1, 4, 0); }
#undef CALL
#undef CALL_D
#undef LAUNCH
        count_launch();
        return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
    }
    size_t smem = (size_t)2 * g.K * g.D * sizeof(float);
    int grid = grid_groups(a.plan.max_seg, 148 * 8);
    if (epi == EPI_ADAM || epi == EPI_EXPORT) {   // wider row slices (use_ring): VEC = 4 with NV = 2 or 4
#define CALL(V, N)                                                                                               \
    do {                                                                                                         \
        if (epi == EPI_ADAM && stash) bwd_rows_kernel<V, N, EPI_ADAM, true><<<grid, BLOCK, smem, stream>>>(a);   \
        else if (epi == EPI_ADAM) bwd_rows_kernel<V, N, EPI_ADAM, false><<<grid, BLOCK, smem, stream>>>(a);      \
        else if (stash) bwd_rows_kernel<V, N, EPI_EXPORT, true><<<grid, BLOCK, smem, stream>>>(a);               \
        else bwd_rows_kernel<V, N, EPI_EXPORT, false><<<grid, BLOCK, smem, stream>>>(a);                         \
    } while (0)
        if (g.NV == 2) CALL(4, 2);
        else CALL(4, 4);
#undef CALL
    } else {
#define CALL(V, N) bwd_rows_kernel<V, N, EPI_ACCUM, false><<<grid, BLOCK, smem, stream>>>(a)
        INVPREF_DISPATCH_VN(g, CALL);
#undef CALL
    }
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_sweep(const Geometry& g, const BwdSideArgs& a, cudaStream_t stream) {
    int grid = grid_groups(a.plan.rows, 148 * 16);
#define CALL(V, N) sweep_kernel<V, N><<<grid, BLOCK, 0, stream>>>(a)
    INVPREF_DISPATCH_VN(g, CALL);
#undef CALL
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_flush(const Geometry& g, const BwdSideArgs& a, cudaStream_t stream) {
    int grid = grid_groups(a.plan.rows, 148 * 16);
#define CALL(V, N) flush_kernel<V, N><<<grid, BLOCK, 0, stream>>>(a)
    INVPREF_DISPATCH_VN(g, CALL);
#undef CALL
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_sched_write(float2* sched, int step, const AdamScalars& s, const invpref_dyn* dyn, cudaStream_t stream) {
    sched_write_kernel<<<1, 1, 0, stream>>>(sched, step, s.step_size, s.inv_bc2_sqrt, dyn);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_tail(const TailArgs& a, cudaStream_t stream) {
    size_t smem = (size_t)(a.P * (1 + TAIL_SLICES) + TAIL_THREADS) * sizeof(double);
    INVPREF_SET_SMEM_ONCE(tail_kernel, smem);
    tail_kernel<<<1, TAIL_THREADS * TAIL_SLICES, smem, stream>>>(a);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

}  // namespace invpref
