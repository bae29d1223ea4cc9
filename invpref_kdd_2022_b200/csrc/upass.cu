// Fused USER PASS: forward + losses + user-side segmented backward + Adam in one sweep over the batch in
// user-sorted order.
//
// Replaces fwd_train_kernel + bwd_rows_kernel(user side) of the unfused path (same reference code:
// models.py:448-467 / 307-326, 206-209; train.py:797-834; embedding_dense_backward; optim.Adam).
// One 16-lane group owns one user segment: the two user rows are loaded ONCE per segment (not once per
// interaction and again for Adam), the item rows once per interaction (not twice), and the per-interaction
// g-pack is only written (for the item pass), never read back here.  The classifier part of the user
// gradient is factored per segment:
//     Q_k[d] = sum_n g_logits[n,k] * c_n[d]        (c = item invariant row)
//     dUinv[u] += sum_n g_z1[n] c_n  +  (-alpha) * sum_k W[k,:] (.) Q_k          (gradient reversal)
//     dW[k,:]  += a_u (.) Q_k                                                     (not reversed)
// so W is applied once per segment instead of once per interaction.
//
//  upass_chunks_kernel : CHUNK-sized pieces of user segments longer than LONG_T (rare: hot users).
//  upass_rows_kernel   : every user segment; long ones only add up their chunk partials.
// Both write per-CTA partial sums (losses, norms, db, env counts, dW, dE) for tail_kernel; all sums run in
// a fixed order (no floating-point atomics).
//
// This file: the staged rows kernel and the launch logic; upass_regs.cu: the chunks kernel and the register-only
// rows kernel (D > 64); upass_common.cuh: the per-interaction arithmetic both share.
#include "upass_common.cuh"

namespace invpref {

namespace {

// ---------------------------------------------------------------------------------------------------------
// Staged rows kernel (row slices of <= 16 bytes per lane, i.e. D <= 64).
//
// ncu on the register-only kernel above (round 1): 30 % of the warp samples wait on the long scoreboard -- the
// (m, v, theta) rows of the segment behind a chain of dependent index loads, and the item rows of each
// interaction -- with only 16 warps per SM to hide it.  Here EVERYTHING a group will need is copied global ->
// shared with cp.async one step before it is used, so that no register (and no register scoreboard: ptxas made
// the inner loop's first branch wait for every load issued at the top of the segment, 35 % of the samples in
// an intermediate version that kept index loads in registers) is tied up while data is in flight:
//   * group A_{m+1}, requested at the top of segment m: the eight rows of the next segment (theta, m, v of both
//     user tables + the two item rows of its first interaction; every lane copies exactly the slice it later
//     reads), the scalars of its first interaction (env, score, weight) and the row's last_step, and the
//     32-byte descriptor {row, begin, end, perm/partner[begin], perm/partner[begin+1]} of the segment after it;
//   * group G_i, requested while interaction i is computed: the item rows and scalars of interaction i+1 and
//     the indices of interaction i+2.
// Row slices are read back by the lane that copied them; the few words shared by the group (descriptors,
// scalars, indices) after cp.async.wait_group + __syncwarp.  The arithmetic is the register-only kernel's,
// value for value.
constexpr int UP_SLOTS = 8;    // per stage: th_i, th_e, m_i, m_e, v_i, v_e, first item inv, first item env
// per-group metadata (32-bit words)
constexpr int UM_DESC = 0;     // [4][8]  descriptor ring, segment ordinal & 3 (ordinal o is read at the top of
                               //         segments o-1 and o; o+3 is requested during segment o: four slots)
constexpr int UM_SEGS = 32;    // [2][4]  {env, score, weight, last_step} of a segment's first interaction, by stage
constexpr int UM_ITS = 40;     // [2][4]  {env, score, weight, -} of interaction i, slot i & 1
constexpr int UM_ITI = 48;     // [2][2]  {perm, partner} of interaction i, slot i & 1
constexpr int UM_WORDS = 56;

// DX > 0: D = DX (64: every lane active; 40: the drivers' factor_num, lanes 0..9 active) and K = KT are compile-time
// constants (bounds guards fold away or become one lane predicate, row offsets are shifts and adds); DX = 0: any D, K.
template <int VEC, int NV, int KT, int EPI, bool LAZY, int DX>
__global__ void __launch_bounds__(BLOCK, 2) upass_rows_staged_kernel(UserPassArgs a, int long_len) {
    extern __shared__ __align__(128) float smem[];
    const int D = DX ? DX : a.side.D, K = DX ? KT : a.side.K, KD = K * D;
    const Smem s = carve_smem(smem, KD);
    float* ring = smem + ring_align_up((4 + 2 * GROUPS_PER_BLOCK) * KD + SB_WORDS);   // [2][8][NV][BLOCK][VEC]
    int32_t* meta = reinterpret_cast<int32_t*>(ring + (size_t)2 * UP_SLOTS * NV * VEC * BLOCK) +
                    (threadIdx.x >> 4) * UM_WORDS;                                          // this group's words
    Running st;
    stage(a, s, KD, st);
    const int lane = threadIdx.x & (GROUP - 1);
    const unsigned gmask = group_mask();
    float* myDE = s.sDE + (threadIdx.x >> 4) * KD;
    float* myDW = s.sDW + (threadIdx.x >> 4) * KD;
    const LossCfg cfg = {K, a.implicit, a.use_class_rw, a.use_rec_rw, a.c_inv, a.c_ea, a.c_env, a.invB};
    const int n_seg = a.side.plan.counters[0];
    const int ng = gridDim.x * GROUPS_PER_BLOCK;
    const int s0 = blockIdx.x * GROUPS_PER_BLOCK + (threadIdx.x >> 4);
    const int32_t* __restrict__ seg_desc = a.side.plan.seg_desc;
    const int32_t* __restrict__ perm = a.side.plan.perm;
    const int32_t* __restrict__ partner = a.side.plan.partner;
    const bool has_w = a.weights != nullptr;

    // descriptor of segment `seg` (ordinal `ord` of this group) -> ring slot ord & 3; lanes 0 and 1, 16 bytes each
    auto request_desc = [&](int ord, int seg) {
        if (seg < n_seg && lane < 2)
            cp_async<16>(smem_addr(meta + UM_DESC + (ord & 3) * 8 + lane * 4), seg_desc + (int64_t)seg * 8 + lane * 4);
    };
    // env / score / weight of interaction n -> dst[0..2] (lanes 8, 9, 10)
    auto request_scalars = [&](int32_t* dst, int n) {
        if (lane == 8) cp_async<4>(smem_addr(dst + 0), reinterpret_cast<const int32_t*>(a.envs + n));   // low word
        if (lane == 9) cp_async<4>(smem_addr(dst + 1), a.scores + n);
        if (lane == 10) {
            if (has_w) cp_async<4>(smem_addr(dst + 2), a.weights + n);
            else dst[2] = __float_as_int(1.f);
        }
    };
    // rows + first-interaction scalars + last_step of the segment described by dsc[] (shared memory) -> stage stg
    auto request_segment = [&](int stg, const int32_t* dsc) {
        const int row = dsc[0], n0 = dsc[3], p0 = dsc[4];
        stage_row_async<VEC, NV>(ring, stg * UP_SLOTS + 0, a.side.own_inv_in, row, D, lane);
        stage_row_async<VEC, NV>(ring, stg * UP_SLOTS + 1, a.side.own_env_in, row, D, lane);
        if (EPI == EPI_ADAM) {
            stage_row_async<VEC, NV>(ring, stg * UP_SLOTS + 2, a.side.m_inv, row, D, lane);
            stage_row_async<VEC, NV>(ring, stg * UP_SLOTS + 3, a.side.m_env, row, D, lane);
            stage_row_async<VEC, NV>(ring, stg * UP_SLOTS + 4, a.side.v_inv, row, D, lane);
            stage_row_async<VEC, NV>(ring, stg * UP_SLOTS + 5, a.side.v_env, row, D, lane);
        }
        stage_row_async<VEC, NV>(ring, stg * UP_SLOTS + 6, a.side.partner_inv, p0, D, lane);
        stage_row_async<VEC, NV>(ring, stg * UP_SLOTS + 7, a.side.partner_env, p0, D, lane);
        request_scalars(meta + UM_SEGS + stg * 4, n0);
        if (LAZY && lane == 11) cp_async<4>(smem_addr(meta + UM_SEGS + stg * 4 + 3), a.side.last_step + row);
    };

    // Segment of this group's ordinal o: round o of the segments, taken in SNAKE order (group g takes g in even
    // rounds and ng-1-g in odd ones).  Segments are sorted by row id and the ids by popularity (the hot users of a
    // batch come first), so with plain strides group 0 would collect the longest segment of every round: on the
    // dataset-scale configs, a few segments per group, the slowest group set the kernel time (18 % of the warp
    // samples sat at the final barrier).  Only the last round can be incomplete, so the first missing segment ends
    // a group's walk.
    auto seg_at = [&](int o) { return o * ng + ((o & 1) ? ng - 1 - s0 : s0); };

    // prologue: descriptors of the first two segments (the only exposed latency), then group A_0
    request_desc(0, seg_at(0));
    request_desc(1, seg_at(1));
    cp_async_commit();
    cp_async_wait<0>();
    __syncwarp(gmask);
    if (s0 < n_seg) request_segment(0, meta + UM_DESC);
    request_desc(2, seg_at(2));
    cp_async_commit();

    int ord = 0;
    for (int sgm = s0; sgm < n_seg; sgm = seg_at(++ord)) {
        const int stg = ord & 1;
        cp_async_wait<0>();      // A_ord: this segment's rows and scalars, the next segment's descriptor
        __syncwarp(gmask);
        // the next segment's stage (group A_{ord+1}), requested at the top of this one: deferring it until the second
        // interaction's item rows are requested measured slower (DESIGN.md §3, finding 2)
        auto request_next = [&]() {
            if (seg_at(ord + 1) < n_seg) request_segment(stg ^ 1, meta + UM_DESC + ((ord + 1) & 3) * 8);
            request_desc(ord + 3, seg_at(ord + 3));     // its slot held this group's previous segment
            cp_async_commit();       // A_{ord+1}
        };
        request_next();

        const int4 dA = *reinterpret_cast<const int4*>(meta + UM_DESC + (ord & 3) * 8);       // row, begin, end, n0
        const int4 dB = *reinterpret_cast<const int4*>(meta + UM_DESC + (ord & 3) * 8 + 4);   // p0, n1, p1, -
        const int4 sS = *reinterpret_cast<const int4*>(meta + UM_SEGS + stg * 4);
        const int64_t row = dA.x;
        const int beg = dA.y, end = dA.z;
        int n = dA.w, n_a = dB.y, it_a = dB.z;     // this interaction's batch position; indices of the next one
        int e = sS.x;
        float y = __int_as_float(sS.y), w = __int_as_float(sS.z);
        const int last = sS.w;
        const bool is_long = end - beg > long_len;

        Row<VEC, NV> ra, rue, gi, ge;
        Row<VEC, NV> m_i, m_e, v_i, v_e;
        read_staged_row<VEC, NV>(ra, ring, stg * UP_SLOTS + 0, D, lane);
        read_staged_row<VEC, NV>(rue, ring, stg * UP_SLOTS + 1, D, lane);
        if (LAZY) {
            // the row may be several steps behind: replay the skipped zero-gradient Adam steps in registers,
            // then stash the caught-up row (what every reader of this step must see) for the item pass
            read_staged_row<VEC, NV>(m_i, ring, stg * UP_SLOTS + 2, D, lane);
            read_staged_row<VEC, NV>(m_e, ring, stg * UP_SLOTS + 3, D, lane);
            read_staged_row<VEC, NV>(v_i, ring, stg * UP_SLOTS + 4, D, lane);
            read_staged_row<VEC, NV>(v_e, ring, stg * UP_SLOTS + 5, D, lane);
            replay_steps<VEC, NV>(a.side, last, __float_as_int(s.sB[SB_STEP]) - 1, ra, rue, m_i, m_e, v_i, v_e);
            store_row<VEC, NV>(ra, a.side.stash, (int64_t)sgm * 2, D, lane);
            store_row<VEC, NV>(rue, a.side.stash, (int64_t)sgm * 2 + 1, D, lane);
            // the caught-up moments go back to their (own) slots: no registers held over the interactions
            write_staged_row<VEC, NV>(m_i, ring, stg * UP_SLOTS + 2, D, lane);
            write_staged_row<VEC, NV>(m_e, ring, stg * UP_SLOTS + 3, D, lane);
            write_staged_row<VEC, NV>(v_i, ring, stg * UP_SLOTS + 4, D, lane);
            write_staged_row<VEC, NV>(v_e, ring, stg * UP_SLOTS + 5, D, lane);
        }
        if (is_long) {   // long segment: its forward + reduction ran in upass_chunks_kernel
            const int c0 = a.side.plan.seg_chunk[sgm], c1 = a.side.plan.seg_chunk[sgm + 1];
#pragma unroll
            for (int x = 0; x < NV * VEC; ++x) { gi.x[x] = 0.f; ge.x[x] = 0.f; }
            for (int c = c0; c < c1; ++c) {
                Row<VEC, NV> pi, pe;
                load_row<VEC, NV>(pi, a.side.chunk_part, (int64_t)c * 2, D, lane);
                load_row<VEC, NV>(pe, a.side.chunk_part, (int64_t)c * 2 + 1, D, lane);
#pragma unroll
                for (int x = 0; x < NV * VEC; ++x) { gi.x[x] += pi.x[x]; ge.x[x] += pe.x[x]; }
            }
        } else {
            float acc0[NV * VEC], Q[KT][NV * VEC];
#pragma unroll
            for (int x = 0; x < NV * VEC; ++x) {
                acc0[x] = 0.f; ge.x[x] = 0.f;
#pragma unroll
                for (int k = 0; k < KT; ++k) Q[k][x] = 0.f;
            }
            for (int k = beg; k < end; ++k) {
                const int par = (k - beg) & 1;
                if (k > beg) {
                    cp_async_wait<0>();      // G_{i-1}: this interaction's rows and scalars, the next one's indices
                    __syncwarp(gmask);
                    const int4 sI = *reinterpret_cast<const int4*>(meta + UM_ITS + par * 4);
                    e = sI.x; y = __int_as_float(sI.y); w = __int_as_float(sI.z);
                    if (k + 1 < end) {
                        const int2 ix = *reinterpret_cast<const int2*>(meta + UM_ITI + (par ^ 1) * 2);
                        n_a = ix.x; it_a = ix.y;
                    }
                }
                Row<VEC, NV> rc, rie;
                read_staged_row<VEC, NV>(rc, ring, stg * UP_SLOTS + 6, D, lane);
                read_staged_row<VEC, NV>(rie, ring, stg * UP_SLOTS + 7, D, lane);
                Inter<VEC, NV, KT> q;
                inter_dots<VEC, NV, KT>(a, s.sE, s.sW, ra, rue, rc, rie, e, lane, q, D, K);
                if (k + 1 < end) {
                    // the item slots are in registers (the sums below depend on every element): request
                    // interaction i+1's rows into them, its scalars, and the indices of interaction i+2
                    asm volatile("" ::"f"(q.z1), "f"(q.z2) : "memory");
                    stage_row_async<VEC, NV>(ring, stg * UP_SLOTS + 6, a.side.partner_inv, it_a, D, lane);
                    stage_row_async<VEC, NV>(ring, stg * UP_SLOTS + 7, a.side.partner_env, it_a, D, lane);
                    request_scalars(meta + UM_ITS + (par ^ 1) * 4, n_a);
                    if (k + 2 < end) {
                        if (lane == 12) cp_async<4>(smem_addr(meta + UM_ITI + par * 2 + 0), perm + k + 2);
                        if (lane == 13) cp_async<4>(smem_addr(meta + UM_ITI + par * 2 + 1), partner + k + 2);
                    }
                    cp_async_commit();       // G_i
                }
                inter_grads<VEC, NV, KT>(a, cfg, myDE, s.sB, rc, rie, q, n, e, y, w, lane, gmask, acc0, Q, ge.x, st, D, K);
                n = n_a;
            }
            finish_range<VEC, NV, KT>(a, s.sW, myDW, ra, lane, acc0, Q, gi, D, K, s.sB);
        }
        // the user rows' own L1/L2 terms (models.py:469-482): every occurrence in the batch counts
        const float cnt = (float)(end - beg);
        float sq = 0.f, ab = 0.f;
#pragma unroll
        for (int x = 0; x < NV * VEC; ++x) {
            sq += ra.x[x] * ra.x[x] + rue.x[x] * rue.x[x];
            ab += fabsf(ra.x[x]) + fabsf(rue.x[x]);
            gi.x[x] += cnt * (a.side.reg2 * ra.x[x] + mul_sign(a.side.reg1, ra.x[x]));
            ge.x[x] += cnt * (a.side.reg2 * rue.x[x] + mul_sign(a.side.reg1, rue.x[x]));
        }
        st.sq += cnt * sq;
        st.ab += cnt * ab;
        if (a.side.grad_inv != nullptr) {
            store_row<VEC, NV>(gi, a.side.grad_inv, row, D, lane);
            store_row<VEC, NV>(ge, a.side.grad_env, row, D, lane);
        }
        if (EPI == EPI_ADAM) {
            read_staged_row<VEC, NV>(m_i, ring, stg * UP_SLOTS + 2, D, lane);
            read_staged_row<VEC, NV>(m_e, ring, stg * UP_SLOTS + 3, D, lane);
            read_staged_row<VEC, NV>(v_i, ring, stg * UP_SLOTS + 4, D, lane);
            read_staged_row<VEC, NV>(v_e, ring, stg * UP_SLOTS + 5, D, lane);
            const AdamScalars adam = adam_from_smem(a.side.adam, s.sB);
#pragma unroll
            for (int x = 0; x < NV * VEC; ++x) {
                adam_update(ra.x[x], m_i.x[x], v_i.x[x], gi.x[x], adam);
                adam_update(rue.x[x], m_e.x[x], v_e.x[x], ge.x[x], adam);
            }
            store_row<VEC, NV>(ra, a.side.own_inv_out, row, D, lane);
            store_row<VEC, NV>(rue, a.side.own_env_out, row, D, lane);
            store_row<VEC, NV, true>(m_i, a.side.m_inv, row, D, lane);
            store_row<VEC, NV, true>(m_e, a.side.m_env, row, D, lane);
            store_row<VEC, NV, true>(v_i, a.side.v_inv, row, D, lane);
            store_row<VEC, NV, true>(v_e, a.side.v_env, row, D, lane);
            if (LAZY && lane == 0) a.side.last_step[row] = __float_as_int(s.sB[SB_STEP]);
        }
    }
    cp_async_wait<0>();
    write_partials(a, s, KD, st, blockIdx.x);
}

inline size_t upass_ring_bytes(const Geometry& g) {   // staged rows + per-group metadata
    return (size_t)2 * UP_SLOTS * g.NV * g.VEC * BLOCK * sizeof(float) + (size_t)GROUPS_PER_BLOCK * UM_WORDS * 4;
}
inline size_t upass_ring_offset(const Geometry& g) {   // bytes before the ring: the carve of upass_smem, 128-byte aligned
    return (size_t)ring_align_up((4 + 2 * GROUPS_PER_BLOCK) * g.K * g.D + SB_WORDS) * sizeof(float);
}

}  // namespace

bool upass_supported(const Geometry& g) { return upass_smem(g) <= 96 * 1024; }

static bool use_staged(const Geometry& g) {
    return g.NV * g.VEC <= 4 && upass_ring_offset(g) + upass_ring_bytes(g) <= 227 * 1024;
}

int upass_rows_grid(const Geometry& g, int64_t max_seg) {
    int64_t need = (max_seg + GROUPS_PER_BLOCK - 1) / GROUPS_PER_BLOCK;
    if (need < 1) need = 1;
    // staged kernel: two CTAs are resident per SM (registers, shared memory) -> one wave
    const int64_t cap = use_staged(g) ? 148 * 2 : 148 * 4;
    return (int)(need < cap ? need : cap);
}


int launch_upass_rows_regs(const Geometry& g, const UserPassArgs& a, int epi, int grid, cudaStream_t stream);   // upass_regs.cu

int launch_upass_rows(const Geometry& g, const UserPassArgs& a, int epi, int grid, cudaStream_t stream) {
    const bool lazy = a.side.last_step != nullptr;
    if (lazy && epi != EPI_ADAM) return INVPREF_ERR_BAD_ARG;
    if (use_staged(g)) {
        const size_t smem = upass_ring_offset(g) + upass_ring_bytes(g);
        const int long_len = 2 * chunk_for(a.side.plan.B);   // plan.cu: segments longer than this are chunked
#define LAUNCH(KERNEL)                                                                                           \
    do {                                                                                                         \
        INVPREF_SET_SMEM_ONCE(KERNEL, smem);                                                                     \
        KERNEL<<<grid, BLOCK, smem, stream>>>(a, long_len);                                                      \
    } while (0)
#define CALL_X(V, N, KT_, X)                                                                                     \
    do {                                                                                                         \
        if (lazy) LAUNCH((upass_rows_staged_kernel<V, N, KT_, EPI_ADAM, true, X>));                              \
        else if (epi == EPI_ADAM) LAUNCH((upass_rows_staged_kernel<V, N, KT_, EPI_ADAM, false, X>));             \
        else LAUNCH((upass_rows_staged_kernel<V, N, KT_, EPI_EXPORT, false, X>));                                \
    } while (0)
#define CALL(V, N, KT_) CALL_X(V, N, KT_, 0)
#define CALL_EXACT(V, N, KT_) CALL_X(V, N, KT_, 64)
#define CALL_EXACT40(V, N, KT_) CALL_X(V, N, KT_, 40)
        const int _k = g.KT;
        if (g.VEC == 4 && g.D == 64 && g.K == g.KT) { INVPREF_DISPATCH_K(4, 1, _k, CALL_EXACT); }
        else if (g.VEC == 4 && g.D == 40 && g.K == g.KT) { INVPREF_DISPATCH_K(4, 1, _k, CALL_EXACT40); }
        else if (g.VEC == 4 && g.D == 40 && g.K == 5) { CALL_EXACT40(4, 1, 5); }     // Yahoo!R3 drivers: K = 5
        else if (g.VEC == 4) { INVPREF_DISPATCH_K(4, 1, _k, CALL); }
        else if (g.VEC == 2 && g.NV == 1) { INVPREF_DISPATCH_K(2, 1, _k, CALL); }
        else if (g.VEC == 2) { INVPREF_DISPATCH_K(2, 2, _k, CALL); }
        else { INVPREF_DISPATCH_K(1, 4, _k, CALL); }
#undef CALL
#undef CALL_EXACT
#undef CALL_EXACT40
#undef CALL_X
#undef LAUNCH
        count_launch();
        return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
    }
    return launch_upass_rows_regs(g, a, epi, grid, stream);
}

}  // namespace invpref
