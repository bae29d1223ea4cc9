// Fused user pass, register-only kernels: upass_chunks_kernel (CHUNK-sized pieces of long user segments, for
// every geometry) and upass_rows_kernel (every user segment; used for row slices wider than 16 bytes per lane,
// i.e. D > 64).  See upass.cu for the staged rows kernel.
#include "upass_common.cuh"

namespace invpref {

namespace {

template <int VEC, int NV, int KT, bool LAZY>
__global__ void __launch_bounds__(BLOCK, 2) upass_chunks_kernel(UserPassArgs a, int cta_offset) {
    extern __shared__ float smem[];
    const int D = a.side.D, KD = a.side.K * a.side.D;
    const Smem s = carve_smem(smem, KD);
    Running st;
    stage(a, s, KD, st);
    const int lane = threadIdx.x & (GROUP - 1);
    const unsigned gmask = group_mask();
    float* myDE = s.sDE + (threadIdx.x >> 4) * KD;
    float* myDW = s.sDW + (threadIdx.x >> 4) * KD;
    const LossCfg cfg = {a.side.K, a.implicit, a.use_class_rw, a.use_rec_rw, a.c_inv, a.c_ea, a.c_env, a.invB};
    const int n_chunks = a.side.plan.counters[1];
    const int ngroups = gridDim.x * GROUPS_PER_BLOCK;
    for (int c = blockIdx.x * GROUPS_PER_BLOCK + (threadIdx.x >> 4); c < n_chunks; c += ngroups) {
        const int4 desc = reinterpret_cast<const int4*>(a.side.plan.chunk_desc)[c];
        const int64_t row = a.side.plan.seg_row[desc.x];
        Row<VEC, NV> ra, rue, gi, ge;
        load_row<VEC, NV>(ra, a.side.own_inv_in, row, D, lane);
        load_row<VEC, NV>(rue, a.side.own_env_in, row, D, lane);
        if (LAZY) {   // bring the row up to step-1 in registers (the rows kernel does the same and stores it)
            Row<VEC, NV> m_i, m_e, v_i, v_e;
            load_row<VEC, NV>(m_i, a.side.m_inv, row, D, lane);
            load_row<VEC, NV>(m_e, a.side.m_env, row, D, lane);
            load_row<VEC, NV>(v_i, a.side.v_inv, row, D, lane);
            load_row<VEC, NV>(v_e, a.side.v_env, row, D, lane);
            replay_steps<VEC, NV>(a.side, a.side.last_step[row], __float_as_int(s.sB[SB_STEP]) - 1, ra, rue, m_i, m_e, v_i, v_e);
        }
        float acc0[NV * VEC], Q[KT][NV * VEC];
#pragma unroll
        for (int x = 0; x < NV * VEC; ++x) {
            acc0[x] = 0.f; ge.x[x] = 0.f;
#pragma unroll
            for (int k = 0; k < KT; ++k) Q[k][x] = 0.f;
        }
        fused_range<VEC, NV, KT>(a, cfg, s.sE, s.sW, myDE, s.sB, ra, rue, desc.y, desc.z, lane, gmask, acc0, Q, ge.x, st);
        finish_range<VEC, NV, KT>(a, s.sW, myDW, ra, lane, acc0, Q, gi, D, a.side.K, s.sB);
        store_row<VEC, NV>(gi, a.side.chunk_part, (int64_t)c * 2, D, lane);
        store_row<VEC, NV>(ge, a.side.chunk_part, (int64_t)c * 2 + 1, D, lane);
    }
    write_partials(a, s, KD, st, cta_offset + blockIdx.x);
}

template <int VEC, int NV, int KT, int EPI, bool LAZY>
__global__ void __launch_bounds__(BLOCK, 2) upass_rows_kernel(UserPassArgs a) {
    extern __shared__ float smem[];
    const int D = a.side.D, KD = a.side.K * a.side.D;
    const Smem s = carve_smem(smem, KD);
    Running st;
    stage(a, s, KD, st);
    const int lane = threadIdx.x & (GROUP - 1);
    const unsigned gmask = group_mask();
    float* myDE = s.sDE + (threadIdx.x >> 4) * KD;
    float* myDW = s.sDW + (threadIdx.x >> 4) * KD;
    const LossCfg cfg = {a.side.K, a.implicit, a.use_class_rw, a.use_rec_rw, a.c_inv, a.c_ea, a.c_env, a.invB};
    const int n_seg = a.side.plan.counters[0];
    const int ngroups = gridDim.x * GROUPS_PER_BLOCK;
    const int s0 = blockIdx.x * GROUPS_PER_BLOCK + (threadIdx.x >> 4);
    // Software pipeline over this group's segments s0, s0+ng, ...: while segment j is processed, the rows
    // that segment j+1 touches first (its two user rows, their Adam state, the item rows and the per-sample
    // scalars of its first interaction) are requested into L2.  Every address a prefetch needs comes from a
    // register that was loaded one iteration earlier, so the (in-order) warp never waits on it.
    const int32_t* __restrict__ seg_row = a.side.plan.seg_row;
    const int32_t* __restrict__ seg_off = a.side.plan.seg_off;
    int row1 = 0, beg1 = 0, pid1 = 0, n1 = 0, row2 = 0, beg2 = 0;
    if (s0 + ngroups < n_seg) {
        row1 = seg_row[s0 + ngroups]; beg1 = seg_off[s0 + ngroups];
        pid1 = a.side.plan.partner[beg1]; n1 = a.side.plan.perm[beg1];
    }
    if (s0 + 2 * ngroups < n_seg) { row2 = seg_row[s0 + 2 * ngroups]; beg2 = seg_off[s0 + 2 * ngroups]; }
    for (int sgm = s0; sgm < n_seg; sgm += ngroups) {
        if (sgm + ngroups < n_seg) {
            prefetch_row(a.side.own_inv_in, row1, D, lane);
            prefetch_row(a.side.own_env_in, row1, D, lane);
            prefetch_row(a.side.partner_inv, pid1, D, lane);
            prefetch_row(a.side.partner_env, pid1, D, lane);
            if (EPI == EPI_ADAM) {
                prefetch_row(a.side.m_inv, row1, D, lane);
                prefetch_row(a.side.m_env, row1, D, lane);
                prefetch_row(a.side.v_inv, row1, D, lane);
                prefetch_row(a.side.v_env, row1, D, lane);
            }
            if (lane == 8) prefetch_l2(a.envs + n1);
            if (lane == 9) prefetch_l2(a.scores + n1);
            if (lane == 10 && a.weights != nullptr) prefetch_l2(a.weights + n1);
        }
        int pid2 = 0, n2 = 0, row3 = 0, beg3 = 0;
        if (sgm + 2 * ngroups < n_seg) { pid2 = a.side.plan.partner[beg2]; n2 = a.side.plan.perm[beg2]; }
        if (sgm + 3 * ngroups < n_seg) { row3 = seg_row[sgm + 3 * ngroups]; beg3 = seg_off[sgm + 3 * ngroups]; }
        const int64_t row = seg_row[sgm];
        const int beg = seg_off[sgm], end = seg_off[sgm + 1];
        const int c0 = a.side.plan.seg_chunk[sgm], c1 = a.side.plan.seg_chunk[sgm + 1];
        Row<VEC, NV> ra, rue, gi, ge;
        Row<VEC, NV> m_i, m_e, v_i, v_e;
        load_row<VEC, NV>(ra, a.side.own_inv_in, row, D, lane);
        load_row<VEC, NV>(rue, a.side.own_env_in, row, D, lane);
        if (LAZY) {
            // the row may be several steps behind: replay the skipped zero-gradient Adam steps in registers,
            // then stash the caught-up row (what every reader of this step must see) for the item pass
            load_row<VEC, NV, true>(m_i, a.side.m_inv, row, D, lane);
            load_row<VEC, NV, true>(m_e, a.side.m_env, row, D, lane);
            load_row<VEC, NV, true>(v_i, a.side.v_inv, row, D, lane);
            load_row<VEC, NV, true>(v_e, a.side.v_env, row, D, lane);
            replay_steps<VEC, NV>(a.side, a.side.last_step[row], __float_as_int(s.sB[SB_STEP]) - 1, ra, rue, m_i, m_e, v_i, v_e);
            store_row<VEC, NV>(ra, a.side.stash, (int64_t)sgm * 2, D, lane);
            store_row<VEC, NV>(rue, a.side.stash, (int64_t)sgm * 2 + 1, D, lane);
        }
        if (c1 > c0) {   // long segment: its forward + reduction ran in upass_chunks_kernel
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
            fused_range<VEC, NV, KT>(a, cfg, s.sE, s.sW, myDE, s.sB, ra, rue, beg, end, lane, gmask, acc0, Q, ge.x, st);
            finish_range<VEC, NV, KT>(a, s.sW, myDW, ra, lane, acc0, Q, gi, D, a.side.K, s.sB);
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
            if (!LAZY) {
                load_row<VEC, NV, true>(m_i, a.side.m_inv, row, D, lane);
                load_row<VEC, NV, true>(m_e, a.side.m_env, row, D, lane);
                load_row<VEC, NV, true>(v_i, a.side.v_inv, row, D, lane);
                load_row<VEC, NV, true>(v_e, a.side.v_env, row, D, lane);
            }
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
        row1 = row2; beg1 = beg2; pid1 = pid2; n1 = n2;
        row2 = row3; beg2 = beg3;
    }
    write_partials(a, s, KD, st, blockIdx.x);
}

}  // namespace

int launch_upass_chunks(const Geometry& g, const UserPassArgs& a, int cta_offset, cudaStream_t stream) {
    const size_t smem = upass_smem(g);
    const bool lazy = a.side.last_step != nullptr;
#define LAUNCH(KERNEL)                                                                                           \
    do {                                                                                                         \
        INVPREF_SET_SMEM_ONCE(KERNEL, smem);                                                                     \
        KERNEL<<<UPASS_CHUNK_CTAS, BLOCK, smem, stream>>>(a, cta_offset);                                        \
    } while (0)
#define CALL(V, N, KT_)                                                                                          \
    do {                                                                                                         \
        if (lazy) LAUNCH((upass_chunks_kernel<V, N, KT_, true>));                                                \
        else LAUNCH((upass_chunks_kernel<V, N, KT_, false>));                                                    \
    } while (0)
    INVPREF_DISPATCH_GEOM(g, CALL);
#undef CALL
#undef LAUNCH
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_upass_rows_regs(const Geometry& g, const UserPassArgs& a, int epi, int grid, cudaStream_t stream) {
    const bool lazy = a.side.last_step != nullptr;
    const size_t smem = upass_smem(g);
#define LAUNCH(KERNEL)                                                                                           \
    do {                                                                                                         \
        INVPREF_SET_SMEM_ONCE(KERNEL, smem);                                                                     \
        KERNEL<<<grid, BLOCK, smem, stream>>>(a);                                                                \
    } while (0)
#define CALL(V, N, KT_)                                                                                          \
    do {                                                                                                         \
        if (lazy) LAUNCH((upass_rows_kernel<V, N, KT_, EPI_ADAM, true>));                                        \
        else if (epi == EPI_ADAM) LAUNCH((upass_rows_kernel<V, N, KT_, EPI_ADAM, false>));                       \
        else LAUNCH((upass_rows_kernel<V, N, KT_, EPI_EXPORT, false>));                                          \
    } while (0)
    // every narrower row slice takes the staged kernel (use_staged, upass.cu): only VEC = 4 with NV = 2 or 4 get here
    if (g.NV == 2) INVPREF_DISPATCH_K(4, 2, g.KT, CALL);
    else INVPREF_DISPATCH_K(4, 4, g.KT, CALL);
#undef CALL
#undef LAUNCH
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

}  // namespace invpref
