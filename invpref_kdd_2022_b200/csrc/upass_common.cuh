// Shared device helpers of the fused user pass (upass.cu: staged rows kernel; upass_regs.cu: chunks kernel and the
// register-only rows kernel).  Everything lives in an anonymous namespace: each translation unit gets its own copy.
#pragma once

#include "common.cuh"
#include "kernels.h"
#include "lossmath.cuh"

namespace invpref {

namespace {

constexpr int P_DB = 8, P_CNT = 16, P_DW = 24;
// sB: the classifier bias [INVPREF_MAX_ENVS], then the step-dependent scalars (launch arguments, or the device record
// invpref_hyper.dyn for CUDA-graph replay), read from shared memory where they are used so that no register holds them
constexpr int SB_STEP_SIZE = INVPREF_MAX_ENVS, SB_INV_BC2 = INVPREF_MAX_ENVS + 1, SB_NEG_ALPHA = INVPREF_MAX_ENVS + 2,
              SB_STEP = INVPREF_MAX_ENVS + 3, SB_WORDS = INVPREF_MAX_ENVS + 4;

// Per-lane sums that persist over all segments a group handles.  The eleven-plus scalar sums (three losses,
// db[K], env counts[K]) are spread over the lanes of the group, one register each, instead of every lane
// carrying all of them: lane 0..2 -> losses, lane 3..3+K-1 -> db[k] (stat1); lane k -> count of env k (stat2).
struct Running {
    float stat1, stat2;
    float sq, ab;         // sum x^2 / |x| over the gathered rows (this lane's dims)
};

// One interaction, part 1: dot products against the user rows -> logits and scores (unreduced per-lane sums).
template <int VEC, int NV, int KT>
struct Inter {
    float z1, z2, sq, ab;
    float lg[KT], t[NV * VEC], ee[NV * VEC];
};

template <int VEC, int NV, int KT>
__device__ __forceinline__ void inter_dots(const UserPassArgs& a, const float* __restrict__ sE,
                                           const float* __restrict__ sW, const Row<VEC, NV>& ra,
                                           const Row<VEC, NV>& rue, const Row<VEC, NV>& rc, const Row<VEC, NV>& rie,
                                           int e, int lane, Inter<VEC, NV, KT>& q, int D, int K) {
    q.z1 = 0.f; q.z2 = 0.f; q.sq = 0.f; q.ab = 0.f;
#pragma unroll
    for (int kk = 0; kk < KT; ++kk) q.lg[kk] = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int d0 = dim_of<VEC>(lane, j);
        if (d0 < D) {
            ldv<VEC>(sE + e * D + d0, &q.ee[j * VEC]);
            float p[VEC], wk[VEC];
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                const int x = j * VEC + v;
                p[v] = ra.x[x] * rc.x[x];
                q.t[x] = rue.x[x] * rie.x[x];
                q.z1 += p[v];
                q.z2 += q.t[x] * q.ee[x];
                q.sq += rc.x[x] * rc.x[x] + rie.x[x] * rie.x[x];
                q.ab += fabsf(rc.x[x]) + fabsf(rie.x[x]);
            }
#pragma unroll
            for (int kk = 0; kk < KT; ++kk) {
                if (kk < K) {
                    ldv<VEC>(sW + kk * D + d0, wk);
#pragma unroll
                    for (int v = 0; v < VEC; ++v) q.lg[kk] += wk[v] * p[v];
                }
            }
        } else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) { q.t[j * VEC + v] = 0.f; q.ee[j * VEC + v] = 0.f; }
        }
    }
}

// One interaction, part 2: group reductions, losses and their backward scalars, the user-side gradient
// pieces, dE, the running sums, and the g-pack of interaction n for the item pass.
template <int VEC, int NV, int KT>
__device__ __forceinline__ void inter_grads(const UserPassArgs& a, const LossCfg& cfg, float* __restrict__ myDE,
                                            const float* __restrict__ sB, const Row<VEC, NV>& rc,
                                            const Row<VEC, NV>& rie, Inter<VEC, NV, KT>& q, int n, int e, float y,
                                            float w, int lane, unsigned gmask, float (&acc0)[NV * VEC],
                                            float (&Q)[KT][NV * VEC], float (&acc_env)[NV * VEC], Running& st,
                                            int D, int K) {
    const float z1 = group_sum(q.z1, gmask);
    const float z2 = group_sum(q.z2, gmask);
    float lg[KT];
#pragma unroll
    for (int kk = 0; kk < KT; ++kk) lg[kk] = (kk < K) ? group_sum(q.lg[kk], gmask) + sB[kk] : -INFINITY;

    float g_z1, g_z2, gl[KT], lw[3];
    loss_grads<KT, true>(cfg, z1, z2, lg, y, w, e, g_z1, g_z2, gl, lw, lane, gmask);
    st.sq += q.sq;
    st.ab += q.ab;
    {
        float v1 = (lane == 0) ? lw[0] : ((lane == 1) ? lw[1] : ((lane == 2) ? lw[2] : 0.f));
#pragma unroll
        for (int kk = 0; kk < KT; ++kk) v1 = (lane == 3 + kk) ? gl[kk] : v1;
        st.stat1 += v1;
        st.stat2 += (lane == e) ? 1.f : 0.f;
    }
    // user-side gradient pieces and dE[e] += g_z2 * ue*ie (this group's shared-memory slice)
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int d0 = dim_of<VEC>(lane, j);
        if (d0 < D) {
            float de[VEC];
            ldv<VEC>(myDE + e * D + d0, de);
#pragma unroll
            for (int v = 0; v < VEC; ++v) {
                const int x = j * VEC + v;
                acc0[x] += g_z1 * rc.x[x];
                acc_env[x] += g_z2 * rie.x[x] * q.ee[x];
                de[v] += g_z2 * q.t[x];
#pragma unroll
                for (int kk = 0; kk < KT; ++kk) Q[kk][x] += gl[kk] * rc.x[x];
            }
            stv<VEC>(myDE + e * D + d0, de);
        }
    }
    if (lane == 0) {   // g-pack for the item pass: g_z1, g_z2, env, -alpha * g_logits
        const int GS = (K <= 5) ? 8 : 12;   // make_geometry
        float* gp = a.gpack_out + (int64_t)n * GS;
        float out[12];
        out[0] = g_z1;
        out[1] = g_z2;
        out[2] = __int_as_float(e);
        const float neg_alpha = sB[SB_NEG_ALPHA];
#pragma unroll
        for (int kk = 0; kk < 9; ++kk) out[3 + kk] = (kk < KT) ? neg_alpha * gl[kk < KT ? kk : 0] : 0.f;
        *reinterpret_cast<float4*>(gp) = make_float4(out[0], out[1], out[2], out[3]);
        *reinterpret_cast<float4*>(gp + 4) = make_float4(out[4], out[5], out[6], out[7]);
        if (KT > 5 && GS > 8)
            *reinterpret_cast<float4*>(gp + 8) = make_float4(out[8], out[9], out[10], out[11]);
    }
}

// Interactions [beg, end) of one user segment, item rows loaded straight from global memory (chunks kernel and
// the unstaged rows kernel).
template <int VEC, int NV, int KT>
__device__ __forceinline__ void fused_range(const UserPassArgs& a, const LossCfg& cfg, const float* __restrict__ sE,
                                            const float* __restrict__ sW, float* __restrict__ myDE,
                                            const float* __restrict__ sB, const Row<VEC, NV>& ra, const Row<VEC, NV>& rue,
                                            int beg, int end, int lane, unsigned gmask, float (&acc0)[NV * VEC],
                                            float (&Q)[KT][NV * VEC], float (&acc_env)[NV * VEC], Running& st) {
    const int D = a.side.D;
    const int32_t* __restrict__ perm = a.side.plan.perm;
    const int32_t* __restrict__ partner = a.side.plan.partner;
    for (int k = beg; k < end; ++k) {
        const int n = perm[k];
        const int it = partner[k];
        const int e = (int)a.envs[n];
        const float y = a.scores[n];
        const float w = (a.weights != nullptr) ? a.weights[n] : 1.f;
        Row<VEC, NV> rc, rie;
        load_row<VEC, NV>(rc, a.side.partner_inv, it, D, lane);
        load_row<VEC, NV>(rie, a.side.partner_env, it, D, lane);
        Inter<VEC, NV, KT> q;
        inter_dots<VEC, NV, KT>(a, sE, sW, ra, rue, rc, rie, e, lane, q, D, a.side.K);
        inter_grads<VEC, NV, KT>(a, cfg, myDE, sB, rc, rie, q, n, e, y, w, lane, gmask, acc0, Q, acc_env, st, D, a.side.K);
    }
}

// gi = acc0 + (-alpha) sum_k W_k (.) Q_k ;  dW_k += a (.) Q_k  (this group's shared-memory slice)
template <int VEC, int NV, int KT>
__device__ __forceinline__ void finish_range(const UserPassArgs& a, const float* __restrict__ sW,
                                             float* __restrict__ myDW, const Row<VEC, NV>& ra, int lane,
                                             const float (&acc0)[NV * VEC], const float (&Q)[KT][NV * VEC],
                                             Row<VEC, NV>& gi, int D, int K, const float* __restrict__ sB) {
    const float neg_alpha = sB[SB_NEG_ALPHA];
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int d0 = dim_of<VEC>(lane, j);
        if (d0 < D) {
#pragma unroll
            for (int v = 0; v < VEC; ++v) gi.x[j * VEC + v] = acc0[j * VEC + v];
#pragma unroll
            for (int kk = 0; kk < KT; ++kk) {
                if (kk < K) {
                    float wk[VEC], dw[VEC];
                    ldv<VEC>(sW + kk * D + d0, wk);
                    ldv<VEC>(myDW + kk * D + d0, dw);
#pragma unroll
                    for (int v = 0; v < VEC; ++v) {
                        const int x = j * VEC + v;
                        gi.x[x] += neg_alpha * wk[v] * Q[kk][x];
                        dw[v] += ra.x[x] * Q[kk][x];
                    }
                    stv<VEC>(myDW + kk * D + d0, dw);
                }
            }
        } else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) gi.x[j * VEC + v] = 0.f;
        }
    }
}

// Lazy mode: replay the zero-gradient Adam steps last+1 .. upto (inclusive) of one user row in registers.
template <int VEC, int NV>
__device__ __forceinline__ void replay_steps(const BwdSideArgs& sd, int last, int upto, Row<VEC, NV>& th_i,
                                             Row<VEC, NV>& th_e, Row<VEC, NV>& m_i, Row<VEC, NV>& m_e,
                                             Row<VEC, NV>& v_i, Row<VEC, NV>& v_e) {
    for (int j = last + 1; j <= upto; ++j) {
        const float2 sc = sd.sched[j];
#pragma unroll
        for (int x = 0; x < NV * VEC; ++x) {
            adam_zero_step(th_i.x[x], m_i.x[x], v_i.x[x], sd.adam, sc.x, sc.y);
            adam_zero_step(th_e.x[x], m_e.x[x], v_e.x[x], sd.adam, sc.x, sc.y);
        }
    }
}

struct Smem {
    float *sE, *sW, *sRed, *sDE, *sDW, *sB;
};

__device__ __forceinline__ AdamScalars adam_from_smem(AdamScalars s, const float* sB) {
    s.step_size = sB[SB_STEP_SIZE];
    s.inv_bc2_sqrt = sB[SB_INV_BC2];
    return s;
}

__device__ __forceinline__ Smem carve_smem(float* smem, int KD) {
    Smem s;
    s.sE = smem;
    s.sW = smem + KD;
    s.sRed = smem + 2 * KD;
    s.sDE = smem + 4 * KD;
    s.sDW = smem + (4 + GROUPS_PER_BLOCK) * KD;
    s.sB = smem + (4 + 2 * GROUPS_PER_BLOCK) * KD;
    return s;
}

__device__ __forceinline__ void stage(const UserPassArgs& a, const Smem& s, int KD, Running& st) {
    for (int t = threadIdx.x; t < KD; t += BLOCK) { s.sE[t] = a.side.E[t]; s.sW[t] = a.side.W[t]; }
    for (int t = threadIdx.x; t < 2 * GROUPS_PER_BLOCK * KD; t += BLOCK) s.sDE[t] = 0.f;   // sDE and sDW
    if (threadIdx.x < INVPREF_MAX_ENVS) s.sB[threadIdx.x] = ((int)threadIdx.x < a.side.K) ? a.b[threadIdx.x] : 0.f;
    if (threadIdx.x == 32) {
        const invpref_dyn* dyn = a.side.dyn;
        s.sB[SB_STEP_SIZE] = dyn ? dyn->step_size : a.side.adam.step_size;
        s.sB[SB_INV_BC2] = dyn ? dyn->inv_bc2_sqrt : a.side.adam.inv_bc2_sqrt;
        s.sB[SB_NEG_ALPHA] = dyn ? dyn->neg_alpha : a.neg_alpha;
        s.sB[SB_STEP] = __int_as_float(dyn ? dyn->step : a.side.step);
    }
    __syncthreads();
    st.stat1 = st.stat2 = st.sq = st.ab = 0.f;
}

// CTA reduction in a fixed order, then this CTA's partial vector
__device__ __forceinline__ void write_partials(const UserPassArgs& a, const Smem& s, int KD, const Running& st,
                                               int cta) {
    __syncthreads();
    for (int t = threadIdx.x; t < KD; t += BLOCK) {
        float w = 0.f, e = 0.f;
        for (int g = 0; g < GROUPS_PER_BLOCK; ++g) { w += s.sDW[g * KD + t]; e += s.sDE[g * KD + t]; }
        s.sRed[t] = w;
        s.sRed[KD + t] = e;
    }
    __shared__ float sScal[BLOCK / 32][24];
    const int glane = threadIdx.x & (GROUP - 1);
    float sc[24];
    sc[0] = (glane == 0) ? st.stat1 : 0.f;
    sc[1] = (glane == 1) ? st.stat1 : 0.f;
    sc[2] = (glane == 2) ? st.stat1 : 0.f;
    sc[3] = st.sq; sc[4] = st.ab; sc[5] = sc[6] = sc[7] = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        sc[8 + k] = (glane == 3 + k) ? st.stat1 : 0.f;
        sc[16 + k] = (glane == k) ? st.stat2 : 0.f;
    }
#pragma unroll
    for (int q = 0; q < 24; ++q) sc[q] = warp_sum(sc[q]);
    const int warp = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
#pragma unroll
        for (int q = 0; q < 24; ++q) sScal[warp][q] = sc[q];
    }
    __syncthreads();
    float* out = a.partials + (int64_t)cta * a.P;
    if (threadIdx.x < 24) {
        float v = 0.f;
        for (int w = 0; w < BLOCK / 32; ++w) v += sScal[w][threadIdx.x];
        out[threadIdx.x] = v;
    }
    for (int t = threadIdx.x; t < 2 * KD; t += BLOCK) out[P_DW + t] = s.sRed[t];
}


inline size_t upass_smem(const Geometry& g) {
    return ((size_t)(4 + 2 * GROUPS_PER_BLOCK) * g.K * g.D + SB_WORDS) * sizeof(float);
}

}  // namespace

}  // namespace invpref
