// EM environment re-assignment (train.py:846-879, 912-957).
//
// The reference runs K full forwards (K x the gather traffic, K wasted classifier passes), cats the
// K distance columns, adds the tie-break eps and argmins.  Here each sample's four rows are gathered
// ONCE, the K env-aware scores are formed in registers against E (staged in shared memory), and the
// first-min argmin, the env histogram (train.py:949) and the diff count (train.py:933-934) come out of
// the same pass.
//
// ncu on the first version (round 1): 57 % of the warp samples waited on the long scoreboard (ids -> rows ->
// perm_idx -> eps chains), 64-bit shared atomics were CAS loops.  Now the four rows of a sample are copied
// global -> shared with cp.async two iterations before they are read (no register held, each lane copies the
// slice it reads back: wait_group only, no barrier), ids (low words) are loaded two iterations before that, the
// per-sample scalars one iteration ahead into one lane-distributed register, this lane's slice of E lives in
// registers, the K! x K tie-break table in shared memory (K <= 6), the K env scores come out of one scattered
// reduction and a (distance, k) butterfly takes the first minimum, and histogram / diff counts are per-group
// registers until the end.  5.5 G samples/s = 0.90 of the measured HBM peak at C5.
#include "common.cuh"
#include "kernels.h"

namespace invpref {

namespace {

// Ring depth of the staged row gathers: a sample's four rows are requested (cp.async, no registers held)
// cl_stages - 1 iterations before they are read.  The kernel and the launcher's shared-memory size both use it.
__host__ __device__ constexpr int cl_stages(int vec, int nv) { return (vec * nv <= 8) ? 3 : 2; }

// DX > 0: D = DX (64 or 40) and K = KT are compile-time constants (bounds guards fold away, row offsets are shifts and
// adds); DX = 0: any D, K.
//
// SORTED: the same re-assignment over a USER-SORTED view of the dataset (ClusterArgs.perm / users32 / items32 / scores
// hold the samples in stable user order; perm[k] = original position).  A group walks a CONTIGUOUS run of sorted
// positions, so consecutive samples share their user: the two user rows are requested again but come out of L2, not
// HBM -- with N / U samples per user (10 at the bench's 96 M samples, 100 at N = 10^9) the DRAM bytes per sample drop
// from 16 D + 44 to about 8 D + 8 D U / N + 130 (ids and scores are read sequentially from the sorted copies; the
// tie-break index, the old environment and the new environment go through perm: three scattered sectors).  Same
// per-sample arithmetic as the plain order, value for value.
template <int VEC, int NV, int KT, int DX, bool SORTED>
__device__ __forceinline__ void cluster_body(const ClusterArgs& a, int eps_rows_smem) {
    extern __shared__ __align__(128) float smem[];
    constexpr int RV = VEC * NV, ST = cl_stages(VEC, NV);
    constexpr bool E_REG = KT * RV <= 32;      // this lane's slice of E lives in registers for the whole kernel
    const int D = DX ? DX : a.D, K = DX ? KT : a.K, KD = K * D;
    float* sE = smem;                                        // [K*D]
    float* sEps = smem + ((KD + 3) & ~3);                    // [eps_rows_smem * K]
    float* ring = smem + ring_align_up(((KD + 3) & ~3) + ((eps_rows_smem * K + 3) & ~3));   // [ST][4 rows][NV][BLOCK][VEC]
    __shared__ unsigned long long sHist[INVPREF_MAX_ENVS + 1];   // [K] histogram, [8] diff
    const int tid = threadIdx.x, lane = tid & (GROUP - 1);
    const unsigned gmask = group_mask();
    for (int t = tid; t < KD; t += BLOCK) sE[t] = a.E[t];
    for (int t = tid; t < eps_rows_smem * K; t += BLOCK) sEps[t] = a.eps_table[t];
    if (tid <= INVPREF_MAX_ENVS) sHist[tid] = 0ull;
    __syncthreads();
    float eR[E_REG ? KT : 1][RV];
    if (E_REG) {
#pragma unroll
        for (int k = 0; k < KT; ++k)
#pragma unroll
            for (int j = 0; j < NV; ++j)
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    const int d = dim_of<VEC>(lane, j) + v;
                    eR[E_REG ? k : 0][j * VEC + v] = (k < K && d < D) ? sE[k * D + d] : 0.f;
                }
    }

    // plain: group g takes samples g, g + n_groups, ... up to B.  SORTED: group g walks sorted positions
    // [g * per, (g + 1) * per), stride 1; end = one past the last.  The plain order reads a.B itself where it
    // compares (a register copy of it costs some plain instances two registers).
    const int64_t n_groups = (int64_t)gridDim.x * GROUPS_PER_BLOCK;
    const int64_t per = SORTED ? (a.B + n_groups - 1) / n_groups : 1;
    const int64_t n0 = ((int64_t)blockIdx.x * GROUPS_PER_BLOCK + (tid >> 4)) * per;
    const int64_t run_end = (n0 + per < a.B) ? n0 + per : a.B;
    const int64_t& end = SORTED ? run_end : a.B;
    const int64_t stride = SORTED ? 1 : n_groups;
    auto issue = [&](int slot, int64_t u, int64_t it) {
        stage_row_async<VEC, NV>(ring, slot * 4 + 0, a.Uinv, u, D, lane);
        stage_row_async<VEC, NV>(ring, slot * 4 + 1, a.Iinv, it, D, lane);
        stage_row_async<VEC, NV>(ring, slot * 4 + 2, a.Uenv, u, D, lane);
        stage_row_async<VEC, NV>(ring, slot * 4 + 3, a.Ienv, it, D, lane);
    };
    // ids are below 2^31 (make_geometry): plain loads only the low word of each int64, SORTED the int32 sorted copies.
    // They run TWO iterations ahead of the row requests (one was not enough: the request stalled on its own ids, ncu
    // round 1).
    constexpr int IW = SORTED ? 1 : 2;     // id word stride
    const int32_t* __restrict__ users_lo = SORTED ? a.users32 : reinterpret_cast<const int32_t*>(a.users);
    const int32_t* __restrict__ items_lo = SORTED ? a.items32 : reinterpret_cast<const int32_t*>(a.items);
    const int32_t* __restrict__ perm = a.perm;
    // prologue: rows of the first ST-1 samples in flight, ids of the next two in registers
#pragma unroll
    for (int q = 0; q < ST - 1; ++q) {
        const int64_t n = n0 + q * stride;
        if (n < end) issue(q, users_lo[IW * n], items_lo[IW * n]);
        cp_async_commit();
    }
    int uq = 0, iq = 0, uq2 = 0, iq2 = 0;
    if (n0 + (ST - 1) * stride < end) { uq = users_lo[IW * (n0 + (ST - 1) * stride)]; iq = items_lo[IW * (n0 + (ST - 1) * stride)]; }
    if (n0 + ST * stride < end) { uq2 = users_lo[IW * (n0 + ST * stride)]; iq2 = items_lo[IW * (n0 + ST * stride)]; }
    // per-sample scalars one iteration ahead, in ONE register spread over lanes 0..2 (score, low words of
    // perm_idx and of the old env), broadcast with shuffles when used.  The score is read at position n of the walk,
    // the tie-break index and the old env at the ORIGINAL position: o when SORTED, n in the plain order.
    const int gbase = tid & 16;
    const bool has_p = a.perm_idx != nullptr, has_d = a.diff != nullptr;
    auto load_scalars = [&](int64_t n, int o) -> int {
        const int32_t* p = reinterpret_cast<const int32_t*>(a.scores + n);
        bool on = lane == 0;
        if (lane == 1 && has_p) { p = reinterpret_cast<const int32_t*>(a.perm_idx + (SORTED ? o : n)); on = true; }
        if (lane == 2 && has_d) { p = reinterpret_cast<const int32_t*>(a.old_envs + (SORTED ? o : n)); on = true; }
        int v = 0;
        if (on) v = *p;
        return v;
    };
    // SORTED: original positions run two samples ahead of their use (perm -> scattered scalar loads -> use)
    int o_cur = 0, o_nx = 0, o_nx2 = 0;
    if (SORTED) {
        o_cur = (n0 < end) ? perm[n0] : 0;
        o_nx = (n0 + 1 < end) ? perm[n0 + 1] : 0;
        o_nx2 = (n0 + 2 < end) ? perm[n0 + 2] : 0;
    }
    int sc = (n0 < end) ? load_scalars(n0, o_cur) : 0;
    unsigned cnt[KT], ndiff = 0;   // lane 0: this group's histogram and diff count
#pragma unroll
    for (int k = 0; k < KT; ++k) cnt[k] = 0u;

    int slot = 0;
    for (int64_t n = n0; n < end; n += stride) {
        // request the rows of sample n + (ST-1) stride (ids loaded one iteration ago), then its successor's ids
        int wslot = slot + ST - 1; if (wslot >= ST) wslot -= ST;
        if (n + (ST - 1) * stride < end) issue(wslot, uq, iq);
        cp_async_commit();
        uq = uq2; iq = iq2;
        if (n + (ST + 1) * stride < end) { uq2 = users_lo[IW * (n + (ST + 1) * stride)]; iq2 = items_lo[IW * (n + (ST + 1) * stride)]; }
        const float y = __int_as_float(__shfl_sync(gmask, sc, gbase));
        const int pidx = __shfl_sync(gmask, sc, gbase + 1);
        const int old = __shfl_sync(gmask, sc, gbase + 2);
        const int o_this = o_cur;   // SORTED: original position of sample n
        if (n + stride < end) sc = load_scalars(n + stride, o_nx);
        if (SORTED) {
            o_cur = o_nx; o_nx = o_nx2;
            if (n + 3 < end) o_nx2 = perm[n + 3];
        }
        cp_async_wait<ST - 1>();
        Row<VEC, NV> ra, rc, rue, rie;
        read_staged_row<VEC, NV>(ra, ring, slot * 4 + 0, D, lane);
        read_staged_row<VEC, NV>(rc, ring, slot * 4 + 1, D, lane);
        read_staged_row<VEC, NV>(rue, ring, slot * 4 + 2, D, lane);
        read_staged_row<VEC, NV>(rie, ring, slot * 4 + 3, D, lane);
        float z1 = 0.f;
        float z2[KT];
#pragma unroll
        for (int k = 0; k < KT; ++k) z2[k] = 0.f;
#pragma unroll
        for (int j = 0; j < NV; ++j) {
            const int d0 = dim_of<VEC>(lane, j);
            if (d0 < D) {
#pragma unroll
                for (int v = 0; v < VEC; ++v) {
                    const int x = j * VEC + v;
                    z1 += ra.x[x] * rc.x[x];
                    const float t = rue.x[x] * rie.x[x];
#pragma unroll
                    for (int k = 0; k < KT; ++k)
                        if (k < K) z2[k] += t * (E_REG ? eR[E_REG ? k : 0][x] : sE[k * D + d0 + v]);
                }
            }
        }
        // K sums with one scattered reduction: lanes [k * 16/NS, (k+1) * 16/NS) end up with z2[k]; each computes
        // the distance under ITS environment, then a (distance, k) butterfly picks the first minimum
        // (torch.argmin: ties go to the lowest k, a NaN orders below every number so the first NaN wins) -- same
        // values as the serial loop of train.py:853-876.
        z1 = group_sum(z1, gmask);
        constexpr int NS = (KT <= 2) ? 2 : ((KT <= 4) ? 4 : 8);
        float zs[NS];
#pragma unroll
        for (int k = 0; k < NS; ++k) zs[k] = (k < KT) ? z2[k < KT ? k : 0] : 0.f;
        const float zk = group_sum_scatter<NS>(zs, lane, gmask);
        int arg = lane / (GROUP / NS);
        float d;
        if (a.implicit) {
            const float s = sigmoidf_(z1) * sigmoidf_(zk);
            d = -(y * fmaxf(logf(s), -100.f) + (1.f - y) * fmaxf(logf(1.f - s), -100.f));
        } else {
            const float r = (z1 + zk) - y;
            d = r * r;
        }
        if (arg < K) {
            if (has_p) d = d + ((eps_rows_smem > 0 ? sEps : a.eps_table) + (int64_t)pidx * K)[arg];
        } else {
            d = INFINITY;   // padding lanes never win (an all-inf row still resolves to the lowest k)
        }
        // torch.argmin returns the first NaN: a distance is never -inf (a square, or a BCE that is >= 0), so a NaN
        // becomes -inf, below every number, and NaN ties still go to the lowest k
        if (isnan(d)) d = -INFINITY;
#pragma unroll
        for (int off = GROUP / NS; off < GROUP; off <<= 1) {
            const float d2 = __shfl_xor_sync(gmask, d, off);
            const int k2 = __shfl_xor_sync(gmask, arg, off);
            if (d2 < d || (d2 == d && k2 < arg)) { d = d2; arg = k2; }
        }
        if (lane == 0) {
            a.new_envs[SORTED ? o_this : n] = (int64_t)arg;
#pragma unroll
            for (int k = 0; k < KT; ++k) cnt[k] += (arg == k) ? 1u : 0u;
            if (has_d && old != arg) ++ndiff;
        }
        if (++slot == ST) slot = 0;
    }
    cp_async_wait<0>();
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < KT; ++k)
            if (k < K && cnt[k] != 0u) atomicAdd(&sHist[k], (unsigned long long)cnt[k]);
        if (ndiff != 0u) atomicAdd(&sHist[INVPREF_MAX_ENVS], (unsigned long long)ndiff);
    }
    __syncthreads();
    if (tid < K && a.hist != nullptr && sHist[tid] != 0ull) atomicAdd(&a.hist[tid], sHist[tid]);
    if (tid == INVPREF_MAX_ENVS && a.diff != nullptr && sHist[tid] != 0ull) atomicAdd(a.diff, sHist[tid]);
}

// The two sample orders keep their own kernel names (profiles and tests tell them apart by name).
template <int VEC, int NV, int KT>
constexpr int cl_min_blocks() { return (VEC * NV <= 4 && KT <= 4) ? 4 : 1; }

template <int VEC, int NV, int KT, int DX>
__global__ void __launch_bounds__(BLOCK, cl_min_blocks<VEC, NV, KT>()) cluster_kernel(ClusterArgs a,
                                                                                      int eps_rows_smem) {
    cluster_body<VEC, NV, KT, DX, false>(a, eps_rows_smem);
}

template <int VEC, int NV, int KT, int DX>
__global__ void __launch_bounds__(BLOCK, cl_min_blocks<VEC, NV, KT>()) cluster_sorted_kernel(ClusterArgs a,
                                                                                             int eps_rows_smem) {
    cluster_body<VEC, NV, KT, DX, true>(a, eps_rows_smem);
}

// Counts in registers (one counter per environment per thread), warp sums with redux, one shared-memory atomic per
// warp and environment, one global atomic per CTA and environment.  Grid-stride over <= 148 * 8 CTAs: the dataset
// configs (3 * 10^5 samples) get a full grid instead of the five CTAs of a 2^16-samples-per-CTA split.
__global__ void __launch_bounds__(256) env_hist_kernel(const int64_t* __restrict__ envs, int64_t N, int K,
                                                       unsigned long long* __restrict__ hist) {
    __shared__ unsigned long long sH[INVPREF_MAX_ENVS];
    if (threadIdx.x < INVPREF_MAX_ENVS) sH[threadIdx.x] = 0ull;
    __syncthreads();
    unsigned cnt[INVPREF_MAX_ENVS];
#pragma unroll
    for (int k = 0; k < INVPREF_MAX_ENVS; ++k) cnt[k] = 0u;
    for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
        const int e = (int)envs[n];
#pragma unroll
        for (int k = 0; k < INVPREF_MAX_ENVS; ++k) cnt[k] += (e == k) ? 1u : 0u;
    }
#pragma unroll
    for (int k = 0; k < INVPREF_MAX_ENVS; ++k) {
        const unsigned w = __reduce_add_sync(0xffffffffu, cnt[k]);
        if ((threadIdx.x & 31) == 0 && w != 0u && k < K) atomicAdd(&sH[k], (unsigned long long)w);
    }
    __syncthreads();
    if ((int)threadIdx.x < K && sH[threadIdx.x] != 0ull) atomicAdd(&hist[threadIdx.x], sH[threadIdx.x]);
}

// class_weights[k] = min(cnt_k + 1, N - 1) / N in double, rounded to fp32 (train.py:950-955);
// sample_weights[n] = class_weights[envs[n]] (train.py:956).
__global__ void __launch_bounds__(256) stat_envs_kernel(const int64_t* __restrict__ envs, int64_t N, int K,
                                                        const int64_t* __restrict__ hist,
                                                        float* __restrict__ class_weights,
                                                        float* __restrict__ sample_weights) {
    __shared__ float sCW[INVPREF_MAX_ENVS];
    if ((int)threadIdx.x < K) {
        double c = (double)hist[threadIdx.x] + 1.0;
        double cap = (double)(N - 1);
        double rate = (c < cap ? c : cap) / (double)N;
        sCW[threadIdx.x] = (float)rate;
        if (blockIdx.x == 0 && class_weights != nullptr) class_weights[threadIdx.x] = (float)rate;
    }
    __syncthreads();
    if (sample_weights == nullptr) return;
    for (int64_t n = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; n < N; n += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = envs[n];
        sample_weights[n] = (e >= 0 && e < K) ? sCW[(int)e] : 0.f;
    }
}

}  // namespace

// ClusterArgs.perm != nullptr: the user-sorted view (cluster_sorted_kernel).
int launch_cluster(const Geometry& g, const ClusterArgs& a, cudaStream_t stream) {
    // a group handles <= 2^32 samples (its counters are 32-bit): B / (grid * 16) is far below that
    int eps_rows = 0;
    if (a.perm_idx != nullptr && a.eps_table != nullptr && g.K <= 6) {
        eps_rows = 1;
        for (int j = 2; j <= g.K; ++j) eps_rows *= j;
    }
    const size_t smem = ((size_t)ring_align_up(((g.K * g.D + 3) & ~3) + ((eps_rows * g.K + 3) & ~3)) +
                         (size_t)cl_stages(g.VEC, g.NV) * 4 * g.NV * g.VEC * BLOCK) * sizeof(float);
    int64_t need = (a.B + GROUPS_PER_BLOCK - 1) / GROUPS_PER_BLOCK;
    int grid = (int)(need < 1 ? 1 : (need < 148 * 16 ? need : 148 * 16));
    const bool sorted = a.perm != nullptr;
#define CALL_F(KERNEL)                                                                                           \
    do {                                                                                                         \
        INVPREF_SET_SMEM_ONCE(KERNEL, smem);                                                                     \
        KERNEL<<<grid, BLOCK, smem, stream>>>(a, eps_rows);                                                      \
    } while (0)
#define CALL_X(V, N, KT_, X)                                                                                     \
    do {                                                                                                         \
        if (sorted) CALL_F((cluster_sorted_kernel<V, N, KT_, X>));                                               \
        else CALL_F((cluster_kernel<V, N, KT_, X>));                                                             \
    } while (0)
#define CALL(V, N, KT_) CALL_X(V, N, KT_, 0)
#define CALL_EXACT(V, N, KT_) CALL_X(V, N, KT_, 64)
#define CALL_EXACT40(V, N, KT_) CALL_X(V, N, KT_, 40)
    if (g.VEC == 4 && g.D == 64 && g.K == g.KT) {
        INVPREF_DISPATCH_K(4, 1, g.KT, CALL_EXACT);
    } else if (g.VEC == 4 && g.D == 40 && g.K == g.KT) {
        INVPREF_DISPATCH_K(4, 1, g.KT, CALL_EXACT40);
    } else if (g.VEC == 4 && g.D == 40 && g.K == 5) {
        CALL_EXACT40(4, 1, 5);
    } else {
        INVPREF_DISPATCH_GEOM(g, CALL);
    }
#undef CALL
#undef CALL_EXACT
#undef CALL_EXACT40
#undef CALL_X
#undef CALL_F
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_env_hist(const int64_t* envs, int64_t N, int K, unsigned long long* hist, cudaStream_t stream) {
    // a thread's 32-bit counters see N / (grid * 256) samples: below 2^32 for any N < 2^50
    const int64_t need = (N + 1023) / 1024;
    const int grid = (int)(need < 1 ? 1 : (need < 148 * 8 ? need : 148 * 8));
    env_hist_kernel<<<grid, 256, 0, stream>>>(envs, N, K, hist);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_stat_envs(const int64_t* envs, int64_t N, int K, const int64_t* hist, float* class_weights,
                     float* sample_weights, cudaStream_t stream) {
    int64_t need = (N + 255) / 256;
    int grid = (int)(need < 1 ? 1 : (need < 148 * 8 ? need : 148 * 8));
    stat_envs_kernel<<<grid, 256, 0, stream>>>(envs, N, K, hist, class_weights, sample_weights);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

}  // namespace invpref
