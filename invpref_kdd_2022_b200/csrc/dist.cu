// Building blocks of the multi-GPU paths (the reference is single-GPU: no counterpart there).
//
//  adam_dense_kernel       : torch.optim.Adam on a flat tensor whose gradient was materialised because it
//                            had to be reduced across ranks first (NCCL all-reduce / all-to-all).
//  gather_rows_kernel      : packs the rows a peer asked for into a contiguous send buffer.
//  scatter_add_rows_kernel : adds one peer's partial row gradients into the owner's shard; indices are
//                            unique within a call, peers are applied in rank order => deterministic.
//
// Over peer memory (the other ranks' buffers, mapped into this process -- e.g. torch symmetric memory; no NCCL on
// the data path, the caller only needs a barrier between producers and consumers):
//  fetch_rows_p2p_kernel   : cache[c] = table_of(owner[c])[rows[c]] for both item tables (NVLink loads): replaces
//                            gather_rows + all-to-all of rows.
//  owner_adam_push_kernel  : for every row of the owner's shard, the partial gradients the ranks' item passes
//                            stored into its staging are summed in rank order (same order and arithmetic as
//                            zero-fill + scatter_add per rank) and consumed by Adam in registers; the updated row is
//                            stored into the requesters' caches (NVLink stores): replaces the all-to-all of
//                            gradients + zero-fill + G scatter-adds + adam_dense + the next batch's row exchange.
#include "common.cuh"
#include "kernels.h"

namespace invpref {

namespace {

__global__ void __launch_bounds__(256) adam_dense_kernel(float* __restrict__ theta, float* __restrict__ m,
                                                         float* __restrict__ v, const float* __restrict__ grad,
                                                         int64_t n, AdamScalars s0, int vec_ok,
                                                         const invpref_dyn* dyn) {
    const AdamScalars s = with_dyn(s0, dyn);
    const int64_t n4 = vec_ok ? (n >> 2) : 0;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int64_t t0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    for (int64_t q = t0; q < n4; q += stride) {
        float p[4], mm[4], vv[4], g[4];
        ldv_stream<4>(theta + q * 4, p);
        ldv_stream<4>(m + q * 4, mm);
        ldv_stream<4>(v + q * 4, vv);
        ldv_stream<4>(grad + q * 4, g);
#pragma unroll
        for (int x = 0; x < 4; ++x) adam_update(p[x], mm[x], vv[x], g[x], s);
        stv<4>(theta + q * 4, p);
        stv_stream<4>(m + q * 4, mm);
        stv_stream<4>(v + q * 4, vv);
    }
    for (int64_t q = n4 * 4 + t0; q < n; q += stride) {
        float p = theta[q], mm = m[q], vv = v[q];
        adam_update(p, mm, vv, grad[q], s);
        theta[q] = p; m[q] = mm; v[q] = vv;
    }
}

template <int VEC>
__global__ void __launch_bounds__(256) gather_rows_kernel(const float* __restrict__ table,
                                                          const int64_t* __restrict__ rows, int64_t n, int dim,
                                                          float* __restrict__ out) {
    const int per_row = dim / VEC;
    const int64_t total = n * per_row;
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t j = q / per_row;
        const int c = (int)(q - j * per_row) * VEC;
        float r[VEC];
        ldv<VEC>(table + rows[j] * dim + c, r);
        stv<VEC>(out + j * dim + c, r);
    }
}

template <int VEC>
__global__ void __launch_bounds__(256) scatter_add_rows_kernel(const float* __restrict__ src,
                                                               const int64_t* __restrict__ rows, int64_t n, int dim,
                                                               float* __restrict__ table) {
    const int per_row = dim / VEC;
    const int64_t total = n * per_row;
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t j = q / per_row;
        const int c = (int)(q - j * per_row) * VEC;
        float a[VEC], b[VEC];
        ldv<VEC>(src + j * dim + c, a);
        float* dst = table + rows[j] * dim + c;
        ldv<VEC>(dst, b);
#pragma unroll
        for (int x = 0; x < VEC; ++x) b[x] += a[x];
        stv<VEC>(dst, b);
    }
}

constexpr int P2P_MAX_WORLD = 16;
struct PeerPtrs { const float* p[2 * P2P_MAX_WORLD]; };   // [t * world + rank]: table t (0 inv, 1 env) of each rank

template <int VEC>
__global__ void __launch_bounds__(256) fetch_rows_p2p_kernel(PeerPtrs tables, int world,
                                                             const int32_t* __restrict__ owner,
                                                             const int64_t* __restrict__ rows, int64_t n, int dim,
                                                             float* __restrict__ out0, float* __restrict__ out1) {
    const int per_row = dim / VEC;
    const int64_t per_table = n * per_row, total = 2 * per_table;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    constexpr int U = 4;   // independent remote loads in flight per thread
    for (int64_t q0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q0 < total; q0 += U * stride) {
        float r[U][VEC];
        float* dst[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int64_t q = q0 + u * stride;
            dst[u] = nullptr;
            if (q < total) {
                const int t = q >= per_table ? 1 : 0;
                const int64_t rem = q - t * per_table;
                const int64_t j = (int64_t)((uint32_t)rem / (uint32_t)per_row);   // per_table < 2^31 (checked at launch)
                const int c = (int)(rem - j * per_row) * VEC;
                const float* src = tables.p[t * world + owner[j]] + rows[j] * dim + c;
                ldv_sys<VEC>(src, r[u]);
                dst[u] = (t ? out1 : out0) + j * dim + c;
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
            if (dst[u] != nullptr) stv<VEC>(dst[u], r[u]);
    }
}

struct PeerOut { float* p[2 * P2P_MAX_WORLD]; };

// Owner side of the PUSH exchange: partials from LOCAL staging (the ranks' item passes stored them there over
// NVLink), summed in rank order, Adam in registers, and the updated row stored into every requester's row cache
// for the next batch (posted NVLink writes).  Same per-element arithmetic and order as the collective path: zero-fill,
// scatter_add_rows_kernel per rank in rank order, adam_dense_kernel.
// WMAX: compile-time bound of the rank loops (2, 4, 8, 16): the position loads, the staging loads and the pushes are
// fully unrolled and all in flight together.
template <int VEC, int WMAX>
__global__ void __launch_bounds__(256) owner_adam_push_kernel(float* __restrict__ th0, float* __restrict__ th1,
                                                              float* __restrict__ m0, float* __restrict__ m1,
                                                              float* __restrict__ v0, float* __restrict__ v1,
                                                              int64_t n_rows, int dim, int world,
                                                              const float* __restrict__ stage0,
                                                              const float* __restrict__ stage1,
                                                              const int32_t* __restrict__ spos, PeerOut caches,
                                                              const int32_t* __restrict__ npos, AdamScalars s0,
                                                              const invpref_dyn* dyn) {
    const AdamScalars s = with_dyn(s0, dyn);
    const int per_row = dim / VEC;
    const int64_t per_table = n_rows * per_row, total = 2 * per_table;
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
        const int t = q >= per_table ? 1 : 0;
        const int64_t rem = q - t * per_table;
        const int64_t j = (int64_t)((uint32_t)rem / (uint32_t)per_row);   // per_table < 2^31 (checked at launch)
        const int c = (int)(rem - j * per_row) * VEC;
        const float* __restrict__ stage = t ? stage1 : stage0;
        int sl[WMAX];
        float part[WMAX][VEC];
#pragma unroll
        for (int p = 0; p < WMAX; ++p) sl[p] = (p < world) ? spos[(int64_t)p * n_rows + j] : -1;
#pragma unroll
        for (int p = 0; p < WMAX; ++p) {
            if (sl[p] >= 0) {
                ldv_sys<VEC>(stage + (int64_t)sl[p] * dim + c, part[p]);   // written by a peer: never from this SM's L1
            } else {
#pragma unroll
                for (int x = 0; x < VEC; ++x) part[p][x] = 0.f;
            }
        }
        float g[VEC];
#pragma unroll
        for (int x = 0; x < VEC; ++x) g[x] = 0.f;
#pragma unroll
        for (int p = 0; p < WMAX; ++p)
            if (sl[p] >= 0) {
#pragma unroll
                for (int x = 0; x < VEC; ++x) g[x] += part[p][x];
            }
        float* th = (t ? th1 : th0) + j * dim + c;
        float* mm = (t ? m1 : m0) + j * dim + c;
        float* vv = (t ? v1 : v0) + j * dim + c;
        float pr[VEC], mr[VEC], vr[VEC];
        ldv_stream<VEC>(th, pr);
        ldv_stream<VEC>(mm, mr);
        ldv_stream<VEC>(vv, vr);
#pragma unroll
        for (int x = 0; x < VEC; ++x) adam_update(pr[x], mr[x], vr[x], g[x], s);
        stv<VEC>(th, pr);
        stv_stream<VEC>(mm, mr);
        stv_stream<VEC>(vv, vr);
        if (npos != nullptr) {
#pragma unroll
            for (int p = 0; p < WMAX; ++p) {
                if (p < world) {
                    const int slot = npos[(int64_t)p * n_rows + j];
                    if (slot >= 0) stv<VEC>(caches.p[t * world + p] + (int64_t)slot * dim + c, pr);
                }
            }
        }
    }
}

// ---- all-reduce of a few KB + barrier over peer memory (invpref_peer_allreduce) -------------------------------
// The sharded step needs two rank-wide synchronisation points per step, one of which carries the gradients of the
// replicated tensors (E, W, b: 2KD + K + 6 floats).  Instead of an NCCL all-reduce per point, every rank
//   post   : stores its vector into slot [parity][rank] of EVERY rank's mapped slot array (posted NVLink writes),
//            fences at system scope and release-stores the sequence number into flag [rank] of every rank;
//   reduce : acquire-spins on its OWN flags until all ranks have posted this sequence number, then sums the slots in
//            rank order -- the same order on every rank, so the replicas stay bit-identical.
// Ordering: everything the stream ran before `post` (the item pass and its pushes into peer staging, the owner kernel
// and its row pushes) happens-before the release store, hence before any peer's kernels that follow its `reduce`.
// The sequence number lives in device memory (`ctr`, advanced by `reduce`), so a captured CUDA graph replays it
// correctly.  Slots are double-buffered by sequence parity: a rank can be at most one synchronisation point ahead of a
// peer (to post point k+2 it must have seen the peer's post of k+1, which the peer issues after its reduce of k).
// The spin is bounded (~seconds); on expiry bit 0 of *status is set and the kernel goes on (the caller raises).
struct PeerSync {
    float* slots[P2P_MAX_WORLD];       // rank p's slot array   [2][world][n_max]
    unsigned* flags[P2P_MAX_WORLD];    // rank p's flag array   [world]
};

__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(256) peer_post_kernel(const float* __restrict__ src, int n, int n_max, int world,
                                                        int rank, PeerSync ps, const unsigned* __restrict__ ctr) {
    const unsigned seq = *ctr + 1u;
    const int64_t off = ((int64_t)(seq & 1u) * world + rank) * n_max;
    for (int idx = threadIdx.x; idx < world * n; idx += blockDim.x) {
        const int p = idx / n, i = idx - p * n;
        ps.slots[p][off + i] = src[i];
    }
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < world) st_release_sys(ps.flags[threadIdx.x] + rank, seq);
}

__global__ void __launch_bounds__(256) peer_reduce_kernel(float* __restrict__ dst, int n, int n_max, int world,
                                                          const float* my_slots, const unsigned* my_flags,
                                                          unsigned* ctr, int32_t* status, unsigned spin_limit) {
    const unsigned seq = *ctr + 1u;
    if ((int)threadIdx.x < world) {
        unsigned it = 0;
        while ((int)(ld_acquire_sys(my_flags + threadIdx.x) - seq) < 0) {
            if (++it > spin_limit) { atomicOr(status, 1); break; }
            __nanosleep(200);
        }
    }
    __syncthreads();
    const float* base = my_slots + (int64_t)(seq & 1u) * world * n_max;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        float s = 0.f;
        for (int p = 0; p < world; ++p) {
            float v;
            ldv_sys<1>(base + (int64_t)p * n_max + i, &v);      // written by a peer: never from this SM's L1
            s += v;
        }
        dst[i] = s;
    }
    __syncthreads();
    if (threadIdx.x == 0) *ctr = seq;
}

inline int grid_1d(int64_t work, int max_blocks = 148 * 16) {
    int64_t need = (work + 255) / 256;
    if (need < 1) need = 1;
    return (int)(need < max_blocks ? need : max_blocks);
}

}  // namespace

int launch_adam_dense(float* theta, float* m, float* v, const float* grad, int64_t n, const AdamScalars& s,
                      const invpref_dyn* dyn, cudaStream_t stream) {
    const int vec_ok = (((uintptr_t)theta | (uintptr_t)m | (uintptr_t)v | (uintptr_t)grad) % 16) == 0;
    adam_dense_kernel<<<grid_1d(vec_ok ? n / 4 + 4 : n), 256, 0, stream>>>(theta, m, v, grad, n, s, vec_ok, dyn);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_gather_rows(const float* table, const int64_t* rows, int64_t n, int dim, float* out, cudaStream_t stream) {
    const bool v4 = dim % 4 == 0 && ((uintptr_t)table % 16 == 0) && ((uintptr_t)out % 16 == 0);
    if (v4) gather_rows_kernel<4><<<grid_1d(n * (dim / 4)), 256, 0, stream>>>(table, rows, n, dim, out);
    else gather_rows_kernel<1><<<grid_1d(n * dim), 256, 0, stream>>>(table, rows, n, dim, out);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_scatter_add_rows(const float* src, const int64_t* rows, int64_t n, int dim, float* table,
                            cudaStream_t stream) {
    const bool v4 = dim % 4 == 0 && ((uintptr_t)table % 16 == 0) && ((uintptr_t)src % 16 == 0);
    if (v4) scatter_add_rows_kernel<4><<<grid_1d(n * (dim / 4)), 256, 0, stream>>>(src, rows, n, dim, table);
    else scatter_add_rows_kernel<1><<<grid_1d(n * dim), 256, 0, stream>>>(src, rows, n, dim, table);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_fetch_rows_p2p(const float* const* tables_host, int world, const int32_t* owner, const int64_t* rows,
                          int64_t n, int dim, float* out0, float* out1, cudaStream_t stream) {
    if (world < 1 || world > P2P_MAX_WORLD || n * (int64_t)dim >= 0x7fffffffLL) return INVPREF_ERR_BAD_ARG;
    PeerPtrs pp = {};
    bool v4 = dim % 4 == 0 && ((uintptr_t)out0 % 16 == 0) && ((uintptr_t)out1 % 16 == 0);
    for (int i = 0; i < 2 * world; ++i) { pp.p[i] = tables_host[i]; v4 = v4 && ((uintptr_t)tables_host[i] % 16 == 0); }
    if (v4) fetch_rows_p2p_kernel<4><<<grid_1d(2 * n * (dim / 4) / 4 + 256), 256, 0, stream>>>(pp, world, owner, rows, n, dim, out0, out1);
    else fetch_rows_p2p_kernel<1><<<grid_1d(2 * n * dim / 4 + 256), 256, 0, stream>>>(pp, world, owner, rows, n, dim, out0, out1);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_owner_adam_push(float* th0, float* th1, float* m0, float* m1, float* v0, float* v1, int64_t n_rows, int dim,
                           int world, const float* stage0, const float* stage1, const int32_t* spos,
                           float* const* caches_host, const int32_t* npos, const AdamScalars& s,
                           const invpref_dyn* dyn, cudaStream_t stream) {
    if (world < 1 || world > P2P_MAX_WORLD || n_rows * (int64_t)dim >= 0x7fffffffLL) return INVPREF_ERR_BAD_ARG;
    PeerOut pp = {};
    bool v4 = dim % 4 == 0 && ((uintptr_t)stage0 % 16 == 0) && ((uintptr_t)stage1 % 16 == 0);
    for (float* q : {th0, th1, m0, m1, v0, v1}) v4 = v4 && ((uintptr_t)q % 16 == 0);
    for (int i = 0; caches_host && i < 2 * world; ++i) {
        pp.p[i] = caches_host[i];
        v4 = v4 && ((uintptr_t)caches_host[i] % 16 == 0);
    }
#define PUSH_CALL(V, W)                                                                                          \
    owner_adam_push_kernel<V, W><<<grid_1d(2 * n_rows * (dim / V)), 256, 0, stream>>>(                           \
        th0, th1, m0, m1, v0, v1, n_rows, dim, world, stage0, stage1, spos, pp, npos, s, dyn)
#define PUSH_W(V)                                                                                                \
    do {                                                                                                         \
        if (world <= 2) PUSH_CALL(V, 2);                                                                         \
        else if (world <= 4) PUSH_CALL(V, 4);                                                                    \
        else if (world <= 8) PUSH_CALL(V, 8);                                                                    \
        else PUSH_CALL(V, 16);                                                                                   \
    } while (0)
    if (v4) PUSH_W(4);
    else PUSH_W(1);
#undef PUSH_W
#undef PUSH_CALL
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_peer_allreduce(float* buf, int n, int n_max, int world, int rank, float* const* slots_host,
                          uint32_t* const* flags_host, uint32_t* ctr, int32_t* status, cudaStream_t stream) {
    if (world < 1 || world > P2P_MAX_WORLD || rank < 0 || rank >= world || n < 0 || n > n_max) return INVPREF_ERR_BAD_ARG;
    PeerSync ps = {};
    for (int p = 0; p < world; ++p) {
        ps.slots[p] = slots_host[p];
        ps.flags[p] = flags_host[p];
    }
    peer_post_kernel<<<1, 256, 0, stream>>>(buf, n, n_max, world, rank, ps, ctr);
    // 200 ns sleeps: 50 M iterations = at least 10 s before a missing peer is reported instead of waited for
    peer_reduce_kernel<<<1, 256, 0, stream>>>(buf, n, n_max, world, ps.slots[rank], ps.flags[rank], ctr, status,
                                              50u * 1000u * 1000u);
    count_launch(2);
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

}  // namespace invpref
