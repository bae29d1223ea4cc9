// Shared device helpers and internal structs for libinvpref_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "invpref_b200.h"

namespace invpref {

// One embedding row is handled by a GROUP of 16 lanes; lane l owns NV vectors of VEC floats at
// dims (j*GROUP + l)*VEC .. +VEC, j < NV.  D = 64 -> 16 x float4 (one 128-bit load per lane per
// row, a half-warp reads a full 256 B row = 8 sectors, coalesced); D = 40 -> 10 active lanes;
// D = 30 -> float2 x 15 lanes.
constexpr int GROUP = 16;
constexpr int BLOCK = 256;                 // threads per CTA for the row kernels (16 groups)
constexpr int GROUPS_PER_BLOCK = BLOCK / GROUP;

// Segments longer than 2*chunk interactions are pre-reduced in chunk-sized pieces by separate groups
// (fixed shape => deterministic), the owner row then sums the partials in order.  A segment is reduced
// serially by one group, so the chunk bounds the critical path: small batches (B = 64K..256K with a few
// hot rows) need small chunks to spread the hot rows over the machine, large ones amortise better with
// big chunks.  chunk is a function of the batch size only.
// Round 2: on the dataset-scale batches (<= 2^18 interactions, everything L2-resident) a group spends ~4-5 us per
// interaction of serial latency, so the longest UNCHUNKED segment (2 * chunk) is the critical path of the rows kernels
// (MIND shape, chunk 32: 64 interactions = 0.30 ms of a 0.55 ms step): chunks of 8 there.
inline int chunk_for(int64_t B) {
    if (B >= ((int64_t)1 << 22)) return 256;
    int64_t c = 8;
    while (c < 128 && c * 32768 < B) c *= 2;
    return (int)c;
}

struct Geometry {
    int D, K;
    int VEC, NV, KT;   // vector width, vectors per lane, compile-time env capacity
    int GS;            // floats per interaction in the g-pack
};

inline int make_geometry(const invpref_desc* d, Geometry* g) {
    if (d == nullptr) return INVPREF_ERR_BAD_ARG;
    if (d->dim < 1 || d->dim > INVPREF_MAX_DIM) return INVPREF_ERR_BAD_DIM;
    if (d->n_envs < 1 || d->n_envs > INVPREF_MAX_ENVS) return INVPREF_ERR_BAD_ENVS;
    if (d->n_users < 1 || d->n_items < 1 || d->n_users > 0x7fffffffLL || d->n_items > 0x7fffffffLL)
        return INVPREF_ERR_BAD_ARG;
    int D = d->dim;
    g->D = D;
    g->K = d->n_envs;
    if (D % 4 == 0) {
        g->VEC = 4;
        g->NV = D <= 64 ? 1 : (D <= 128 ? 2 : 4);
    } else if (D % 2 == 0) {
        g->VEC = 2;
        if (D > 64) return INVPREF_ERR_BAD_DIM;
        g->NV = D <= 32 ? 1 : 2;
    } else {
        g->VEC = 1;
        if (D > 64) return INVPREF_ERR_BAD_DIM;
        g->NV = 4;
    }
    g->KT = g->K <= 2 ? 2 : (g->K <= 4 ? 4 : (g->K <= 6 ? 6 : 8));
    g->GS = g->K <= 5 ? 8 : 12;
    return INVPREF_OK;
}

// Invokes F<VEC,NV,KT>() for the instantiated combinations.
#define INVPREF_DISPATCH_GEOM(geom, CALL)                                                   \
    do {                                                                                    \
        const int _v = (geom).VEC, _n = (geom).NV, _k = (geom).KT;                          \
        if (_v == 4 && _n == 1) { INVPREF_DISPATCH_K(4, 1, _k, CALL); }                     \
        else if (_v == 4 && _n == 2) { INVPREF_DISPATCH_K(4, 2, _k, CALL); }                \
        else if (_v == 4 && _n == 4) { INVPREF_DISPATCH_K(4, 4, _k, CALL); }                \
        else if (_v == 2 && _n == 1) { INVPREF_DISPATCH_K(2, 1, _k, CALL); }                \
        else if (_v == 2 && _n == 2) { INVPREF_DISPATCH_K(2, 2, _k, CALL); }                \
        else { INVPREF_DISPATCH_K(1, 4, _k, CALL); }                                        \
    } while (0)

#define INVPREF_DISPATCH_K(V, N, k, CALL)                                                   \
    do {                                                                                    \
        if ((k) == 2) { CALL(V, N, 2); }                                                    \
        else if ((k) == 4) { CALL(V, N, 4); }                                               \
        else if ((k) == 6) { CALL(V, N, 6); }                                               \
        else { CALL(V, N, 8); }                                                             \
    } while (0)

// Same, for kernels that do not depend on the env capacity.
#define INVPREF_DISPATCH_VN(geom, CALL)                                                     \
    do {                                                                                    \
        const int _v = (geom).VEC, _n = (geom).NV;                                          \
        if (_v == 4 && _n == 1) { CALL(4, 1); }                                             \
        else if (_v == 4 && _n == 2) { CALL(4, 2); }                                        \
        else if (_v == 4 && _n == 4) { CALL(4, 4); }                                        \
        else if (_v == 2 && _n == 1) { CALL(2, 1); }                                        \
        else if (_v == 2 && _n == 2) { CALL(2, 2); }                                        \
        else { CALL(1, 4); }                                                                \
    } while (0)

extern long long g_launch_count;   // host-side counter (api.cu)
inline void count_launch(int n = 1) { g_launch_count += n; }

// Exclusive prefix of `v` over the CTA (blockDim.x a multiple of 32, <= 1024); *total = the CTA's sum.
// `sm` = 33 ints of shared memory; may be reused right after the call.
__device__ __forceinline__ int block_exclusive_scan(int v, int* total, int* sm) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) sm[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        const int w = lane < nwarps ? sm[lane] : 0;
        int winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += y;
        }
        sm[lane] = winc - w;
        if (lane == 31) sm[32] = winc;
    }
    __syncthreads();
    const int res = inc - v + sm[warp];
    *total = sm[32];
    __syncthreads();
    return res;
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per kernel instantiation (and again only if a larger size is
// asked for), not on every launch: each textual expansion owns its static.  One process drives one GPU.
#define INVPREF_SET_SMEM_ONCE(KERNEL, BYTES)                                                                     \
    do {                                                                                                         \
        static int _smem_set = 0;                                                                                \
        if ((int)(BYTES) > _smem_set) {                                                                          \
            cudaFuncSetAttribute(KERNEL, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(BYTES));             \
            _smem_set = (int)(BYTES);                                                                            \
        }                                                                                                        \
    } while (0)

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// ---- plan layout (one side = one sort order) ----------------------------------------------
struct PlanSide {
    int32_t* counters;    // [0] n_seg, [1] n_chunks, [2] error flag ; 16 ints
    int32_t* perm;        // [B]   sorted position -> original index in the batch
    int32_t* partner;     // [B]   id of the OTHER table's row, in sorted order
    int32_t* seg_of;      // [B]   segment index on THIS side of interaction n (original order)
    int32_t* pseg;        // [B]   segment index on the OTHER side of the partner row, in sorted order
    int32_t* seg_row;     // [S]   unique ids ascending                     (S <= min(B, rows))
    int32_t* seg_off;     // [S+1] offsets into perm
    int32_t* seg_chunk;   // [S+1] exclusive scan of per-segment chunk counts (0 for short segments)
    int32_t* chunk_desc;  // [max_chunks*4] (seg, begin, end, unused)
    int32_t* seg_desc;    // [S*8] (row, begin, end, perm[begin]; partner[begin], perm[begin+1], partner[begin+1], -):
                          //       everything a kernel needs to request a segment's rows and its first two
                          //       interactions, in one 32-byte record
    int32_t* range_start; // [R+1] cost-balanced contiguous segment ranges: range r = segments
                          //       [range_start[r], range_start[r+1]); R = counters[3] = plan_ranges(B)
    uint32_t* touched;    // [ceil(rows/32)] bitmap of rows that have a segment
    int32_t* hot_list;    // [max_chunks / HOT_CHUNKS + 1] segments with more than HOT_CHUNKS chunks (counters[4] of
                          //       them, in no particular order): their chunk partials are summed by a whole CTA
    int64_t max_seg, max_chunks, rows, B;
};

// A segment that was cut into more than HOT_CHUNKS chunks (a hot item: > 16 * chunk interactions in one batch) would
// have its chunk partials summed one after the other by a single 16-lane group -- the critical path of the whole item
// pass on the dataset-scale configs (Yahoo: item 0 = 820 partials = 0.3 ms of a 0.38 ms step).  Such rows are listed
// by the plan and reduced by all 16 groups of a CTA in a fixed two-level order.
constexpr int HOT_CHUNKS = 16;

inline int64_t plan_max_seg(int64_t B, int64_t rows) { return B < rows ? B : rows; }
// Work ranges of the ring rows kernel: contiguous runs of segments of about equal cost (PLAN_CSEG per segment
// + 1 per interaction), a few dozen interactions each; a group takes ranges g, g + G, ... so that whatever the
// cost model misses averages out.  The count depends on the batch size only.
constexpr int PLAN_CSEG = 2;
inline int64_t plan_ranges(int64_t B) { int64_t r = B / 64; return r < 1 ? 1 : (r > 65536 ? 65536 : r); }
// Upper bound on the chunk count of a batch of AT MOST B interactions (monotonic in B, so a workspace sized
// for the largest batch also fits every shorter one): chunks <= 1.5 * B' / chunk_for(B') for any B' <= B.
inline int64_t plan_max_chunks(int64_t B) {
    int64_t small = B / 8 < 32768 ? B / 8 : 32768;     // B' / chunk_for(B') <= 32768 for every B' < 2^22
    int64_t big = B / 256;
    return 3 * (small > big ? small : big) / 2 + 4;
}

inline size_t plan_side_bytes(int64_t B, int64_t rows) {
    int64_t S = plan_max_seg(B, rows);
    size_t n = 0;
    n += align_up(16 * 4);
    n += align_up((size_t)B * 4) * 4;
    n += align_up((size_t)S * 4);
    n += align_up((size_t)(S + 1) * 4) * 2;
    n += align_up((size_t)plan_max_chunks(B) * 16);
    n += align_up((size_t)S * 32);
    n += align_up((size_t)(plan_ranges(B) + 1) * 4);
    n += align_up((size_t)((rows + 31) / 32) * 4);
    n += align_up((size_t)(plan_max_chunks(B) / HOT_CHUNKS + 1) * 4);
    return n;
}

inline PlanSide carve_plan_side(char* base, int64_t B, int64_t rows) {
    PlanSide p;
    int64_t S = plan_max_seg(B, rows);
    p.max_seg = S;
    p.max_chunks = plan_max_chunks(B);
    p.rows = rows;
    p.B = B;
    char* c = base;
    p.counters = (int32_t*)c;   c += align_up(16 * 4);
    p.perm = (int32_t*)c;       c += align_up((size_t)B * 4);
    p.partner = (int32_t*)c;    c += align_up((size_t)B * 4);
    p.seg_of = (int32_t*)c;     c += align_up((size_t)B * 4);
    p.pseg = (int32_t*)c;       c += align_up((size_t)B * 4);
    p.seg_row = (int32_t*)c;    c += align_up((size_t)S * 4);
    p.seg_off = (int32_t*)c;    c += align_up((size_t)(S + 1) * 4);
    p.seg_chunk = (int32_t*)c;  c += align_up((size_t)(S + 1) * 4);
    p.chunk_desc = (int32_t*)c; c += align_up((size_t)p.max_chunks * 16);
    p.seg_desc = (int32_t*)c;   c += align_up((size_t)S * 32);
    p.range_start = (int32_t*)c; c += align_up((size_t)(plan_ranges(B) + 1) * 4);
    p.touched = (uint32_t*)c;    c += align_up((size_t)((rows + 31) / 32) * 4);
    p.hot_list = (int32_t*)c;
    return p;
}

// ---- workspace layout ------------------------------------------------------------------------
constexpr int FWD_MAX_BLOCKS = 148 * 4 + 148;   // upper bound on CTAs that write a partial-sum vector

struct Workspace {
    float* stash;        // [min(B, n_users) * 2 * D]  lazy mode: caught-up user rows of the batch
    float* gpack;        // [B * GS]
    float* partials;     // [FWD_MAX_BLOCKS * P]   per-CTA partial sums of the forward kernel
    float* chunk_part_u; // [max_chunks * 2 * D]
    float* chunk_part_i; // [max_chunks * 2 * D]
    char* plan;          // scratch plan (when the caller passes none)
    char* sort_tmp;      // keys / ping-pong arrays / segment ids + tile counts of the radix sort and scans (sort.cuh)
    size_t sort_tmp_bytes;
    size_t plan_bytes;
};

// number of floats one forward CTA writes: 8 scalars, db[KT], cnt[KT], dW[K*D], dE[K*D]
inline int fwd_partial_floats(const Geometry& g) { return 8 + 2 * 8 + 2 * g.K * g.D; }

size_t sort_tmp_bytes_for(int64_t B, int64_t max_rows);   // plan.cu

inline size_t workspace_bytes_impl(const invpref_desc* d, const Geometry& g, int64_t B, Workspace* w, char* base) {
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes); return base ? base + o : (char*)nullptr; };
    int64_t Bp = B > 0 ? B : 1;
    int64_t Su = Bp < d->n_users ? Bp : d->n_users;
    char* sh = take((size_t)Su * 2 * g.D * 4);
    char* gp = take((size_t)Bp * g.GS * 4);
    char* pa = take((size_t)FWD_MAX_BLOCKS * fwd_partial_floats(g) * 4);
    char* cu = take((size_t)plan_max_chunks(Bp) * 2 * g.D * 4);
    char* ci = take((size_t)plan_max_chunks(Bp) * 2 * g.D * 4);
    size_t pb = plan_side_bytes(Bp, d->n_users) + plan_side_bytes(Bp, d->n_items);
    char* pl = take(pb);
    int64_t mr = d->n_users > d->n_items ? d->n_users : d->n_items;
    size_t sb = sort_tmp_bytes_for(Bp, mr);
    char* st = take(sb);
    if (w) {
        w->stash = (float*)sh;
        w->gpack = (float*)gp; w->partials = (float*)pa; w->chunk_part_u = (float*)cu; w->chunk_part_i = (float*)ci;
        w->plan = pl; w->sort_tmp = st; w->sort_tmp_bytes = sb; w->plan_bytes = pb;
    }
    return off;
}

// =============================== device helpers ================================================
#ifdef __CUDACC__

template <int VEC> struct VecT;
template <> struct VecT<4> { using type = float4; };
template <> struct VecT<2> { using type = float2; };
template <> struct VecT<1> { using type = float; };

// plain (cached) vector load of VEC floats
template <int VEC> __device__ __forceinline__ void ldv(const float* p, float* r);
template <> __device__ __forceinline__ void ldv<4>(const float* p, float* r) {
    float4 v = *reinterpret_cast<const float4*>(p); r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
}
template <> __device__ __forceinline__ void ldv<2>(const float* p, float* r) {
    float2 v = *reinterpret_cast<const float2*>(p); r[0] = v.x; r[1] = v.y;
}
template <> __device__ __forceinline__ void ldv<1>(const float* p, float* r) { r[0] = *p; }

// streaming load (read once: evict-first, do not allocate in L1)
template <int VEC> __device__ __forceinline__ void ldv_stream(const float* p, float* r);
template <> __device__ __forceinline__ void ldv_stream<4>(const float* p, float* r) {
    float4 v = __ldcs(reinterpret_cast<const float4*>(p)); r[0] = v.x; r[1] = v.y; r[2] = v.z; r[3] = v.w;
}
template <> __device__ __forceinline__ void ldv_stream<2>(const float* p, float* r) {
    float2 v = __ldcs(reinterpret_cast<const float2*>(p)); r[0] = v.x; r[1] = v.y;
}
template <> __device__ __forceinline__ void ldv_stream<1>(const float* p, float* r) { r[0] = __ldcs(p); }

// system-scope (volatile) load: for memory another GPU writes between kernels (peer memory over NVLink):
// never served from this SM's L1
template <int VEC> __device__ __forceinline__ void ldv_sys(const float* p, float* r);
template <> __device__ __forceinline__ void ldv_sys<4>(const float* p, float* r) {
    asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(r[0]), "=f"(r[1]), "=f"(r[2]), "=f"(r[3]) : "l"(p));
}
template <> __device__ __forceinline__ void ldv_sys<2>(const float* p, float* r) {
    asm volatile("ld.volatile.global.v2.f32 {%0, %1}, [%2];" : "=f"(r[0]), "=f"(r[1]) : "l"(p));
}
template <> __device__ __forceinline__ void ldv_sys<1>(const float* p, float* r) {
    asm volatile("ld.volatile.global.f32 %0, [%1];" : "=f"(r[0]) : "l"(p));
}

template <int VEC> __device__ __forceinline__ void stv(float* p, const float* r);
template <> __device__ __forceinline__ void stv<4>(float* p, const float* r) {
    *reinterpret_cast<float4*>(p) = make_float4(r[0], r[1], r[2], r[3]);
}
template <> __device__ __forceinline__ void stv<2>(float* p, const float* r) {
    *reinterpret_cast<float2*>(p) = make_float2(r[0], r[1]);
}
template <> __device__ __forceinline__ void stv<1>(float* p, const float* r) { *p = r[0]; }

template <int VEC> __device__ __forceinline__ void stv_stream(float* p, const float* r);
template <> __device__ __forceinline__ void stv_stream<4>(float* p, const float* r) {
    __stcs(reinterpret_cast<float4*>(p), make_float4(r[0], r[1], r[2], r[3]));
}
template <> __device__ __forceinline__ void stv_stream<2>(float* p, const float* r) {
    __stcs(reinterpret_cast<float2*>(p), make_float2(r[0], r[1]));
}
template <> __device__ __forceinline__ void stv_stream<1>(float* p, const float* r) { __stcs(p, r[0]); }

// A row slice held by one lane: NV vectors of VEC floats.
template <int VEC, int NV> struct Row {
    float x[NV * VEC];
};

// dim index of element (j, v) for this lane
template <int VEC> __device__ __forceinline__ int dim_of(int lane, int j) { return (j * GROUP + lane) * VEC; }

template <int VEC, int NV, bool STREAM = false>
__device__ __forceinline__ void load_row(Row<VEC, NV>& r, const float* __restrict__ table, int64_t row, int D, int lane) {
    const float* p = table + row * (int64_t)D;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        int d0 = dim_of<VEC>(lane, j);
        if (d0 < D) {
            if (STREAM) ldv_stream<VEC>(p + d0, &r.x[j * VEC]);
            else ldv<VEC>(p + d0, &r.x[j * VEC]);
        } else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) r.x[j * VEC + v] = 0.f;
        }
    }
}

template <int VEC, int NV, bool STREAM = false>
__device__ __forceinline__ void store_row(const Row<VEC, NV>& r, float* __restrict__ table, int64_t row, int D, int lane) {
    float* p = table + row * (int64_t)D;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        int d0 = dim_of<VEC>(lane, j);
        if (d0 < D) {
            if (STREAM) stv_stream<VEC>(p + d0, &r.x[j * VEC]);
            else stv<VEC>(p + d0, &r.x[j * VEC]);
        }
    }
}

// The two 16-lane groups of a warp run loops with different trip counts, so every in-loop shuffle names
// only its own half-warp: a full-warp mask there would wait for lanes that have already left the loop.
__device__ __forceinline__ unsigned group_mask() { return 0xffffu << (threadIdx.x & 16); }

// Software pipelining of the random row gathers: a row that a group will need one iteration later is
// requested into L2 now (no register is tied up), so the later load pays L2 latency instead of DRAM
// latency.  One request per 128-byte line of the row, issued by the first lanes of the group.
__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ void prefetch_row(const float* __restrict__ table, int64_t row, int D, int lane) {
    const char* base = reinterpret_cast<const char*>(table + row * (int64_t)D);
    const int bytes = D * 4;
    if (lane * 128 < bytes) prefetch_l2(base + lane * 128);
    if (lane == GROUP - 1 && (bytes & 127)) prefetch_l2(base + bytes - 4);   // trailing partial line
}

// ---- cp.async staging: global -> shared copies that tie up no register while in flight -----------------
// Every lane copies ITS OWN slice of a row (the same VEC floats it later reads back), so completion only has to
// be visible to the issuing thread: cp.async.wait_group is enough, no barrier.  A slot a lane reads is always
// one it wrote itself.
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <int BYTES> __device__ __forceinline__ void cp_async(uint32_t dst, const void* src) {
    if constexpr (BYTES == 16)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");   // L2 only
    else
        asm volatile("cp.async.ca.shared.global [%0], [%1], %2;" ::"r"(dst), "l"(src), "n"(BYTES) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int PENDING> __device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(PENDING) : "memory");
}

// The staging rings start on a 128-byte boundary of shared memory (RING_ALIGN floats).  A warp-wide 16-byte cp.async
// writes 512 contiguous bytes; when that span straddles 128-byte lines unevenly the LSU splits the instruction and
// re-requests sectors from L2: ncu on the round-2 user pass whose ring had slipped from offset 32 to 48 (mod 128)
// showed TWICE the L2 -> L1 sectors for LDGSTS (7.5 -> 14.7 GB per launch) and an 11 % longer kernel.
constexpr int RING_ALIGN = 32;
__host__ __device__ inline int ring_align_up(int floats) { return (floats + RING_ALIGN - 1) & ~(RING_ALIGN - 1); }

// Per-thread slot of a staged row slice: [slot][j][thread][VEC] floats (consecutive threads -> consecutive
// VEC*4 bytes: conflict-free for the 128-bit shared loads).
template <int VEC, int NV>
__device__ __forceinline__ float* stage_slot(float* ring, int slot) {
    return ring + ((size_t)slot * NV * BLOCK + threadIdx.x) * VEC;
}

template <int VEC, int NV>
__device__ __forceinline__ void stage_row_async(float* ring, int slot, const float* __restrict__ table, int64_t row,
                                                int D, int lane) {
    const float* p = table + row * (int64_t)D;
    float* s = stage_slot<VEC, NV>(ring, slot);
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int d0 = dim_of<VEC>(lane, j);
        if (d0 < D) cp_async<VEC * 4>(smem_addr(s + (size_t)j * BLOCK * VEC), p + d0);
    }
}

template <int VEC, int NV>
__device__ __forceinline__ void read_staged_row(Row<VEC, NV>& r, const float* ring, int slot, int D, int lane) {
    const float* s = stage_slot<VEC, NV>(const_cast<float*>(ring), slot);
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int d0 = dim_of<VEC>(lane, j);
        if (d0 < D) {
            ldv<VEC>(s + (size_t)j * BLOCK * VEC, &r.x[j * VEC]);
        } else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) r.x[j * VEC + v] = 0.f;
        }
    }
}

template <int VEC, int NV>
__device__ __forceinline__ void write_staged_row(const Row<VEC, NV>& r, float* ring, int slot, int D, int lane) {
    float* s = stage_slot<VEC, NV>(ring, slot);
#pragma unroll
    for (int j = 0; j < NV; ++j) {
        const int d0 = dim_of<VEC>(lane, j);
        if (d0 < D) stv<VEC>(s + (size_t)j * BLOCK * VEC, &r.x[j * VEC]);
    }
}

// sum over the 16 lanes of a group; every lane gets the result (xor butterfly stays inside the
// aligned half-warp)
__device__ __forceinline__ float group_sum(float v, unsigned mask) {
    v += __shfl_xor_sync(mask, v, 8);
    v += __shfl_xor_sync(mask, v, 4);
    v += __shfl_xor_sync(mask, v, 2);
    v += __shfl_xor_sync(mask, v, 1);
    return v;
}

// N sums at once (N = 2, 4, 8 or 16): every lane passes v[0..N-1] and gets back the 16-lane sum of v[k],
// k = lane / (16 / N).  At each level a lane keeps one half of its values and sends the other half to its
// partner (keep + received, the butterfly's own + partner), so the result is bitwise group_sum(v[k]) with
// N - 1 + log2(16 / N) shuffles instead of 4 N.
template <int N>
__device__ __forceinline__ float group_sum_scatter(float (&v)[N], int lane, unsigned mask) {
    static_assert(N == 2 || N == 4 || N == 8 || N == 16, "N must divide the group");
    int off = GROUP / 2;
#pragma unroll
    for (int n = N; n > 1; n >>= 1, off >>= 1) {
        const bool hi = (lane & off) != 0;
#pragma unroll
        for (int j = 0; j < n / 2; ++j) {
            const float keep = hi ? v[n / 2 + j] : v[j];
            const float send = hi ? v[j] : v[n / 2 + j];
            v[j] = keep + __shfl_xor_sync(mask, send, off);
        }
    }
    float x = v[0];
#pragma unroll
    for (int o = GROUP / (2 * N); o >= 1; o >>= 1) x += __shfl_xor_sync(mask, x, o);
    return x;
}

// all 32 lanes must be converged (used after the loops only)
__device__ __forceinline__ float warp_sum(float v) {
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    return group_sum(v, 0xffffffffu);
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

__device__ __forceinline__ float signf_(float x) { return (x > 0.f) ? 1.f : ((x < 0.f) ? -1.f : 0.f); }

// c * sign(x) with sign(0) = 0 (torch's norm(1) backward), three instructions
__device__ __forceinline__ float mul_sign(float c, float x) { return (x == 0.f) ? 0.f : copysignf(c, x); }

// Scalars of one dense torch.optim.Adam update (torch/optim/adam.py, single-tensor path):
// computed on the host in double from the integer step, used as fp32 in the tensor ops.
struct AdamScalars {
    float one_minus_b1, b2, one_minus_b2, step_size, bc2_sqrt, inv_bc2_sqrt, eps;
};

// MUFU.SQRT / MUFU.RCP, max rel. error 2^-23, ONE instruction each: the .ftz forms skip the subnormal pre-/post-scaling
// that the plain .approx forms expand to (5 and 4 instructions per element in the round-1 SASS, 13 % of the fused
// user pass).  Flushing is invisible here: sqrt of a subnormal v is < 1.1e-19, which vanishes against eps = 1e-8 in
// the fp32 sum, and the reciprocal's argument is >= eps.
__device__ __forceinline__ float sqrt_approx(float x) {
    float r;
    asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}

// exp_avg.lerp_(g, 1-b1); exp_avg_sq.mul_(b2).addcmul_(g, g, 1-b2);
// denom = sqrt(v)/sqrt(bc2) + eps; p.addcdiv_(m, denom, value=-lr/bc1)
// m and v (the state that carries over) use exactly torch's operations.  The step itself uses the
// hardware sqrt / reciprocal approximations (<= 3 ulp on the UPDATE, i.e. ~1e-7 * lr on the parameter):
// the IEEE sqrt + two divisions made the dense sweep issue-bound instead of HBM-bound (ncu, round 1).
__device__ __forceinline__ void adam_update(float& p, float& m, float& v, float g, const AdamScalars& s) {
    m = m + (g - m) * s.one_minus_b1;
    v = v * s.b2 + (s.one_minus_b2 * g) * g;
    const float denom = fmaf(sqrt_approx(v), s.inv_bc2_sqrt, s.eps);
    p = p - s.step_size * (m * rcp_approx(denom));
}

// The step-dependent Adam scalars come from the launch arguments or, for CUDA-graph replay, from a device record.
__device__ __forceinline__ AdamScalars with_dyn(AdamScalars s, const invpref_dyn* dyn) {
    if (dyn != nullptr) { s.step_size = dyn->step_size; s.inv_bc2_sqrt = dyn->inv_bc2_sqrt; }
    return s;
}

// One dense Adam step with ZERO gradient (what torch.optim.Adam does to a row that is not in the batch),
// with the bias-correction scalars of that step: used to replay skipped steps of lazily updated rows.
// It is adam_update with g = 0 written out (m + (0 - m) c = fma(-m, c, m); v b2 + 0 = v b2 since v >= 0), and
// it is what the dense sweep itself calls, so lazy replay and dense sweep are the same arithmetic by
// construction.
__device__ __forceinline__ void adam_zero_step(float& p, float& m, float& v, const AdamScalars& s, float step_size,
                                               float inv_bc2_sqrt) {
    m = fmaf(-m, s.one_minus_b1, m);
    v = v * s.b2;
    const float denom = fmaf(sqrt_approx(v), inv_bc2_sqrt, s.eps);
    p = fmaf(-step_size, m * rcp_approx(denom), p);
}

#endif  // __CUDACC__

}  // namespace invpref
