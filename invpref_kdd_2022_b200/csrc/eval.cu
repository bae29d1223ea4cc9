// Device-side helpers of the implicit evaluator (reference evaluate.py:94-135, SURVEY.md §8f rank 1).
//
// The reference builds, per test batch, python lists of (row, item) pairs from per-user python sets to mask the
// train positives (rating = -1024), highlight the item pool (+1024) and, after top-k, looks every predicted
// item up in the user's ground-truth set.  Here the per-user item lists live on the device once, as CSR over
// user ids (ascending items within a user), and two small kernels do the masking and the look-ups.
#include <cooperative_groups.h>

#include "common.cuh"
#include "kernels.h"

namespace invpref {

namespace {

// one warp per batch row: rating[r, items(users[r])] = value  (add == 0)  or  += value  (add != 0)
__global__ void __launch_bounds__(256) mask_scores_kernel(float* __restrict__ rating, int64_t b, int64_t n_items,
                                                          const int64_t* __restrict__ users,
                                                          const int64_t* __restrict__ off,
                                                          const int64_t* __restrict__ items, float value, int add) {
    const int lane = threadIdx.x & 31;
    const int64_t warps = (int64_t)gridDim.x * (blockDim.x >> 5);
    for (int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); r < b; r += warps) {
        const int64_t u = users[r];
        const int64_t lo = off[u], hi = off[u + 1];
        float* row = rating + r * n_items;
        for (int64_t p = lo + lane; p < hi; p += 32) {
            const int64_t it = items[p];
            if (it >= 0 && it < n_items) {      // lists hold unique items: no two lanes touch the same element
                if (add) row[it] += value;
                else row[it] = value;
            }
        }
    }
}

// one thread per (row, rank): hits[r, j] = top[r, j] in items(users[r]) (binary search in the ascending list)
__global__ void __launch_bounds__(256) hits_from_csr_kernel(const int64_t* __restrict__ top, int64_t b, int k,
                                                            const int64_t* __restrict__ users,
                                                            const int64_t* __restrict__ off,
                                                            const int64_t* __restrict__ items,
                                                            uint8_t* __restrict__ hits, int64_t* __restrict__ n_list) {
    const int64_t total = b * k;
    for (int64_t q = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; q < total; q += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = q / k;
        const int64_t u = users[r];
        int64_t lo = off[u], hi = off[u + 1];
        if (q - r * k == 0 && n_list != nullptr) n_list[r] = hi - lo;
        const int64_t want = top[q];
        while (lo < hi) {
            const int64_t mid = (lo + hi) >> 1;
            if (items[mid] < want) lo = mid + 1; else hi = mid;
        }
        hits[q] = (lo < off[u + 1] && items[lo] == want) ? 1 : 0;
    }
}

// ---------------------------------------------------------------------------------------------------------
// Streaming top-k over a whole catalogue table for a batch of query rows -- ONE kernel, no [b, n] matrix:
//   the evaluator (invpref_eval_topk, EVAL mode: evaluate.py:88-135 + models.py:393-407): users against Iinv;
//   invpref_recommend (EXCLUDE mode): users against Iinv;  invpref_top_users (EXCLUDE mode): items against Uinv;
//   invpref_similar_items (EXCLUDE mode, COS): items against Iinv by cosine, the query row itself skipped.
// Below, "users" are the query rows and "items" the catalogue rows.
//
// A CTA owns a tile of TK_TU users (their rows in shared memory) and streams its item range in ascending tiles
// of TK_TI items.  The [TU, TI] block of dot products is a register micro-tile of 4 x 4 per thread, accumulated in
// ascending d with explicit fmaf from +0 (eval_topk_kernel's arithmetic: bit-identical scores in any tiling).  The item
// tile is staged with cp.async, double-buffered, in chunks of at most 32 dims (large D keeps TI and the d order).
//
// COS (a template parameter, so that the other modes compile exactly as without it): the query ids index the
// catalogue table itself and inv_norm holds 1 / |row| of every catalogue row (row_inv_norm_kernel).  The score is
// (z * inv_norm[q]) * inv_norm[i] + 0, rounded after each operation (the + 0 turns a -0 product into +0: one key
// for a zero cosine), with no sigmoid; the catalogue row equal to the query id is never a candidate.
//
// Exact streaming selection per user: a candidate buffer of C composites (order_key << 32 | ~item; C = 256 or 512 >= k + TK_TI), a count and
// a threshold T (start 0; every real score has a key >= 1).  An item is appended when key > T.  Before a tile that
// might overflow the buffer, one warp sorts it (bitonic, descending composite = key descending, item ascending),
// keeps the top k and sets T to the k-th key: a later item with key == T has a larger id, so it ranks below every
// kept item with that key -- dropping it is exact.
//
// With few users the item range is split over a thread-block cluster of S CTAs (one slice each, same user tile).
// Each CTA sorts its per-user lists; after cluster.sync() the CTAs place the S sorted lists of their share of the
// tile's users by rank (an element's rank = its index + the number of greater elements in the other S - 1 lists,
// binary searched through distributed shared memory) and write the results: no global workspace.
constexpr int TK_THREADS = 256;
constexpr int TK_TU = 32;            // users per CTA: 2 warp rows x 16
constexpr int TK_TI = 128;           // items per tile: 4 warp columns x 32
constexpr int TK_DC = 32;            // at most this many dims per staged chunk
constexpr int TK_MAX_SLICES = 8;

// Every NaN maps to the largest key, so that NaN scores rank above +inf as in torch.topk and tie with each other
// (lowest item id first) whatever their sign and payload; by its bits alone a NaN with the sign bit set would sort
// below -inf.  The explicit test is also what keeps a computed NaN on top at all: nvcc folds `b | 0x80000000u` of
// a float computed in this kernel into a negated absolute value, `FADD R, -|s|, -RZ` in the SASS, and that add
// turns a NaN into the canonical NaN 0x7fffffff -- the key of -0.0, just below +0 (exact for every other float).
// Every non-NaN float has a key >= 0x007fffff (-inf): key 0 is free.
__device__ __forceinline__ uint32_t order_key(float s) {      // ascending integer order == ascending float order
    const uint32_t b = __float_as_uint(s);
    if (s != s) return 0xffffffffu;
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__device__ __forceinline__ float key_score(uint32_t k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

struct TopkArgs {
    const float *Q, *X;               // query table, catalogue table
    const int64_t* qids;              // [b] rows of Q
    const float* inv_norm;            // COS: [n_rows] 1 / |X row| (Q == X)
    // EVAL: list 0 = mask (score := -1024), list 1 = pool (+= 1024).  EXCLUDE: list 0 = excluded items, no list 1.
    // Lists are CSR over query ids.
    const int64_t* off[2];
    const int64_t* items[2];
    const int64_t *gt_off, *gt_items;
    int64_t b, n_rows, slice;         // n_rows: catalogue rows; slice: catalogue rows per cluster rank
    int D, DUS, DC, DCS, nch, k, C, implicit, exclude, vec16;
    int64_t* top_items;
    float* top_scores;
    uint8_t* hits;
    int64_t* n_gt;
};

__device__ __forceinline__ bool in_sorted(const int64_t* __restrict__ items, int64_t lo, int64_t hi, int64_t want) {
    const int64_t end = hi;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (items[mid] < want) lo = mid + 1; else hi = mid;
    }
    return lo < end && items[lo] == want;
}

__device__ __forceinline__ int64_t lower_bound(const int64_t* __restrict__ items, int64_t lo, int64_t hi,
                                               int64_t want) {
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (items[mid] < want) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// One warp sorts buf[0, n) descending (bitonic over the next power of two >= n, padded with 0, below every
// candidate) and keeps the first min(n, k).  Returns the key of the k-th element when n >= k, else 0.
__device__ uint32_t warp_sort_keep(unsigned long long* buf, uint32_t* cnt, int k, int lane) {
    const int n = (int)*cnt;
    int m = 32;
    while (m < n) m <<= 1;
    for (int i = n + lane; i < m; i += 32) buf[i] = 0ull;
    __syncwarp();
    for (int size = 2; size <= m; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = lane; t < (m >> 1); t += 32) {
                const int i = ((t & ~(stride - 1)) << 1) | (t & (stride - 1));
                const int j = i + stride;
                const unsigned long long x = buf[i], y = buf[j];
                if ((x < y) == ((i & size) == 0)) { buf[i] = y; buf[j] = x; }
            }
            __syncwarp();
        }
    }
    const uint32_t T = n >= k ? (uint32_t)(buf[k - 1] >> 32) : 0u;
    __syncwarp();
    if (lane == 0) *cnt = (uint32_t)(n < k ? n : k);
    __syncwarp();
    return T;
}

// Fused implicit evaluation of one test batch on a SMALL item table (below EV_STREAM_MIN_ITEMS; larger ones go to
// topk_stream_kernel below): score every item, mask the train positives, highlight the item pool, take the top k,
// look the hits up -- ONE kernel, no [b, I] rating matrix.
//
// One CTA per test user.  The score of item i is recomputed wherever it is needed (a D <= 256 dot product against
// the user row held in shared memory costs less than a round trip of the [b, I] matrix through HBM).  The k-th
// largest adjusted score is found exactly by a 3-pass radix select over the order-preserving integer image of the
// fp32 score (11 + 11 + 10 bits, shared-memory histogram); items above the threshold are taken as they come, items
// EQUAL to it in ascending item order (so the result does not depend on thread scheduling: ties go to the lowest
// item id), and the k survivors are ordered by (score descending, item ascending).
constexpr int EV_THREADS = 256;
constexpr int EV_MAXK = 256;
constexpr int64_t EV_STREAM_MIN_ITEMS = 2048;

struct EvalArgs {
    const float *Uinv, *Iinv;
    const int64_t* users;
    const int64_t *mask_off, *mask_items, *pool_off, *pool_items, *gt_off, *gt_items;
    int64_t n_items;
    int D, k, implicit, use_bitmap, use_cache;
    int64_t* top_items;
    float* top_scores;
    uint8_t* hits;
    int64_t* n_gt;
};

__global__ void __launch_bounds__(EV_THREADS) eval_topk_kernel(EvalArgs a) {
    extern __shared__ __align__(16) unsigned char ev_smem[];
    float* sU = reinterpret_cast<float*>(ev_smem);                                   // [D padded to 4]
    uint32_t* sHist = reinterpret_cast<uint32_t*>(sU + ((a.D + 3) & ~3));            // [2048]
    uint32_t* sPart = sHist + 2048;                                                  // [256] partial sums
    uint32_t* sCandKey = sPart + EV_THREADS;                                         // [EV_MAXK]
    int32_t* sCandIdx = reinterpret_cast<int32_t*>(sCandKey + EV_MAXK);              // [EV_MAXK]
    uint32_t* sMaskBits = reinterpret_cast<uint32_t*>(sCandIdx + EV_MAXK);           // [words] (use_bitmap)
    const int words = a.use_bitmap ? (int)((a.n_items + 31) >> 5) : 0;
    uint32_t* sPoolBits = sMaskBits + words;
    float* sScore = reinterpret_cast<float*>(sPoolBits + words);                     // [n_items] (use_cache)
    __shared__ uint32_t sPrefix, sNeed, sCount, sBase;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int r = blockIdx.x;
    const int64_t u = a.users[r];
    const int D = a.D, k = a.k;
    const int64_t I = a.n_items;
    for (int d = tid; d < D; d += EV_THREADS) sU[d] = a.Uinv[u * D + d];
    const int64_t m_lo = a.mask_off ? a.mask_off[u] : 0, m_hi = a.mask_off ? a.mask_off[u + 1] : 0;
    const int64_t p_lo = a.pool_off ? a.pool_off[u] : 0, p_hi = a.pool_off ? a.pool_off[u + 1] : 0;
    if (a.use_bitmap) {
        for (int w = tid; w < 2 * words; w += EV_THREADS) sMaskBits[w] = 0u;
        __syncthreads();
        for (int64_t p = m_lo + tid; p < m_hi; p += EV_THREADS) {
            const int64_t it = a.mask_items[p];
            if (it >= 0 && it < I) atomicOr(&sMaskBits[it >> 5], 1u << (it & 31));
        }
        for (int64_t p = p_lo + tid; p < p_hi; p += EV_THREADS) {
            const int64_t it = a.pool_items[p];
            if (it >= 0 && it < I) atomicOr(&sPoolBits[it >> 5], 1u << (it & 31));
        }
    }
    __syncthreads();
    const bool vec4 = (D & 3) == 0;
    // adjusted score of item i: models.py:393-407 (sigmoid of the invariant dot product for the implicit model),
    // evaluate.py:98 (train positives := -1024), evaluate.py:110 (item pool += 1024)
    auto score = [&](int64_t i) -> float {
        const float* __restrict__ row = a.Iinv + i * D;
        float z = 0.f;
        if (vec4) {
            for (int d = 0; d < D; d += 4) {
                const float4 v = *reinterpret_cast<const float4*>(row + d);
                const float4 w = *reinterpret_cast<const float4*>(sU + d);
                z = fmaf(v.x, w.x, z); z = fmaf(v.y, w.y, z); z = fmaf(v.z, w.z, z); z = fmaf(v.w, w.w, z);
            }
        } else {
            for (int d = 0; d < D; ++d) z = fmaf(row[d], sU[d], z);
        }
        float s = a.implicit ? sigmoidf_(z) : z;
        bool masked, pooled;
        if (a.use_bitmap) {
            masked = (sMaskBits[i >> 5] >> (i & 31)) & 1u;
            pooled = (sPoolBits[i >> 5] >> (i & 31)) & 1u;
        } else {
            masked = m_hi > m_lo && in_sorted(a.mask_items, m_lo, m_hi, i);
            pooled = p_hi > p_lo && in_sorted(a.pool_items, p_lo, p_hi, i);
        }
        if (masked) s = -1024.f;
        if (pooled) s += 1024.f;
        return s;
    };

    // small item sets: every adjusted score is computed once and kept in shared memory; large ones (MIND: 51 K items)
    // recompute it in each of the five sweeps below
    if (a.use_cache) {
        for (int64_t i = tid; i < I; i += EV_THREADS) sScore[i] = score(i);
        __syncthreads();
    }
    auto get = [&](int64_t i) -> float { return a.use_cache ? sScore[i] : score(i); };

    // ---- exact k-th largest key: radix select, most significant digit first ----
    if (tid == 0) { sPrefix = 0u; sNeed = (uint32_t)k; }
    uint32_t known = 0u;                       // mask of the key bits fixed so far
    const int shifts[3] = {21, 10, 0}, bits[3] = {11, 11, 10};
    for (int pass = 0; pass < 3; ++pass) {
        const int shift = shifts[pass];
        const uint32_t nb = 1u << bits[pass];
        for (int b = tid; b < 2048; b += EV_THREADS) sHist[b] = 0u;
        __syncthreads();
        const uint32_t prefix = sPrefix;
        for (int64_t i = tid; i < I; i += EV_THREADS) {
            const uint32_t key = order_key(get(i));
            if ((key & known) == prefix) atomicAdd(&sHist[(key >> shift) & (nb - 1)], 1u);
        }
        __syncthreads();
        // bins from the top: the bin where the running count reaches `need`
        const int per = 2048 / EV_THREADS;                   // 8 bins per thread, thread 0 owns the highest bins
        uint32_t mine = 0u;
        for (int j = 0; j < per; ++j) {
            const int b = 2047 - (tid * per + j);
            mine += (b < (int)nb) ? sHist[b] : 0u;
        }
        sPart[tid] = mine;
        __syncthreads();
        if (tid == 0) {
            uint32_t need = sNeed, cum = 0u;
            int t = 0;
            for (; t < EV_THREADS; ++t) {
                if (cum + sPart[t] >= need) break;
                cum += sPart[t];
            }
            int b = 2047 - t * per;
            for (int j = 0; j < per; ++j, --b) {
                const uint32_t h = (b < (int)nb) ? sHist[b] : 0u;
                if (cum + h >= need) break;
                cum += h;
            }
            sNeed = need - cum;                               // still needed inside the chosen bin
            sPrefix = prefix | ((uint32_t)b << shift);
        }
        known |= (nb - 1) << shift;
        __syncthreads();
    }
    const uint32_t T = sPrefix;                               // key of the k-th largest adjusted score
    const uint32_t need_eq = sNeed;                           // how many items with key == T belong to the top k
    // ---- collect: keys above T as they come, keys equal to T in ascending item order ----
    if (tid == 0) { sCount = 0u; sBase = 0u; }
    __syncthreads();
    __shared__ uint32_t sWarpCnt[EV_THREADS / 32];
    for (int64_t i0 = 0; i0 < I; i0 += EV_THREADS) {
        const int64_t i = i0 + tid;
        uint32_t key = 0u;
        bool gt = false, eq = false;
        if (i < I) {
            key = order_key(get(i));
            gt = key > T;
            eq = key == T;
        }
        if (gt) {
            const uint32_t pos = atomicAdd(&sCount, 1u);
            sCandKey[pos] = key;
            sCandIdx[pos] = (int32_t)i;
        }
        // ordered selection among the equal keys: rank inside this stripe of 256 consecutive items
        const uint32_t bal = __ballot_sync(0xffffffffu, eq);
        if (lane == 0) sWarpCnt[warp] = __popc(bal);
        __syncthreads();
        uint32_t before = sBase;
        for (int w = 0; w < warp; ++w) before += sWarpCnt[w];
        const uint32_t rank = before + __popc(bal & ((1u << lane) - 1u));
        if (eq && rank < need_eq) {
            const uint32_t pos = (uint32_t)k - need_eq + rank;        // the equal keys fill the tail of the list
            sCandKey[pos] = key;
            sCandIdx[pos] = (int32_t)i;
        }
        __syncthreads();
        if (tid == 0) {
            uint32_t tot = 0u;
            for (int w = 0; w < EV_THREADS / 32; ++w) tot += sWarpCnt[w];
            sBase += tot;
        }
        __syncthreads();
    }
    __syncthreads();
    // ---- order the k survivors: (key descending, item ascending); one thread per survivor ----
    if (tid < k) {
        const uint32_t mk = sCandKey[tid];
        const int32_t mi = sCandIdx[tid];
        int pos = 0;
        for (int j = 0; j < k; ++j) {
            const uint32_t ok = sCandKey[j];
            const int32_t oi = sCandIdx[j];
            pos += (ok > mk || (ok == mk && oi < mi)) ? 1 : 0;
        }
        a.top_items[(int64_t)r * k + pos] = (int64_t)mi;
        if (a.top_scores != nullptr) {
            const uint32_t kb = (mk & 0x80000000u) ? (mk & 0x7fffffffu) : ~mk;
            a.top_scores[(int64_t)r * k + pos] = __uint_as_float(kb);
        }
        if (a.hits != nullptr) {
            const int64_t g_lo = a.gt_off[u], g_hi = a.gt_off[u + 1];
            a.hits[(int64_t)r * k + pos] = in_sorted(a.gt_items, g_lo, g_hi, (int64_t)mi) ? 1 : 0;
        }
    }
    if (tid == 0 && a.n_gt != nullptr) a.n_gt[r] = a.gt_off ? a.gt_off[u + 1] - a.gt_off[u] : 0;
}

template <bool COS>
__global__ void __launch_bounds__(TK_THREADS, 2) topk_stream_kernel(TopkArgs a) {
    extern __shared__ __align__(128) unsigned char tk_smem[];
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    const int S = (int)cluster.num_blocks(), rank = (int)cluster.block_rank();
    float* sRing = reinterpret_cast<float*>(tk_smem);                                       // [2][TI][DCS]
    float* sU = sRing + ring_align_up(2 * TK_TI * a.DCS);                                     // [TU][DUS]
    unsigned long long* sBuf = reinterpret_cast<unsigned long long*>(sU + ring_align_up(TK_TU * a.DUS));  // [TU][C]
    uint32_t* sBits = reinterpret_cast<uint32_t*>(sBuf + (size_t)TK_TU * a.C);              // [2][TU][TI / 32]
    int64_t* sQid = reinterpret_cast<int64_t*>(sBits + 2 * TK_TU * (TK_TI / 32));           // COS: [TU]
    float* sQn = reinterpret_cast<float*>(sQid + TK_TU);                                     // COS: [TU]
    __shared__ uint32_t sCnt[TK_TU], sT[TK_TU];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t row0 = (int64_t)(blockIdx.x / S) * TK_TU;
    const int rows = (int)(a.b - row0 < TK_TU ? a.b - row0 : TK_TU);
    const int D = a.D, C = a.C, k = a.k;
    const int64_t lo = (int64_t)rank * a.slice;
    const int64_t hi = lo + a.slice < a.n_rows ? lo + a.slice : a.n_rows;
    const int64_t n_tiles = hi > lo ? (hi - lo + TK_TI - 1) / TK_TI : 0;
    const int nsteps = (int)n_tiles * a.nch;

    // ---- item tile staging: step s = (tile s / nch, dims [c * DC, min(D, c * DC + DC)) with c = s % nch) ----
    auto stage = [&](int s) {
        const int64_t i0 = lo + (int64_t)(s / a.nch) * TK_TI;
        const int d0 = (s % a.nch) * a.DC;
        const int w = D - d0 < a.DC ? D - d0 : a.DC;
        const int nr = (int)(hi - i0 < TK_TI ? hi - i0 : TK_TI);
        float* dst = sRing + (size_t)(s & 1) * TK_TI * a.DCS;
        const float* src = a.X + i0 * D + d0;
        if (a.vec16) {
            const int q = w >> 2;
            for (int p = tid; p < nr * q; p += TK_THREADS) {
                const int r = p / q, c = p - r * q;
                cp_async<16>(smem_addr(dst + r * a.DCS + 4 * c), src + (int64_t)r * D + 4 * c);
            }
        } else {
            for (int p = tid; p < nr * w; p += TK_THREADS) {
                const int r = p / w, c = p - r * w;
                cp_async<4>(smem_addr(dst + r * a.DCS + c), src + (int64_t)r * D + c);
            }
        }
    };
    if (nsteps > 0) stage(0);
    cp_async_commit();

    // ---- user rows, counters, list cursors (cursor p = list p / TU of user row p % TU) ----
    __shared__ int64_t sCur[2 * TK_TU], sEnd[2 * TK_TU];
    for (int p = tid; p < TK_TU * a.DUS; p += TK_THREADS) {
        const int r = p / a.DUS, d = p - r * a.DUS;
        sU[p] = (r < rows && d < D) ? a.Q[a.qids[row0 + r] * D + d] : 0.f;
    }
    if (tid < TK_TU) { sCnt[tid] = 0u; sT[tid] = 0u; }
    if (COS && tid < TK_TU) {
        const int64_t q = tid < rows ? a.qids[row0 + tid] : -1;
        sQid[tid] = q;
        sQn[tid] = q >= 0 ? a.inv_norm[q] : 0.f;
    }
    if (tid < 2 * TK_TU) {
        const int l = tid / TK_TU, r = tid % TK_TU;
        int64_t cur = 0, end = 0;
        if (a.items[l] != nullptr && r < rows) {
            const int64_t u = a.qids[row0 + r];
            end = a.off[l][u + 1];
            cur = lower_bound(a.items[l], a.off[l][u], end, lo);
        }
        sCur[tid] = cur;
        sEnd[tid] = end;
    }

    const int wu = warp >> 2, wi = warp & 3, lu = lane >> 3, li = lane & 7;
    const int ur = wu * 16 + lu;        // this thread's users: ur + 4 j
    const int ir = wi * 32 + li;        // this thread's tile items: ir + 8 j
    float acc[4][4];
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) acc[x][y] = 0.f;

    for (int s = 0; s < nsteps; ++s) {
        if (s + 1 < nsteps) stage(s + 1);
        cp_async_commit();
        cp_async_wait<1>();
        __syncthreads();
        {
            const float* sI = sRing + (size_t)(s & 1) * TK_TI * a.DCS;
            const int d0 = (s % a.nch) * a.DC;
            const int w = D - d0 < a.DC ? D - d0 : a.DC;
            const float* pu = sU + ur * a.DUS + d0;
            const float* pi = sI + ir * a.DCS;
            const int w4 = w >> 2;
            for (int q = 0; q < w4; ++q) {
                float4 uv[4], iv[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) uv[j] = *reinterpret_cast<const float4*>(pu + 4 * j * a.DUS + 4 * q);
#pragma unroll
                for (int j = 0; j < 4; ++j) iv[j] = *reinterpret_cast<const float4*>(pi + 8 * j * a.DCS + 4 * q);
#pragma unroll
                for (int x = 0; x < 4; ++x)
#pragma unroll
                    for (int y = 0; y < 4; ++y) {
                        float z = acc[x][y];
                        z = fmaf(iv[y].x, uv[x].x, z); z = fmaf(iv[y].y, uv[x].y, z);
                        z = fmaf(iv[y].z, uv[x].z, z); z = fmaf(iv[y].w, uv[x].w, z);
                        acc[x][y] = z;
                    }
            }
            for (int d = 4 * w4; d < w; ++d) {
#pragma unroll
                for (int x = 0; x < 4; ++x)
#pragma unroll
                    for (int y = 0; y < 4; ++y) acc[x][y] = fmaf(pi[8 * y * a.DCS + d], pu[4 * x * a.DUS + d], acc[x][y]);
            }
        }
        if (s % a.nch == a.nch - 1) {
            const int64_t i0 = lo + (int64_t)(s / a.nch) * TK_TI;
            __syncthreads();
            // list entries inside [i0, i0 + TI) -> tile bits (merge-join: the cursors only move forward); one warp
            // per cursor reads 32 consecutive entries at a time, the entries below i0 + TI being a prefix of them
            for (int p = warp; p < 2 * TK_TU; p += TK_THREADS / 32) {
                uint32_t* bits = sBits + p * (TK_TI / 32);
                if (lane < TK_TI / 32) bits[lane] = 0u;
                __syncwarp();
                const int64_t* items = a.items[p / TK_TU];
                const int64_t i1 = i0 + TK_TI, end = sEnd[p];
                int64_t cur = sCur[p];
                while (cur < end) {
                    const int64_t it = cur + lane < end ? items[cur + lane] : i1;
                    const bool in = it < i1;
                    if (in && it >= i0) atomicOr(&bits[(it - i0) >> 5], 1u << ((it - i0) & 31));
                    const int n = __popc(__ballot_sync(0xffffffffu, in));
                    cur += n;
                    if (n < 32) break;
                }
                if (lane == 0) sCur[p] = cur;
            }
            // buffers that this tile might overflow: reduce to the top k, raise T
            for (int r = warp; r < rows; r += TK_THREADS / 32)
                if ((int)sCnt[r] > C - TK_TI) {
                    const uint32_t T = warp_sort_keep(sBuf + (size_t)r * C, &sCnt[r], k, lane);
                    if (lane == 0) sT[r] = T;
                }
            __syncthreads();
            float inv_i[4];                 // COS: 1 / |row| of this thread's four tile items
            if (COS) {
#pragma unroll
                for (int y = 0; y < 4; ++y) inv_i[y] = i0 + ir + 8 * y < hi ? a.inv_norm[i0 + ir + 8 * y] : 0.f;
            }
#pragma unroll
            for (int x = 0; x < 4; ++x) {
                const int r = ur + 4 * x;
                const uint32_t T = sT[r];
#pragma unroll
                for (int y = 0; y < 4; ++y) {
                    const int c = ir + 8 * y;
                    const int64_t item = i0 + c;
                    const float z = acc[x][y];
                    acc[x][y] = 0.f;
                    if (r >= rows || item >= hi) continue;
                    float sc;
                    if (COS) {
                        if (item == sQid[r]) continue;
                        sc = __fadd_rn(__fmul_rn(__fmul_rn(z, sQn[r]), inv_i[y]), 0.f);   // never contracted
                    } else {
                        const bool in0 = (sBits[r * (TK_TI / 32) + (c >> 5)] >> (c & 31)) & 1u;
                        if (a.exclude && in0) continue;
                        sc = a.implicit ? sigmoidf_(z) : z;
                        if (!a.exclude) {
                            if (in0) sc = -1024.f;
                            if ((sBits[(TK_TU + r) * (TK_TI / 32) + (c >> 5)] >> (c & 31)) & 1u) sc += 1024.f;
                        }
                    }
                    const uint32_t key = order_key(sc);
                    if (key > T) {
                        const uint32_t pos = atomicAdd(&sCnt[r], 1u);
                        // item < n_items < 2^31 (make_geometry): ~item in the low 32 bits ranks lower ids first
                        sBuf[(size_t)r * C + pos] = ((unsigned long long)key << 32) | (uint32_t)~(uint32_t)item;
                    }
                }
            }
        }
        __syncthreads();
    }
    cp_async_wait<0>();

    // ---- per-slice sorted lists, then the ranked merge over the cluster ----
    for (int r = warp; r < rows; r += TK_THREADS / 32) warp_sort_keep(sBuf + (size_t)r * C, &sCnt[r], k, lane);
    cluster.sync();
    const int share = TK_TU / S;
    for (int r = rank * share; r < (rank + 1) * share && r < rows; ++r) {
        const int64_t row = row0 + r;
        const int64_t u = a.qids[row];
        int total = 0;
        for (int j = 0; j < S; ++j) total += (int)*cluster.map_shared_rank(&sCnt[r], j);
        for (int e = tid; e < S * k; e += TK_THREADS) {
            const int j = e / k, p = e - j * k;
            const unsigned long long* L = cluster.map_shared_rank(sBuf, j) + (size_t)r * C;
            if (p >= (int)*cluster.map_shared_rank(&sCnt[r], j)) continue;
            const unsigned long long x = L[p];
            int pos = p;
            for (int o = 0; o < S && pos < k; ++o) {
                if (o == j) continue;
                const unsigned long long* M = cluster.map_shared_rank(sBuf, o) + (size_t)r * C;
                int l = 0, h = (int)*cluster.map_shared_rank(&sCnt[r], o);
                while (l < h) {
                    const int mid = (l + h) >> 1;
                    if (M[mid] > x) l = mid + 1; else h = mid;
                }
                pos += l;
            }
            if (pos >= k) continue;
            const int64_t item = (int64_t)(uint32_t)~(uint32_t)x;
            a.top_items[row * k + pos] = item;
            if (a.top_scores != nullptr) a.top_scores[row * k + pos] = key_score((uint32_t)(x >> 32));
            if (a.hits != nullptr)
                a.hits[row * k + pos] = in_sorted(a.gt_items, a.gt_off[u], a.gt_off[u + 1], item) ? 1 : 0;
        }
        for (int p = total + tid; p < k; p += TK_THREADS) {        // EXCLUDE / COS: fewer than k eligible items
            a.top_items[row * k + p] = -1;
            a.top_scores[row * k + p] = -__int_as_float(0x7f800000);
        }
        if (tid == 0 && a.n_gt != nullptr) a.n_gt[row] = a.gt_off[u + 1] - a.gt_off[u];
    }
    cluster.sync();                      // no CTA exits while a peer may still read its shared memory
}

// One thread per row: inv_norm[i] = 1 / sqrtf(n2), n2 = sum over d of x[d] * x[d] as one fmaf per d in ascending d
// from +0 (the order of the dot products above), IEEE sqrtf and division.  n2 == 0 gives 0, +inf (a non-finite
// entry, or a sum that overflows fp32) gives 1 / inf = 0, NaN gives NaN.
__global__ void __launch_bounds__(256) row_inv_norm_kernel(const float* __restrict__ x, int64_t n, int D, int vec4,
                                                           float* __restrict__ inv_norm) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float* __restrict__ row = x + i * D;
        float n2 = 0.f;
        if (vec4) {
            for (int d = 0; d < D; d += 4) {
                const float4 v = *reinterpret_cast<const float4*>(row + d);
                n2 = fmaf(v.x, v.x, n2); n2 = fmaf(v.y, v.y, n2); n2 = fmaf(v.z, v.z, n2); n2 = fmaf(v.w, v.w, n2);
            }
        } else {
            for (int d = 0; d < D; ++d) n2 = fmaf(row[d], row[d], n2);
        }
        inv_norm[i] = n2 == 0.f ? 0.f : 1.f / sqrtf(n2);
    }
}

template <bool COS>
int launch_topk_stream_impl(TopkArgs& a, cudaStream_t stream) {
    const int64_t b = a.b, n_rows = a.n_rows;
    const size_t smem = (size_t)ring_align_up(2 * TK_TI * a.DCS) * 4 + (size_t)ring_align_up(TK_TU * a.DUS) * 4 +
                        (size_t)TK_TU * a.C * 8 + 2 * TK_TU * (TK_TI / 32) * 4 + (COS ? TK_TU * (8 + 4) : 0);
    INVPREF_SET_SMEM_ONCE(topk_stream_kernel<COS>, smem);
    // cluster size: the slice count (1, 2, 4, 8; every slice at least one item tile) that fills the resident CTA
    // slots best, the smaller one on a tie
    // resident CTAs per SM for each shared-memory size seen (a few: D and k decide it), queried once each; one
    // process drives one GPU
    static int n_sm = 0;
    static size_t occ_smem[16];
    static int occ_ctas[16], n_occ = 0;
    if (n_sm == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
    }
    int per_sm = 0;
    for (int j = 0; j < n_occ && per_sm == 0; ++j)
        if (occ_smem[j] == smem) per_sm = occ_ctas[j];
    if (per_sm == 0) {
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, topk_stream_kernel<COS>, TK_THREADS, smem);
        per_sm = per_sm > 0 ? per_sm : 1;
        if (n_occ < 16) { occ_smem[n_occ] = smem; occ_ctas[n_occ] = per_sm; ++n_occ; }
    }
    const int64_t slots = (int64_t)(n_sm > 0 ? n_sm : 148) * per_sm;
    const int64_t tiles = (b + TK_TU - 1) / TK_TU;
    int S = 1;
    double best = 0.0;
    for (int s = 1; s <= TK_MAX_SLICES && (s == 1 || n_rows >= (int64_t)s * TK_TI); s *= 2) {
        const int64_t ctas = tiles * s;
        const double fill = (double)ctas / (double)(((ctas + slots - 1) / slots) * slots);
        if (fill > best + 1e-9) { best = fill; S = s; }
    }
    a.slice = (n_rows + S - 1) / S;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(tiles * S));
    cfg.blockDim = dim3(TK_THREADS);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)S;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t e = cudaLaunchKernelEx(&cfg, topk_stream_kernel<COS>, a);
    count_launch();
    return (e == cudaSuccess && cudaGetLastError() == cudaSuccess) ? INVPREF_OK : INVPREF_ERR_CUDA;
}

}  // namespace

int launch_topk_stream(const float* Q, const int64_t* qids, int64_t b, const float* X, int64_t n_rows, int D,
                       int implicit, const float* inv_norm, const int64_t* list0_off, const int64_t* list0_items,
                       const int64_t* list1_off, const int64_t* list1_items, int exclude, const int64_t* gt_off,
                       const int64_t* gt_items, int k, int64_t* top_items, float* top_scores, uint8_t* hits,
                       int64_t* n_gt, cudaStream_t stream) {
    TopkArgs a;
    a.Q = Q; a.X = X; a.qids = qids; a.inv_norm = inv_norm;
    a.off[0] = list0_items ? list0_off : nullptr; a.items[0] = list0_off ? list0_items : nullptr;
    a.off[1] = list1_items ? list1_off : nullptr; a.items[1] = list1_off ? list1_items : nullptr;
    a.gt_off = gt_off; a.gt_items = gt_items;
    a.b = b; a.n_rows = n_rows; a.D = D; a.k = k; a.implicit = implicit; a.exclude = exclude;
    a.top_items = top_items; a.top_scores = top_scores; a.hits = hits; a.n_gt = n_gt;
    // float4 reads need a row stride of 4 floats; a stride / 4 that is odd puts the 8 rows one LDS.128 of a warp
    // reads on 8 different 16-byte bank groups
    const int DP = (D + 3) & ~3;
    auto odd4 = [](int w) { return ((w >> 2) & 1) ? w : w + 4; };
    a.DUS = odd4(DP);
    a.nch = (DP + TK_DC - 1) / TK_DC;
    a.DC = ((DP + a.nch - 1) / a.nch + 3) & ~3;
    a.DCS = odd4(a.DC);
    a.vec16 = (D % 4 == 0 && ((uintptr_t)X & 15) == 0) ? 1 : 0;
    a.C = k + TK_TI <= 256 ? 256 : 512;                  // a power of two >= k + TI
    return inv_norm ? launch_topk_stream_impl<true>(a, stream) : launch_topk_stream_impl<false>(a, stream);
}

int launch_row_inv_norm(const float* x, int64_t n, int D, float* inv_norm, cudaStream_t stream) {
    const int64_t need = (n + 255) / 256;
    const int grid = (int)(need < 1 ? 1 : (need < 148 * 16 ? need : 148 * 16));
    const int vec4 = (D % 4 == 0 && ((uintptr_t)x & 15) == 0) ? 1 : 0;
    row_inv_norm_kernel<<<grid, 256, 0, stream>>>(x, n, D, vec4, inv_norm);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_mask_scores(float* rating, int64_t b, int64_t n_items, const int64_t* users, const int64_t* off,
                       const int64_t* items, float value, int add, cudaStream_t stream) {
    int64_t need = (b + 7) / 8;
    int grid = (int)(need < 1 ? 1 : (need < 148 * 8 ? need : 148 * 8));
    mask_scores_kernel<<<grid, 256, 0, stream>>>(rating, b, n_items, users, off, items, value, add);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_hits_from_csr(const int64_t* top, int64_t b, int k, const int64_t* users, const int64_t* off,
                         const int64_t* items, uint8_t* hits, int64_t* n_list, cudaStream_t stream) {
    int64_t need = (b * k + 255) / 256;
    int grid = (int)(need < 1 ? 1 : (need < 148 * 8 ? need : 148 * 8));
    hits_from_csr_kernel<<<grid, 256, 0, stream>>>(top, b, k, users, off, items, hits, n_list);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int launch_eval_topk(const float* Uinv, const float* Iinv, int64_t n_items, int D, int implicit, const int64_t* users,
                     int64_t b, const int64_t* mask_off, const int64_t* mask_items, const int64_t* pool_off,
                     const int64_t* pool_items, const int64_t* gt_off, const int64_t* gt_items, int k,
                     int64_t* top_items, float* top_scores, uint8_t* hits, int64_t* n_gt, cudaStream_t stream) {
    // Below EV_STREAM_MIN_ITEMS items a user's scores fit one CTA's shared memory and one CTA per user is the faster
    // kernel (Yahoo-implicit: 1 000 items, b = 1 024); from there on the user tiles' shared item reads win
    // (MovieLens: 3 706 items, MIND: 51 283; profiles/r3_topk_stream*.json).  Both give the same results.
    if (n_items >= EV_STREAM_MIN_ITEMS)
        return launch_topk_stream(Uinv, users, b, Iinv, n_items, D, implicit, nullptr, mask_off, mask_items,
                                  pool_off, pool_items, 0, gt_off, gt_items, k, top_items, top_scores, hits, n_gt,
                                  stream);
    EvalArgs a;
    a.Uinv = Uinv; a.Iinv = Iinv; a.users = users; a.mask_off = mask_off; a.mask_items = mask_items;
    a.pool_off = pool_off; a.pool_items = pool_items; a.gt_off = gt_off; a.gt_items = gt_items;
    a.n_items = n_items; a.D = D; a.k = k; a.implicit = implicit;
    a.top_items = top_items; a.top_scores = top_scores; a.hits = hits; a.n_gt = n_gt;
    const size_t words = (size_t)((n_items + 31) / 32);
    size_t base = (size_t)((D + 3) & ~3) * 4 + 2048 * 4 + EV_THREADS * 4 + EV_MAXK * 8;
    a.use_bitmap = (base + 2 * words * 4 <= 200 * 1024) ? 1 : 0;      // else: binary search in the sorted lists
    if (a.use_bitmap) base += 2 * words * 4;
    a.use_cache = (base + (size_t)n_items * 4 <= 200 * 1024) ? 1 : 0; // else: scores are recomputed per sweep
    const size_t smem = base + (a.use_cache ? (size_t)n_items * 4 : 0);
    INVPREF_SET_SMEM_ONCE(eval_topk_kernel, 200 * 1024);
    eval_topk_kernel<<<(unsigned)b, EV_THREADS, smem, stream>>>(a);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

}  // namespace invpref
