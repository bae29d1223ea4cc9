// Device-side helpers of the implicit evaluator (reference evaluate.py:94-135, SURVEY.md §8f rank 1).
//
// The reference builds, per test batch, python lists of (row, item) pairs from per-user python sets to mask the
// train positives (rating = -1024), highlight the item pool (+1024) and, after top-k, looks every predicted
// item up in the user's ground-truth set.  Here the per-user item lists live on the device once, as CSR over
// user ids (ascending items within a user), and two small kernels do the masking and the look-ups.
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
// Fused implicit evaluation of one test batch (evaluate.py:88-135 + models.py:393-407): score every item, mask the
// train positives, highlight the item pool, take the top k, look the hits up -- ONE kernel, no [b, I] rating matrix.
//
// One CTA per test user.  The score of item i is recomputed wherever it is needed (a D <= 256 dot product against
// the user row held in shared memory costs less than a round trip of the [b, I] matrix through HBM).  The k-th
// largest adjusted score is found exactly by a 3-pass radix select over the order-preserving integer image of the
// fp32 score (11 + 11 + 10 bits, shared-memory histogram); items above the threshold are taken as they come, items
// EQUAL to it in ascending item order (so the result does not depend on thread scheduling: ties go to the lowest
// item id), and the k survivors are ordered by (score descending, item ascending).
constexpr int EV_THREADS = 256;
constexpr int EV_MAXK = 256;

// Every NaN maps to the largest key, so that NaN scores rank above +inf as in torch.topk and tie with each other
// (lowest item id first) whatever their sign and payload; by its bits alone a NaN with the sign bit set would sort
// below -inf.  The explicit test is also what keeps a computed NaN on top at all: nvcc folds `b | 0x80000000u` of
// a float computed in this kernel into a negated absolute value, `FADD R, -|s|, -RZ` in the SASS, and that add
// turns a NaN into the canonical NaN 0x7fffffff -- the key of -0.0, just below +0 (exact for every other float).
__device__ __forceinline__ uint32_t order_key(float s) {      // ascending integer order == ascending float order
    const uint32_t b = __float_as_uint(s);
    if (s != s) return 0xffffffffu;
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

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

__device__ __forceinline__ bool in_sorted(const int64_t* __restrict__ items, int64_t lo, int64_t hi, int64_t want) {
    const int64_t end = hi;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (items[mid] < want) lo = mid + 1; else hi = mid;
    }
    return lo < end && items[lo] == want;
}

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

}  // namespace

int launch_eval_topk(const float* Uinv, const float* Iinv, int64_t n_items, int D, int implicit, const int64_t* users,
                     int64_t b, const int64_t* mask_off, const int64_t* mask_items, const int64_t* pool_off,
                     const int64_t* pool_items, const int64_t* gt_off, const int64_t* gt_items, int k,
                     int64_t* top_items, float* top_scores, uint8_t* hits, int64_t* n_gt, cudaStream_t stream) {
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

}  // namespace invpref
