// numpy's legacy global stream (RandomState / MT19937) continued on the device, bit for bit.
//
// np.random.randint(0, high, n) with 1 <= high <= 2^32 takes one tempered MT19937 word w per attempt and accepts
// w & mask when it is <= high - 1 (mask = 2^bitlen(high - 1) - 1: masked rejection); high == 1 takes no word.  The
// reference draws its initial environments (train.py:711) and its tie-break rows (train.py:870-871) this way.  On the
// host the stream costs ~10 ns per sample; here it is split into segments that run in parallel:
//
//   * One twist of the 624-word key is a linear map T over GF(2)^19968.  Row k of the matrix A_1 is T(e_k) (a twisted
//     unit vector), so that the key as a row vector s gives T(s) = s A_1 (XOR of the rows of the set bits).  The jump
//     table holds A_{S0 2^i} = T^{S0 2^i} for i < MT_NJUMPS, each by squaring the one before (49.8 MB each).
//   * A round of G segments of S = S0 2^a blocks: start states s_g = T^{gS}(base) for g = 0..G come out of
//     ceil(log2 G) batched row-vector products, level j computing s_{2^j + g} = s_g A_{S 2^j} for all g < 2^j at once.
//   * Count pass: each segment (one CTA, the block in shared memory) twists S times in the three dependent sub-ranges
//     of numpy's twist, tempers, masks and counts acceptances.  A one-CTA exclusive scan gives each segment its first
//     rank; a write pass regenerates the words and stores every accepted value at its rank (segments that start at or
//     past n return at once).  The CTA that places value n-1 writes the key of its block and pos = index + 1.
//   * Rounds are sized from the expected number of words.  Whatever is still missing after the last round (the
//     count fell short) is produced by one CTA continuing sequentially from the round's end state, so exactness never
//     depends on a size margin.
#include <cmath>

#include "common.cuh"

namespace invpref {

namespace {

constexpr int MT_N = 624, MT_M = 397;
constexpr uint32_t MT_MATRIX_A = 0x9908b0dfu, MT_UPPER = 0x80000000u, MT_LOWER = 0x7fffffffu;
constexpr int MT_BITS = MT_N * 32;                    // 19 968: the key as a GF(2) vector
constexpr size_t MT_MAT_WORDS = (size_t)MT_BITS * MT_N;
constexpr int MT_THREADS = 640;                       // one thread per key word (20 warps)
constexpr int MT_S0_LOG = 3;                          // smallest segment: S0 = 8 blocks
constexpr int MT_A_MAX = 4;                           // largest segment: S0 * 2^4 = 128 blocks
constexpr int MT_J_MAX = 8;                           // 2^8 <= G < 2^9 segments per round
constexpr int MT_NJUMPS = MT_A_MAX + MT_J_MAX + 1;    // A_{8}, A_{16}, ..., A_{32768}: 13 matrices
constexpr int MT_GMAX = (1 << (MT_J_MAX + 1)) - 1;   // 511
constexpr int GF_W = 128;                             // words of a product tile
constexpr int GF_THREADS = 256;

__device__ __forceinline__ uint32_t mt_mag(uint32_t a, uint32_t b) {
    const uint32_t y = (a & MT_UPPER) | (b & MT_LOWER);
    return (y >> 1) ^ ((y & 1u) ? MT_MATRIX_A : 0u);
}

__device__ __forceinline__ uint32_t mt_temper(uint32_t y) {
    y ^= y >> 11;
    y ^= (y << 7) & 0x9d2c5680u;
    y ^= (y << 15) & 0xefc60000u;
    return y ^ (y >> 18);
}

// numpy's mt19937_gen (in place) as cur -> nxt, in its three dependent sub-ranges: i < 227 reads cur only, i < 454
// reads nxt[i - 227] of the first range, the rest (i = 623 last: nxt[0], nxt[396]) of the second.
__device__ __forceinline__ void mt_twist(const uint32_t* cur, uint32_t* nxt, int t) {
    if (t < MT_N - MT_M) nxt[t] = cur[t + MT_M] ^ mt_mag(cur[t], cur[t + 1]);
    __syncthreads();
    if (t >= MT_N - MT_M && t < 2 * (MT_N - MT_M)) nxt[t] = nxt[t - (MT_N - MT_M)] ^ mt_mag(cur[t], cur[t + 1]);
    __syncthreads();
    if (t >= 2 * (MT_N - MT_M) && t < MT_N - 1) nxt[t] = nxt[t - (MT_N - MT_M)] ^ mt_mag(cur[t], cur[t + 1]);
    else if (t == MT_N - 1) nxt[t] = nxt[MT_M - 1] ^ mt_mag(cur[t], nxt[0]);
    __syncthreads();
}

// Row k of A_1: the twist of unit vector e_k.
__global__ void __launch_bounds__(MT_THREADS) mt_unit_twist_kernel(uint32_t* __restrict__ A) {
    __shared__ uint32_t cur[MT_N + 1], nxt[MT_N];
    const int t = threadIdx.x, k = blockIdx.x;
    if (t < MT_N) cur[t] = (t == (k >> 5)) ? (1u << (k & 31)) : 0u;
    __syncthreads();
    mt_twist(cur, nxt, t);
    if (t < MT_N) A[(size_t)k * MT_N + t] = nxt[t];
}

// Y[b, :] ^= XOR over bits k of X[b, :] in [kw0 * 32, kw1 * 32) of A[k, :]  (b < B; rows of 624 words).
// A CTA owns 16 RB rows x 128 words of Y and one k range (blockIdx.z); partial products meet in Y by atomicXor (GF(2)
// addition: order-free), so Y must be zeroed first.  Thread (bg, wg) holds rows bg + 16 r and words wg + 16 q.
template <int RB>
__global__ void __launch_bounds__(GF_THREADS) gf2_mul_kernel(const uint32_t* __restrict__ X, int B,
                                                             const uint32_t* __restrict__ A, uint32_t* __restrict__ Y,
                                                             int kw_per_split) {
    __shared__ uint32_t sA[32][GF_W];
    __shared__ uint32_t sX[16 * RB];
    const int tid = threadIdx.x, bg = tid >> 4, wg = tid & 15;
    const int b0 = blockIdx.x * 16 * RB, w0 = blockIdx.y * GF_W;
    const int kw0 = blockIdx.z * kw_per_split, kw1 = min(MT_N, kw0 + kw_per_split);
    uint32_t acc[RB][8];
#pragma unroll
    for (int r = 0; r < RB; ++r)
#pragma unroll
        for (int q = 0; q < 8; ++q) acc[r][q] = 0u;
    for (int kw = kw0; kw < kw1; ++kw) {
        if (tid < 16 * RB) sX[tid] = (b0 + tid < B) ? X[(size_t)(b0 + tid) * MT_N + kw] : 0u;
        for (int e = tid; e < 32 * GF_W; e += GF_THREADS) {
            const int j = e / GF_W, c = e % GF_W;
            sA[j][c] = (w0 + c < MT_N) ? A[(size_t)(kw * 32 + j) * MT_N + w0 + c] : 0u;
        }
        __syncthreads();
        uint32_t x[RB];
#pragma unroll
        for (int r = 0; r < RB; ++r) x[r] = sX[bg + 16 * r];
#pragma unroll 4
        for (int j = 0; j < 32; ++j) {
            uint32_t m[RB];
#pragma unroll
            for (int r = 0; r < RB; ++r) m[r] = (uint32_t)((int32_t)(x[r] << (31 - j)) >> 31);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const uint32_t a = sA[j][wg + 16 * q];
#pragma unroll
                for (int r = 0; r < RB; ++r) acc[r][q] ^= m[r] & a;
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < RB; ++r) {
        const int b = b0 + bg + 16 * r;
        if (b >= B) continue;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            const int w = w0 + wg + 16 * q;
            if (w < MT_N && acc[r][q]) atomicXor(&Y[(size_t)b * MT_N + w], acc[r][q]);
        }
    }
}

struct MtDraw {
    uint32_t rng, mask;     // high - 1, 2^bitlen(high - 1) - 1
    int64_t n;
    int64_t* out;
    uint32_t* key_out;
    int32_t* pos_out;
};

// One segment per CTA: state states[g] with words [off, 624) unconsumed (off = off0 for g == 0, else 624), then up to
// S twisted blocks.  COUNT: counts[g] = acceptances.  Otherwise: write acceptances from rank first[g] on (stop at n);
// the block holding value n - 1 also writes key_out / pos_out.  S < 0: no block limit (the sequential tail).
template <bool COUNT>
__global__ void __launch_bounds__(MT_THREADS, 3) mt_segment_kernel(const uint32_t* __restrict__ states, int off0,
                                                                   int S, MtDraw d, int32_t* __restrict__ counts,
                                                                   const int64_t* __restrict__ first) {
    __shared__ uint32_t buf[2][MT_N + 1];
    __shared__ int sm[33];
    const int t = threadIdx.x, g = blockIdx.x;
    int64_t rank = COUNT ? 0 : first[g];
    if (!COUNT && rank >= d.n) return;
    if (t < MT_N) buf[0][t] = states[(size_t)g * MT_N + t];
    __syncthreads();
    int off = g == 0 ? off0 : MT_N, cnt = 0, c = 0;
    for (int blk = 0;; ++blk) {
        const uint32_t* cur = buf[c];
        const uint32_t v = (t < MT_N) ? (mt_temper(cur[t]) & d.mask) : 0u;
        const int acc = (t >= off && t < MT_N && v <= d.rng) ? 1 : 0;
        if (COUNT) {
            cnt += __syncthreads_count(acc);
        } else {
            int total;
            const int64_t r = rank + block_exclusive_scan(acc, &total, sm);
            if (acc && r < d.n) d.out[r] = (int64_t)v;
            if (rank < d.n && rank + total >= d.n) {          // this block holds value n - 1: numpy's state after it
                if (t < MT_N) d.key_out[t] = cur[t];
                if (acc && r == d.n - 1) *d.pos_out = t + 1;
                return;
            }
            rank += total;
        }
        if (blk == S) break;
        mt_twist(cur, buf[c ^ 1], t);
        c ^= 1;
        off = 0;
    }
    if (COUNT && t == 0) counts[g] = cnt;
}

// first[g] = *done + exclusive prefix of counts; *done += total.  One CTA, G < 1024.
__global__ void __launch_bounds__(1024) mt_scan_kernel(const int32_t* __restrict__ counts, int G,
                                                       int64_t* __restrict__ first, int64_t* __restrict__ done) {
    __shared__ int sm[33];
    const int t = threadIdx.x;
    const int64_t base = *done;
    int total;
    const int ex = block_exclusive_scan(t < G ? counts[t] : 0, &total, sm);
    if (t < G) first[t] = base + ex;
    if (t == 0) *done = base + total;
}

// n == 0 or high == 1: no word is consumed; the state passes through.
__global__ void mt_copy_state_kernel(const uint32_t* __restrict__ key_in, int pos_in, uint32_t* __restrict__ key_out,
                                     int32_t* __restrict__ pos_out) {
    for (int t = threadIdx.x; t < MT_N; t += blockDim.x) key_out[t] = key_in[t];
    if (threadIdx.x == 0) *pos_out = pos_in;
}

struct MtWs {
    uint32_t* states;   // [MT_GMAX + 1][624]
    int32_t* counts;    // [MT_GMAX]
    int64_t* first;     // [MT_GMAX]
    int64_t* done;      // [1]
};

size_t mt_ws_layout(char* base, MtWs* w) {
    size_t o = 0;
    auto take = [&](size_t bytes) { char* p = base ? base + o : nullptr; o += align_up(bytes); return p; };
    char* s = take((size_t)(MT_GMAX + 1) * MT_N * 4);
    char* c = take((size_t)MT_GMAX * 4);
    char* f = take((size_t)MT_GMAX * 8);
    char* d = take(8);
    if (w) *w = MtWs{(uint32_t*)s, (int32_t*)c, (int64_t*)f, (int64_t*)d};
    return o;
}

// Y[0..B) = X[0..B) A over GF(2) (Y zeroed here; Y must not overlap X).
int gf2_mul(const uint32_t* X, int B, const uint32_t* A, uint32_t* Y, int n_sm, cudaStream_t stream) {
    if (cudaMemsetAsync(Y, 0, (size_t)B * MT_N * 4, stream) != cudaSuccess) return INVPREF_ERR_CUDA;
    const int RBig = B > 16;
    const int rows = RBig ? 64 : 16;
    const int bt = (B + rows - 1) / rows, wt = (MT_N + GF_W - 1) / GF_W;
    int splits = (4 * n_sm) / (bt * wt);
    splits = splits < 1 ? 1 : (splits > MT_N ? MT_N : splits);
    const int kwps = (MT_N + splits - 1) / splits;
    splits = (MT_N + kwps - 1) / kwps;
    const dim3 grid((unsigned)bt, (unsigned)wt, (unsigned)splits);
    if (RBig) gf2_mul_kernel<4><<<grid, GF_THREADS, 0, stream>>>(X, B, A, Y, kwps);
    else gf2_mul_kernel<1><<<grid, GF_THREADS, 0, stream>>>(X, B, A, Y, kwps);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

int device_sms() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
        return 148;
    return n > 0 ? n : 148;
}

}  // namespace

}  // namespace invpref

using namespace invpref;

extern "C" {

int invpref_mt_jump_bytes(size_t* jump_bytes, size_t* ws_bytes) {
    if (!jump_bytes && !ws_bytes) return INVPREF_ERR_BAD_ARG;
    if (jump_bytes) *jump_bytes = (size_t)MT_NJUMPS * MT_MAT_WORDS * 4;
    if (ws_bytes) *ws_bytes = mt_ws_layout(nullptr, nullptr);
    return INVPREF_OK;
}

int invpref_mt_build_jumps(void* jumps, size_t jump_bytes, void* stream_) {
    if (!jumps) return INVPREF_ERR_BAD_ARG;
    if (jump_bytes < (size_t)MT_NJUMPS * MT_MAT_WORDS * 4) return INVPREF_ERR_WORKSPACE;
    cudaStream_t stream = (cudaStream_t)stream_;
    uint32_t* J = (uint32_t*)jumps;
    auto mat = [&](int i) { return J + (size_t)i * MT_MAT_WORDS; };
    const int n_sm = device_sms();
    mt_unit_twist_kernel<<<MT_BITS, MT_THREADS, 0, stream>>>(mat(1));   // A_1 (slots 1, 2 are scratch until A_8)
    count_launch();
    if (cudaGetLastError() != cudaSuccess) return INVPREF_ERR_CUDA;
    static_assert(MT_S0_LOG == 3, "A_1 -> A_8 below takes three squarings");
    int rc = gf2_mul(mat(1), MT_BITS, mat(1), mat(2), n_sm, stream);         // A_2
    if (rc == INVPREF_OK) rc = gf2_mul(mat(2), MT_BITS, mat(2), mat(1), n_sm, stream);   // A_4
    if (rc == INVPREF_OK) rc = gf2_mul(mat(1), MT_BITS, mat(1), mat(0), n_sm, stream);   // A_8
    for (int i = 0; i + 1 < MT_NJUMPS && rc == INVPREF_OK; ++i)
        rc = gf2_mul(mat(i), MT_BITS, mat(i), mat(i + 1), n_sm, stream);
    return rc;
}

int invpref_mt_randint(const uint32_t* key_in, int32_t pos_in, int64_t high, int64_t n, int64_t* out,
                       uint32_t* key_out, int32_t* pos_out, const void* jumps, void* ws, size_t ws_bytes,
                       void* stream_) {
    if (high < 1 || high > (int64_t(1) << 32) || n < 0 || pos_in < 0 || pos_in > MT_N) return INVPREF_ERR_BAD_ARG;
    if (!key_in || !key_out || !pos_out || !jumps || !ws || (n > 0 && !out)) return INVPREF_ERR_BAD_ARG;
    if (ws_bytes < mt_ws_layout(nullptr, nullptr)) return INVPREF_ERR_WORKSPACE;
    cudaStream_t stream = (cudaStream_t)stream_;
    if (n == 0 || high == 1) {                                  // numpy returns zeros without drawing
        if (n > 0 && cudaMemsetAsync(out, 0, (size_t)n * 8, stream) != cudaSuccess) return INVPREF_ERR_CUDA;
        mt_copy_state_kernel<<<1, 256, 0, stream>>>(key_in, pos_in, key_out, pos_out);
        count_launch();
        return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
    }
    MtWs w;
    mt_ws_layout((char*)ws, &w);
    const uint32_t rng = (uint32_t)(high - 1);
    const uint32_t mask = rng ? (0xffffffffu >> __builtin_clz(rng)) : 0u;
    const MtDraw d{rng, mask, n, out, key_out, pos_out};
    const uint32_t* J = (const uint32_t*)jumps;
    const int n_sm = device_sms();
    const int gmax = 3 * n_sm < MT_GMAX ? 3 * n_sm : MT_GMAX;   // one wave of segment CTAs
    // expected words for n acceptances, minus the unconsumed words of the current key, in blocks
    const double p = ((double)rng + 1.0) / ((double)mask + 1.0);
    double left = std::ceil(((double)n / p - (double)(MT_N - pos_in)) / MT_N);
    if (cudaMemsetAsync(w.done, 0, 8, stream) != cudaSuccess) return INVPREF_ERR_CUDA;
    const uint32_t* tail_state = key_in;
    int tail_off = pos_in;
    bool first_round = true;
    while (left >= (double)(2 << MT_S0_LOG)) {
        int a = 0;
        while (a < MT_A_MAX && left > (double)gmax * (double)(1 << (MT_S0_LOG + a))) ++a;
        const int S = 1 << (MT_S0_LOG + a);
        const double segs = std::ceil(left / S);
        const int G = segs < gmax ? (int)segs : gmax;
        if (first_round &&
            cudaMemcpyAsync(w.states, key_in, MT_N * 4, cudaMemcpyDeviceToDevice, stream) != cudaSuccess)
            return INVPREF_ERR_CUDA;
        if (!first_round &&       // the next round starts where the last one ended
            cudaMemcpyAsync(w.states, w.states + (size_t)MT_GMAX * MT_N, MT_N * 4, cudaMemcpyDeviceToDevice, stream)
                != cudaSuccess)
            return INVPREF_ERR_CUDA;
        for (int j = 0; (1 << j) <= G; ++j) {                  // s_{2^j + g} = s_g A_{S 2^j}
            const int lo = 1 << j, cnt = (G + 1 - lo) < lo ? (G + 1 - lo) : lo;
            const int rc = gf2_mul(w.states, cnt, J + (size_t)(a + j) * MT_MAT_WORDS, w.states + (size_t)lo * MT_N,
                                   n_sm, stream);
            if (rc != INVPREF_OK) return rc;
        }
        const int off0 = first_round ? pos_in : MT_N;
        mt_segment_kernel<true><<<G, MT_THREADS, 0, stream>>>(w.states, off0, S, d, w.counts, nullptr);
        mt_scan_kernel<<<1, 1024, 0, stream>>>(w.counts, G, w.first, w.done);
        mt_segment_kernel<false><<<G, MT_THREADS, 0, stream>>>(w.states, off0, S, d, nullptr, w.first);
        count_launch(3);
        if (cudaGetLastError() != cudaSuccess) return INVPREF_ERR_CUDA;
        // s_G: park it in the last slot (the next round's jumps overwrite slots 1..G)
        if (G != MT_GMAX && cudaMemcpyAsync(w.states + (size_t)MT_GMAX * MT_N, w.states + (size_t)G * MT_N, MT_N * 4,
                            cudaMemcpyDeviceToDevice, stream) != cudaSuccess)
            return INVPREF_ERR_CUDA;
        tail_state = w.states + (size_t)MT_GMAX * MT_N;
        tail_off = MT_N;
        left -= (double)G * S;
        first_round = false;
    }
    // the rest, sequentially from where the rounds ended: first rank = *done
    mt_segment_kernel<false><<<1, MT_THREADS, 0, stream>>>(tail_state, tail_off, -1, d, nullptr, w.done);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

}  // extern "C"
