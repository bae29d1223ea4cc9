// Hand-written device primitives of the sort-segment plan (plan.cu): a stable LSD radix sort of (int32 key, int32
// value) pairs and int32 prefix sums.  No library calls (round 1 used cub::DeviceRadixSort / DeviceScan here).
//
// Radix sort: 8-bit digits, ceil(bits / 8) passes over the key bits that can be set (`bits` = log2 of the table's row
// count: 24 for 10 M users -> 3 passes, 10 for Yahoo's 1 000 items -> 2).  A pass is three launches without any
// spin-wait between CTAs:
//   rs_hist_kernel     per-tile digit counts (4 096 keys per tile, shared-memory atomics) + digit totals
//   rs_offsets_kernel  one CTA per digit: exclusive sum of that digit's tile counts behind the digits below it
//   rs_scatter_kernel  re-reads the tile, ranks every key among the equal digits before it, orders the tile in shared
//                      memory and writes each digit's run with consecutive threads
// Stability: a warp owns 512 consecutive keys and takes them 32 at a time, so (tile, warp, round, lane) is memory
// order; a key's rank among equal digits = equal digits of earlier tiles + of earlier warps of the tile + of earlier
// rounds of the warp + of lower lanes of the round (peer mask from nine ballots).  The result is therefore THE stable
// sort: `perm` is bit-equal to torch.sort(ids, stable=True).indices (tests/test_gpu_hotpath.py, test_gpu_fullsize.py).
//
// Scans: reduce (per 2 048-element tile) -> one-CTA exclusive scan of the tile sums -> per-tile scan.  MODE 1 scans
// the head flags of a sorted key array without materialising them.
#pragma once
#include "common.cuh"

namespace invpref {
namespace psort {

constexpr int RS_THREADS = 256;
constexpr int RS_WARPS = RS_THREADS / 32;
constexpr int RS_IPT = 16;                            // keys per thread
constexpr int RS_TILE = RS_THREADS * RS_IPT;          // 4 096 keys per CTA
constexpr int RS_BINS = 256;
constexpr int RS_MAX_PASSES = 4;
constexpr int SC_THREADS = 256;
constexpr int SC_IPT = 8;
constexpr int SC_TILE = SC_THREADS * SC_IPT;          // 2 048 elements per CTA

inline int64_t rs_tiles(int64_t n) { return (n + RS_TILE - 1) / RS_TILE; }
inline int64_t sc_tiles(int64_t n) { return (n + SC_TILE - 1) / SC_TILE; }

// scratch of radix_sort_pairs (besides the ping-pong arrays): tile counts + digit totals
inline size_t rs_scratch_bytes(int64_t n) {
    return align_up((size_t)rs_tiles(n) * RS_BINS * 4) + align_up((size_t)RS_MAX_PASSES * RS_BINS * 4);
}
inline size_t sc_scratch_bytes(int64_t n) { return align_up((size_t)(sc_tiles(n) + 1) * 4); }

// ---------------------------------------------------------------------------------------------- radix sort
__global__ void __launch_bounds__(RS_THREADS)
rs_hist_kernel(const int32_t* __restrict__ keys, int64_t n, int shift, unsigned mask, int32_t* __restrict__ tile_hist,
               int32_t* __restrict__ digit_total) {
    __shared__ int32_t hist[RS_BINS];
    hist[threadIdx.x] = 0;
    __syncthreads();
    const int64_t base = (int64_t)blockIdx.x * RS_TILE + threadIdx.x;
    int32_t key[RS_IPT];
#pragma unroll
    for (int j = 0; j < RS_IPT; ++j) {
        const int64_t k = base + (int64_t)j * RS_THREADS;
        key[j] = k < n ? keys[k] : 0;
    }
#pragma unroll
    for (int j = 0; j < RS_IPT; ++j)   // plain shared-memory atomics: MATCH.ANY costs more than the conflicts it saves
        if (base + (int64_t)j * RS_THREADS < n) atomicAdd(&hist[((unsigned)key[j] >> shift) & mask], 1);
    __syncthreads();
    const int32_t c = hist[threadIdx.x];
    tile_hist[(int64_t)blockIdx.x * RS_BINS + threadIdx.x] = c;
    if (c != 0) atomicAdd(&digit_total[threadIdx.x], c);   // integer: order-independent
}

// CTA d: tile_hist[t][d] <- (keys with a digit < d) + (keys with digit d in tiles < t)
__global__ void __launch_bounds__(1024)
rs_offsets_kernel(int32_t* __restrict__ tile_hist, int64_t n_tiles, const int32_t* __restrict__ digit_total) {
    __shared__ int sm[33];
    const int d = blockIdx.x;
    int carry;
    (void)block_exclusive_scan((int)threadIdx.x < d ? digit_total[threadIdx.x] : 0, &carry, sm);
    for (int64_t t0 = 0; t0 < n_tiles; t0 += blockDim.x) {
        const int64_t t = t0 + threadIdx.x;
        const int c = t < n_tiles ? tile_hist[t * RS_BINS + d] : 0;
        int total;
        const int ex = block_exclusive_scan(c, &total, sm);
        if (t < n_tiles) tile_hist[t * RS_BINS + d] = carry + ex;
        carry += total;
    }
}

// Lanes of the warp holding the same 9-bit value (8 digit bits + the past-the-end bit): nine ballots.  (MATCH.ANY gives
// the same mask in one instruction but measured 2-3x slower here: 75 us per 4 M-key pass against the ballot form.)
__device__ __forceinline__ unsigned same_digit_lanes(unsigned d) {
    unsigned peers = 0xffffffffu;
#pragma unroll
    for (int b = 0; b < 9; ++b) {
        const bool bit = (d >> b) & 1u;
        const unsigned bal = __ballot_sync(0xffffffffu, bit);
        peers &= bit ? bal : ~bal;
    }
    return peers;
}

// vals_in == nullptr: the value of key k is k (first pass of an argsort)
__global__ void __launch_bounds__(RS_THREADS)
rs_scatter_kernel(const int32_t* __restrict__ keys_in, const int32_t* __restrict__ vals_in,
                  int32_t* __restrict__ keys_out, int32_t* __restrict__ vals_out, int64_t n, int shift, unsigned mask,
                  const int32_t* __restrict__ tile_off) {
    __shared__ int32_t whist[RS_WARPS][RS_BINS + 1];    // bin 256: lanes past the end
    __shared__ int32_t skey[RS_TILE], sval[RS_TILE];
    __shared__ int32_t lstart[RS_BINS], gbase[RS_BINS];
    __shared__ int sm[33];
    for (int i = threadIdx.x; i < RS_WARPS * (RS_BINS + 1); i += RS_THREADS) (&whist[0][0])[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t base = (int64_t)blockIdx.x * RS_TILE + (int64_t)warp * (32 * RS_IPT) + lane;
    int32_t key[RS_IPT], val[RS_IPT], rank[RS_IPT];
#pragma unroll
    for (int j = 0; j < RS_IPT; ++j) {
        const int64_t k = base + j * 32;
        key[j] = k < n ? keys_in[k] : 0;
        val[j] = vals_in != nullptr ? (k < n ? vals_in[k] : 0) : (int32_t)k;
    }
    const unsigned lt = (1u << lane) - 1u;
#pragma unroll
    for (int j = 0; j < RS_IPT; ++j) {
        const bool ok = base + j * 32 < n;
        const unsigned d = ok ? (((unsigned)key[j] >> shift) & mask) : (unsigned)RS_BINS;
        const unsigned peers = same_digit_lanes(d);
        const int leader = __ffs(peers) - 1;
        int before = 0;
        if (lane == leader) {
            before = whist[warp][d];
            whist[warp][d] = before + __popc(peers);
        }
        before = __shfl_sync(0xffffffffu, before, leader);
        rank[j] = before + __popc(peers & lt);
        __syncwarp();
    }
    __syncthreads();
    {   // thread d: digit d's run inside the tile (start, per-warp starts) and where the run goes in the output
        const int d = threadIdx.x;
        int cnt = 0;
#pragma unroll
        for (int w = 0; w < RS_WARPS; ++w) {
            const int c = whist[w][d];
            whist[w][d] = cnt;
            cnt += c;
        }
        int total;
        const int start = block_exclusive_scan(cnt, &total, sm);
        lstart[d] = start;
        gbase[d] = tile_off[(int64_t)blockIdx.x * RS_BINS + d] - start;
    }
    __syncthreads();
    // stage the tile in sorted order in shared memory, then write runs of equal digits with consecutive threads:
    // a 4-byte store per key straight from the ranking order costs one L2 request per key (56 us per 4 M-key pass)
#pragma unroll
    for (int j = 0; j < RS_IPT; ++j) {
        if (base + j * 32 < n) {
            const unsigned d = ((unsigned)key[j] >> shift) & mask;
            const int lp = lstart[d] + whist[warp][d] + rank[j];
            skey[lp] = key[j];
            sval[lp] = val[j];
        }
    }
    __syncthreads();
    const int64_t left = n - (int64_t)blockIdx.x * RS_TILE;
    const int n_valid = left < RS_TILE ? (int)left : RS_TILE;
#pragma unroll
    for (int j = 0; j < RS_IPT; ++j) {
        const int i = threadIdx.x + j * RS_THREADS;
        if (i < n_valid) {
            const int32_t k = skey[i];
            const int pos = gbase[((unsigned)k >> shift) & mask] + i;
            keys_out[pos] = k;
            vals_out[pos] = sval[i];
        }
    }
}

// Stable sort of n (key, value) pairs by the low `bits` bits of the key (keys are non-negative ids).
// keys_in is read only; the result lands in keys_out / vals_out; keys_tmp / vals_tmp are ping-pong scratch of n ints;
// vals_in == nullptr sorts the identity (argsort).  Returns the number of launches.
inline int radix_sort_pairs(const int32_t* keys_in, const int32_t* vals_in, int32_t* keys_out, int32_t* vals_out,
                            int32_t* keys_tmp, int32_t* vals_tmp, int64_t n, int bits, char* scratch,
                            cudaStream_t stream) {
    int passes = (bits + 7) / 8;
    if (passes < 1) passes = 1;
    if (passes > RS_MAX_PASSES) passes = RS_MAX_PASSES;
    const int64_t T = rs_tiles(n);
    int32_t* tile_hist = (int32_t*)scratch;
    int32_t* digit_total = (int32_t*)(scratch + align_up((size_t)T * RS_BINS * 4));
    cudaMemsetAsync(digit_total, 0, (size_t)RS_MAX_PASSES * RS_BINS * 4, stream);
    const int32_t* src_k = keys_in;
    const int32_t* src_v = vals_in;
    for (int p = 0; p < passes; ++p) {
        const int shift = 8 * p;
        const int left = bits - shift;
        const unsigned mask = left >= 8 ? 0xffu : ((1u << left) - 1u);
        const bool to_out = ((passes - 1 - p) & 1) == 0;   // the last pass writes the outputs
        int32_t* dst_k = to_out ? keys_out : keys_tmp;
        int32_t* dst_v = to_out ? vals_out : vals_tmp;
        rs_hist_kernel<<<(unsigned)T, RS_THREADS, 0, stream>>>(src_k, n, shift, mask, tile_hist,
                                                               digit_total + p * RS_BINS);
        rs_offsets_kernel<<<RS_BINS, 1024, 0, stream>>>(tile_hist, T, digit_total + p * RS_BINS);
        rs_scatter_kernel<<<(unsigned)T, RS_THREADS, 0, stream>>>(src_k, src_v, dst_k, dst_v, n, shift, mask,
                                                                  tile_hist);
        src_k = dst_k;
        src_v = dst_v;
    }
    return 3 * passes;
}

// ---------------------------------------------------------------------------------------------- prefix sums
// MODE 0: the element itself.  MODE 1: head flag of a sorted array (1 where a new key starts).
// A thread takes SC_IPT = 8 consecutive elements: two 16-byte loads (arrays are 16-byte aligned, k0 is a multiple of 8).
template <int MODE>
__device__ __forceinline__ void sc_load8(const int32_t* in, int64_t k0, int64_t n, int (&x)[SC_IPT]) {
    int raw[SC_IPT];
    if (k0 + SC_IPT <= n) {
        const int4 a = *reinterpret_cast<const int4*>(in + k0);
        const int4 b = *reinterpret_cast<const int4*>(in + k0 + 4);
        raw[0] = a.x; raw[1] = a.y; raw[2] = a.z; raw[3] = a.w;
        raw[4] = b.x; raw[5] = b.y; raw[6] = b.z; raw[7] = b.w;
    } else {
#pragma unroll
        for (int i = 0; i < SC_IPT; ++i) raw[i] = k0 + i < n ? in[k0 + i] : 0;
    }
    if (MODE == 0) {
#pragma unroll
        for (int i = 0; i < SC_IPT; ++i) x[i] = k0 + i < n ? raw[i] : 0;
    } else {
        int prev = (k0 > 0 && k0 < n) ? in[k0 - 1] : 0;
#pragma unroll
        for (int i = 0; i < SC_IPT; ++i) {
            x[i] = (k0 + i < n && (k0 + i == 0 || raw[i] != prev)) ? 1 : 0;
            prev = raw[i];
        }
    }
}

template <int MODE>
__global__ void __launch_bounds__(SC_THREADS)
sc_reduce_kernel(const int32_t* __restrict__ in, int64_t n, int32_t* __restrict__ tile_sum) {
    __shared__ int sm[33];
    const int64_t k0 = (int64_t)blockIdx.x * SC_TILE + (int64_t)threadIdx.x * SC_IPT;
    int x[SC_IPT];
    sc_load8<MODE>(in, k0, n, x);
    int s = 0;
#pragma unroll
    for (int i = 0; i < SC_IPT; ++i) s += x[i];
    int total;
    (void)block_exclusive_scan(s, &total, sm);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}

// one CTA: tile_sum[0..T) <- exclusive prefix, tile_sum[T] <- grand total
__global__ void __launch_bounds__(1024) sc_mid_kernel(int32_t* __restrict__ tile_sum, int64_t T) {
    __shared__ int sm[33];
    int carry = 0;
    for (int64_t t0 = 0; t0 < T; t0 += blockDim.x) {
        const int64_t t = t0 + threadIdx.x;
        const int c = t < T ? tile_sum[t] : 0;
        int total;
        const int ex = block_exclusive_scan(c, &total, sm);
        if (t < T) tile_sum[t] = carry + ex;
        carry += total;
    }
    if (threadIdx.x == 0) tile_sum[T] = carry;
}

template <int MODE, bool INCLUSIVE>
__global__ void __launch_bounds__(SC_THREADS)
sc_scan_kernel(const int32_t* in, int32_t* out, int64_t n, const int32_t* __restrict__ tile_sum) {
    __shared__ int sm[33];
    const int64_t k0 = (int64_t)blockIdx.x * SC_TILE + (int64_t)threadIdx.x * SC_IPT;
    int x[SC_IPT];
    sc_load8<MODE>(in, k0, n, x);
    int s = 0;
#pragma unroll
    for (int i = 0; i < SC_IPT; ++i) s += x[i];
    int total;
    int run = block_exclusive_scan(s, &total, sm) + tile_sum[blockIdx.x];
    int y[SC_IPT];
#pragma unroll
    for (int i = 0; i < SC_IPT; ++i) {
        if (INCLUSIVE) run += x[i];
        y[i] = run;
        if (!INCLUSIVE) run += x[i];
    }
    if (k0 + SC_IPT <= n) {
        *reinterpret_cast<int4*>(out + k0) = make_int4(y[0], y[1], y[2], y[3]);
        *reinterpret_cast<int4*>(out + k0 + 4) = make_int4(y[4], y[5], y[6], y[7]);
    } else {
#pragma unroll
        for (int i = 0; i < SC_IPT; ++i)
            if (k0 + i < n) out[k0 + i] = y[i];
    }
}

// out[k] = sum of f(in[0..k]) (INCLUSIVE) or f(in[0..k)) ; in == out is allowed for MODE 0.  3 launches.
template <int MODE, bool INCLUSIVE>
inline int prefix_sum(const int32_t* in, int32_t* out, int64_t n, char* scratch, cudaStream_t stream) {
    if (n <= 0) return 0;
    const int64_t T = sc_tiles(n);
    int32_t* tile_sum = (int32_t*)scratch;
    sc_reduce_kernel<MODE><<<(unsigned)T, SC_THREADS, 0, stream>>>(in, n, tile_sum);
    sc_mid_kernel<<<1, 1024, 0, stream>>>(tile_sum, T);
    sc_scan_kernel<MODE, INCLUSIVE><<<(unsigned)T, SC_THREADS, 0, stream>>>(in, out, n, tile_sum);
    return 3;
}

}  // namespace psort
}  // namespace invpref
