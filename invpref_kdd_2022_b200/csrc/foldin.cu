// Fold-in of rows that are not in the tables: for each history (CSR of (id, score) pairs against a fixed catalogue
// table V) the fp64 solution u of a ridge (explicit model) or L2-regularised logistic (implicit model) problem
// whose score is <u, V[id]>, rounded to fp32 once.  The definition, stopping rule and edge cases are in the header
// (invpref_fold_in_users).
//
// One CTA per folded row (grid-stride).  Per pass over the history, the rows of V are staged in chunks of CH entries
// with double-buffered cp.async, converted to fp64 once, and the lower triangle of the augmented (D + 1) x (D + 1)
// Gram matrix [V^T W V, V^T c; ., .] is accumulated in registers: every 2 x 2 tile of it is owned by one thread,
// which adds the entries in CSR order.  The system is then eliminated in those registers (LDL^T, unscaled columns: each
// column is published to shared memory once final, one barrier per column; the augmented last row carries the
// forward solve) and back-substituted by one warp from the published factor.  The
// implicit model repeats this per damped Newton step and re-streams the history for each line-search trial (the
// catalogue tables of the drivers are L2-resident).  No global workspace.
#include <math.h>

#include "common.cuh"
#include "kernels.h"

namespace invpref {
namespace {

constexpr int FI_THREADS = 256;
constexpr int FI_WARPS = FI_THREADS / 32;
constexpr int FI_MAX_DIM = 128;
constexpr int FI_SLOTS = 9;              // 2 x 2 tiles per thread: 65 * 66 / 2 = 2145 <= 9 * 256 at D = 128
constexpr int FI_HALVINGS = 30;          // line-search trials t = 1, 1/2, ..., 2^-30
constexpr double FI_ARMIJO = 1e-4;

struct FoldArgs {
    const float* V;           // catalogue table [n_cat, D]
    int64_t n_cat;
    const int64_t *off, *ids;
    const float* scores;
    int64_t b;
    double l2;
    int D, max_iter, CH, vec16;
    float* out;               // [b, D]
    int32_t* iters;           // [b] or null
};

// Shared-memory layout (offsets in bytes; every array starts on a 128-byte boundary).
struct FoldLayout {
    int n, XS, DF;            // augmented size D + 1, fp64 row stride (even), fp32 staging row stride (multiple of 4)
    size_t L, xa, xb, u, dl, g, rw, rc, rt, red, raw, sc, valid, total;
};

__host__ __device__ inline size_t fi_up(size_t x) { return (x + 127) & ~(size_t)127; }

__host__ __device__ inline FoldLayout fold_layout(int D, int CH, bool implicit) {
    FoldLayout l;
    l.n = D + 1;
    l.XS = (l.n + 1) & ~1;
    l.DF = (D + 3) & ~3;
    size_t o = 0;
    l.L = o;   o = fi_up(o + (size_t)l.n * (l.n + 1) / 2 * 8);
    l.xa = o;  o = fi_up(o + (size_t)CH * l.XS * 8);
    l.xb = o;  if (implicit) o = fi_up(o + (size_t)CH * l.XS * 8);
    l.u = o;   o = fi_up(o + (size_t)l.XS * 8);
    l.dl = o;  o = fi_up(o + (size_t)l.XS * 8);
    l.g = o;   o = fi_up(o + (size_t)l.XS * 8);
    l.rw = o;  o = fi_up(o + (size_t)CH * 8);
    l.rc = o;  o = fi_up(o + (size_t)CH * 8);
    l.rt = o;  o = fi_up(o + (size_t)CH * 8);
    l.red = o; o = fi_up(o + (size_t)8 * FI_WARPS * 8);
    l.raw = o; o = fi_up(o + (size_t)2 * CH * l.DF * 4);
    l.sc = o;  o = fi_up(o + (size_t)2 * CH * 4);
    l.valid = o; o = fi_up(o + (size_t)2 * CH * 4);
    l.total = o;
    return l;
}

// packed column-major lower triangle of the n x n augmented matrix: column j holds rows j..n-1
__device__ __forceinline__ int col_start(int j, int n) { return j * n - j * (j - 1) / 2; }

// sigmoid and 1 - sigmoid without cancellation
__device__ __forceinline__ void sigmoid2(double z, double& s, double& sm) {
    const double e = exp(-fabs(z));
    const double inv = 1.0 / (1.0 + e);
    s = z >= 0.0 ? inv : e * inv;
    sm = z >= 0.0 ? e * inv : inv;
}

__device__ __forceinline__ double softplus(double z) { return fmax(z, 0.0) + log1p(exp(-fabs(z))); }

// softplus(z + dz) - softplus(z) - y dz: log1p(sigmoid(z) expm1(dz)) keeps the difference accurate when dz is small
// (near the optimum the decrease the Armijo test looks for is far below the rounding of the objective itself)
__device__ __forceinline__ double loss_diff(double z, double dz, double y) {
    double s, sm;
    sigmoid2(z, s, sm);
    const double q = s * expm1(dz);
    const double d = q > -0.5 ? log1p(q) : softplus(z + dz) - softplus(z);
    return d - y * dz;
}

// Deterministic CTA reduction of NS sums followed by NM maxima (fixed shuffle tree, warps summed in order); every
// thread gets the results.
template <int NS, int NM>
__device__ __forceinline__ void block_reduce(double (&v)[NS + NM], double* red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < NS + NM; ++q) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const double y = __shfl_xor_sync(0xffffffffu, v[q], o);
            v[q] = q < NS ? v[q] + y : fmax(v[q], y);
        }
        if (lane == 0) red[q * FI_WARPS + warp] = v[q];
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < NS + NM; ++q) {
        double t = red[q * FI_WARPS];
        for (int w = 1; w < FI_WARPS; ++w) t = q < NS ? t + red[q * FI_WARPS + w] : fmax(t, red[q * FI_WARPS + w]);
        v[q] = t;
    }
    __syncthreads();
}

template <bool IMPLICIT>
__global__ void __launch_bounds__(FI_THREADS, 2) fold_in_kernel(FoldArgs a) {
    extern __shared__ __align__(128) unsigned char fi_smem[];
    const int D = a.D, CH = a.CH;
    const FoldLayout ly = fold_layout(D, CH, IMPLICIT);
    const int n = ly.n, XS = ly.XS, DF = ly.DF;
    double* sL = reinterpret_cast<double*>(fi_smem + ly.L);
    double* sXa = reinterpret_cast<double*>(fi_smem + ly.xa);
    double* sXb = IMPLICIT ? reinterpret_cast<double*>(fi_smem + ly.xb) : sXa;
    double* sU = reinterpret_cast<double*>(fi_smem + ly.u);
    double* sDl = reinterpret_cast<double*>(fi_smem + ly.dl);
    double* sG = reinterpret_cast<double*>(fi_smem + ly.g);
    double* sW = reinterpret_cast<double*>(fi_smem + ly.rw);
    double* sC = reinterpret_cast<double*>(fi_smem + ly.rc);
    double* sT = reinterpret_cast<double*>(fi_smem + ly.rt);
    double* sRed = reinterpret_cast<double*>(fi_smem + ly.red);
    float* sRaw = reinterpret_cast<float*>(fi_smem + ly.raw);
    float* sSc = reinterpret_cast<float*>(fi_smem + ly.sc);
    int* sValid = reinterpret_cast<int*>(fi_smem + ly.valid);
    __shared__ int sBad, sStatus;     // sStatus: the row's iters, written by thread 0 only
    __shared__ double sSum;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // this thread's 2 x 2 tiles (tile-row bi >= tile-column bj, row-major over the lower triangle of tiles)
    const int nb = XS / 2, ntiles = nb * (nb + 1) / 2;
    // two tiles per register (16 bits each: tile-row bi << 8 | tile-column bj, both < 65), to stay at 128 registers
    int tile[(FI_SLOTS + 1) / 2];
#pragma unroll
    for (int s = 0; s < (FI_SLOTS + 1) / 2; ++s) tile[s] = 0;
#pragma unroll
    for (int s = 0; s < FI_SLOTS; ++s) {
        const int e = tid + s * FI_THREADS;
        int bi = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
        while (bi * (bi + 1) / 2 > e) --bi;
        while ((bi + 1) * (bi + 2) / 2 <= e) ++bi;
        const int bj = e - bi * (bi + 1) / 2;
        tile[s >> 1] |= ((bi & 0xff) << 8 | (bj & 0xff)) << (16 * (s & 1));
    }
    auto ti = [&](int s) { return 2 * ((tile[s >> 1] >> (16 * (s & 1) + 8)) & 0xff); };
    auto tj = [&](int s) { return 2 * ((tile[s >> 1] >> (16 * (s & 1))) & 0xff); };

    for (int64_t r = blockIdx.x; r < a.b; r += gridDim.x) {
        const int64_t p0 = a.off[r], len = a.off[r + 1] - p0;
        const int nchunks = (int)((len + CH - 1) / CH);

        // ---- one pass over the history in CSR order: stage, then body(buf, nr) on each chunk ----
        // an entry's score and whether its id is in the catalogue (else the entry is skipped), by the thread that
        // copies the first floats of its row
        auto stage_score = [&](int buf, int h, int64_t q0, bool ok) {
            sValid[buf * CH + h] = ok;
            if (ok)
                cp_async<4>(smem_addr(sSc + buf * CH + h), a.scores + q0 + h);
            else
                sSc[buf * CH + h] = 0.f;
        };
        auto stage = [&](int c) {
            const int buf = c & 1;
            const int64_t q0 = p0 + (int64_t)c * CH;
            const int nr = (int)(len - (int64_t)c * CH < CH ? len - (int64_t)c * CH : CH);
            float* dst = sRaw + (size_t)buf * CH * DF;
            if (a.vec16) {
                const int qv = D >> 2;
                for (int t = tid; t < nr * qv; t += FI_THREADS) {
                    const int h = t / qv, c4 = t - h * qv;
                    const int64_t id = a.ids[q0 + h];
                    const bool ok = id >= 0 && id < a.n_cat;
                    if (ok)
                        cp_async<16>(smem_addr(dst + h * DF + 4 * c4), a.V + id * D + 4 * c4);
                    else
                        *reinterpret_cast<float4*>(dst + h * DF + 4 * c4) = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (c4 == 0) stage_score(buf, h, q0, ok);
                }
            } else {
                for (int t = tid; t < nr * D; t += FI_THREADS) {
                    const int h = t / D, d = t - h * D;
                    const int64_t id = a.ids[q0 + h];
                    const bool ok = id >= 0 && id < a.n_cat;
                    if (ok)
                        cp_async<4>(smem_addr(dst + h * DF + d), a.V + id * D + d);
                    else
                        dst[h * DF + d] = 0.f;
                    if (d == 0) stage_score(buf, h, q0, ok);
                }
            }
        };
        auto pass = [&](auto&& body) {
            if (nchunks > 0) stage(0);
            cp_async_commit();
            for (int c = 0; c < nchunks; ++c) {
                if (c + 1 < nchunks) stage(c + 1);
                cp_async_commit();
                cp_async_wait<1>();
                __syncthreads();
                const int nr = (int)(len - (int64_t)c * CH < CH ? len - (int64_t)c * CH : CH);
                body(c & 1, nr);
                __syncthreads();
            }
            cp_async_wait<0>();
        };
        // <sU, row h> and <sDl, row h> of the staged chunk (fixed order: lane-strided, then a shuffle tree)
        auto dots = [&](const float* row, double& zu, double& zd, bool both) {
            zu = 0.0;
            zd = 0.0;
            for (int d = lane; d < D; d += 32) {
                const double v = (double)row[d];
                zu = fma(sU[d], v, zu);
                if (both) zd = fma(sDl[d], v, zd);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                zu += __shfl_xor_sync(0xffffffffu, zu, o);
                if (both) zd += __shfl_xor_sync(0xffffffffu, zd, o);
            }
        };

        if (tid == 0) sBad = 0;
        for (int d = tid; d < XS; d += FI_THREADS) sU[d] = 0.0;
        __syncthreads();
        if (tid == 0) sStatus = len == 0 ? 0 : (IMPLICIT ? -a.max_iter : 1);

        for (int it = 1; len > 0 && it <= (IMPLICIT ? a.max_iter : 1); ++it) {
            // ---- Gram pass: acc = lower triangle of sum_h [w_h v_h; c_h] [v_h; 0]^T in CSR order ----
            double acc[FI_SLOTS][4];
#pragma unroll
            for (int s = 0; s < FI_SLOTS; ++s)
#pragma unroll
                for (int q = 0; q < 4; ++q) acc[s][q] = 0.0;
            pass([&](int buf, int nr) {
                const float* raw = sRaw + (size_t)buf * CH * DF;
                const float* sc = sSc + buf * CH;
                const int* ok = sValid + buf * CH;
                if (IMPLICIT) {
                    for (int h = warp; h < nr; h += FI_WARPS) {
                        double z, unused;
                        dots(raw + h * DF, z, unused, false);
                        if (lane == 0) {
                            double s, sm;
                            sigmoid2(z, s, sm);
                            sW[h] = ok[h] ? s * sm : 0.0;
                            sC[h] = ok[h] ? s - (double)sc[h] : 0.0;
                        }
                    }
                }
                // explicit: x-side and a-side are one array, [v, y];  implicit: x-side [v, 0] here, a-side below
                for (int t = tid; t < nr * XS; t += FI_THREADS) {
                    const int h = t / XS, d = t - h * XS;
                    double v = 0.0;
                    if (d < D) {
                        const float f = raw[h * DF + d];
                        if (!isfinite(f)) sBad = 1;
                        v = (double)f;
                    } else if (d == D) {
                        if (!isfinite(sc[h])) sBad = 1;
                        v = IMPLICIT ? 0.0 : (double)sc[h];
                    }
                    sXb[h * XS + d] = v;
                }
                if (IMPLICIT) {
                    __syncthreads();
                    for (int t = tid; t < nr * XS; t += FI_THREADS) {
                        const int h = t / XS, d = t - h * XS;
                        sXa[h * XS + d] = d < D ? sW[h] * (double)raw[h * DF + d] : (d == D ? sC[h] : 0.0);
                    }
                }
                __syncthreads();
                for (int h = 0; h < nr; ++h) {
                    const double* ra = sXa + h * XS;
                    const double* rb = sXb + h * XS;
#pragma unroll
                    for (int s = 0; s < FI_SLOTS; ++s) {
                        if (tid + s * FI_THREADS < ntiles) {
                            const double2 ai = *reinterpret_cast<const double2*>(ra + ti(s));
                            const double2 xj = *reinterpret_cast<const double2*>(rb + tj(s));
                            acc[s][0] = fma(ai.x, xj.x, acc[s][0]);
                            acc[s][1] = fma(ai.x, xj.y, acc[s][1]);
                            acc[s][2] = fma(ai.y, xj.x, acc[s][2]);
                            acc[s][3] = fma(ai.y, xj.y, acc[s][3]);
                        }
                    }
                }
            });
            // ---- the system, in the registers that hold the triangle: (G + l2 I) u = V^T y  |  (H + l2 I) dl = -g,
            //      g = V^T c + l2 u (the last row); column 0 goes to shared memory ----
#pragma unroll
            for (int s = 0; s < FI_SLOTS; ++s) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int i = ti(s) + (q >> 1), j = tj(s) + (q & 1);
                    if (tid + s * FI_THREADS < ntiles && j <= i && i < n) {
                        if (i == j && i < D) acc[s][q] += a.l2;
                        if (IMPLICIT && i == D && j < D) {
                            const double g = acc[s][q] + a.l2 * sU[j];
                            sG[j] = g;
                            acc[s][q] = -g;
                        }
                        if (j == 0) sL[i] = acc[s][q];
                    }
                }
            }
            __syncthreads();
            // ---- LDL^T elimination on the register-resident entries: step k subtracts (A[i][k] / A[k][k]) A[j][k]
            //      from every entry (i, j), j > k, and publishes column k + 1, final from then on, to shared memory.
            //      Afterwards column k holds L[i][k] * d_k and the last row the forward-solved right-hand side.
            //      Entries above the diagonal of a diagonal tile take garbage and are never published. ----
            for (int k = 0; k + 1 < D; ++k) {
                const int ck = col_start(k, n), c1 = col_start(k + 1, n);
                const double rpiv = 1.0 / sL[ck];
#pragma unroll
                for (int s = 0; s < FI_SLOTS; ++s) {
                    if (tid + s * FI_THREADS < ntiles && tj(s) >= k) {      // ti >= tj: both rows are >= k
                        const double l0 = sL[ck + ti(s) - k] * rpiv, l1 = sL[ck + ti(s) + 1 - k] * rpiv;
                        const double m0 = sL[ck + tj(s) - k], m1 = sL[ck + tj(s) + 1 - k];
                        acc[s][0] = fma(-l0, m0, acc[s][0]);
                        acc[s][1] = fma(-l0, m1, acc[s][1]);
                        acc[s][2] = fma(-l1, m0, acc[s][2]);
                        acc[s][3] = fma(-l1, m1, acc[s][3]);
                        if (tj(s) == k || tj(s) == k + 1) {
                            const bool odd = tj(s) == k;                     // column k + 1 is this tile's second
                            const int i0 = ti(s), i1 = ti(s) + 1;
                            if (i0 >= k + 1 && i0 < n) sL[c1 + i0 - (k + 1)] = odd ? acc[s][1] : acc[s][0];
                            if (i1 >= k + 1 && i1 < n) sL[c1 + i1 - (k + 1)] = odd ? acc[s][3] : acc[s][2];
                        }
                    }
                }
                __syncthreads();
            }
            // ---- back substitution by warp 0: x_i = (y_i - sum_{k > i} A[k][i] x_k) / d_i, i descending ----
            if (warp == 0) {
                double rr[FI_MAX_DIM / 32];
#pragma unroll
                for (int q = 0; q < FI_MAX_DIM / 32; ++q) {
                    const int k = lane + 32 * q;
                    rr[q] = k < D ? sL[col_start(k, n) + D - k] : 0.0;
                }
                for (int i = D - 1; i >= 0; --i) {
                    const int qi = i >> 5;
                    double mine = rr[0];
#pragma unroll
                    for (int q = 1; q < FI_MAX_DIM / 32; ++q) mine = qi == q ? rr[q] : mine;
                    const double xi = __shfl_sync(0xffffffffu, mine / sL[col_start(i, n)], i & 31);
                    if (lane == (i & 31)) sDl[i] = xi;
#pragma unroll
                    for (int q = 0; q < FI_MAX_DIM / 32; ++q) {
                        const int k = lane + 32 * q;
                        if (k < i) rr[q] = fma(-sL[col_start(k, n) + i - k], xi, rr[q]);
                    }
                }
            }
            __syncthreads();
            if (!IMPLICIT) {
                for (int d = tid; d < D; d += FI_THREADS) sU[d] = sDl[d];
                __syncthreads();
                break;
            }
            // ---- damped Newton step ----
            double red[5];
            {
                const double dl = tid < D ? sDl[tid] : 0.0, u = tid < D ? sU[tid] : 0.0;
                red[0] = tid < D ? sG[tid] * dl : 0.0;
                red[1] = u * dl;
                red[2] = dl * dl;
                red[3] = fabs(dl);
                red[4] = fabs(u);
            }
            block_reduce<3, 2>(red, sRed);
            const double gd = red[0], ud = red[1], dd = red[2];
            if (sBad || !isfinite(gd) || !isfinite(red[3])) {
                sBad = 1;      // a non-finite entry in the history, or an overflow: the row is NaN
                break;
            }
            if (red[3] <= 0x1p-30 * fmax(1.0, red[4])) {          // converged: take the full step and stop
                for (int d = tid; d < D; d += FI_THREADS) sU[d] += sDl[d];
                if (tid == 0) sStatus = it;
                __syncthreads();
                break;
            }
            double t = 1.0;
            for (int m = 0; m <= FI_HALVINGS; ++m) {
                t = ldexp(1.0, -m);
                double sum = 0.0;                                 // held by thread 0
                pass([&](int buf, int nr) {
                    const float* raw = sRaw + (size_t)buf * CH * DF;
                    const float* sc = sSc + buf * CH;
                    const int* ok = sValid + buf * CH;
                    for (int h = warp; h < nr; h += FI_WARPS) {
                        double zu, zd;
                        dots(raw + h * DF, zu, zd, true);
                        if (lane == 0) sT[h] = ok[h] ? loss_diff(zu, t * zd, (double)sc[h]) : 0.0;
                    }
                    __syncthreads();
                    if (tid == 0)
                        for (int h = 0; h < nr; ++h) sum += sT[h];
                });
                if (tid == 0) sSum = sum + a.l2 * (t * ud + 0.5 * t * t * dd);
                __syncthreads();
                const bool accept = sSum <= FI_ARMIJO * t * gd;
                __syncthreads();
                if (accept) break;
            }
            for (int d = tid; d < D; d += FI_THREADS) sU[d] = fma(t, sDl[d], sU[d]);
            __syncthreads();
        }

        // ---- result ----
        if (tid < D && !isfinite(sU[tid])) sBad = 1;
        __syncthreads();
        const bool bad = sBad != 0;
        for (int d = tid; d < D; d += FI_THREADS) a.out[r * D + d] = bad ? __int_as_float(0x7fc00000) : (float)sU[d];
        if (tid == 0 && a.iters != nullptr) a.iters[r] = bad && IMPLICIT ? -a.max_iter : sStatus;
        __syncthreads();
    }
}

template <bool IMPLICIT>
int launch_fold_in_impl(FoldArgs& a, cudaStream_t stream) {
    // the largest chunk that keeps two CTAs on an SM
    int CH = 32;
    while (CH > 8 && fold_layout(a.D, CH, IMPLICIT).total > 110 * 1024) CH >>= 1;
    a.CH = CH;
    const size_t smem = fold_layout(a.D, CH, IMPLICIT).total;
    INVPREF_SET_SMEM_ONCE(fold_in_kernel<IMPLICIT>, smem);
    static int n_sm = 0;
    if (n_sm == 0) {
        int dev = 0;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&n_sm, cudaDevAttrMultiProcessorCount, dev);
        n_sm = n_sm > 0 ? n_sm : 148;
    }
    const int64_t cap = (int64_t)n_sm * 2;
    const unsigned grid = (unsigned)(a.b < cap ? a.b : cap);
    fold_in_kernel<IMPLICIT><<<grid, FI_THREADS, smem, stream>>>(a);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? INVPREF_OK : INVPREF_ERR_CUDA;
}

}  // namespace

int fold_in_max_dim() { return FI_MAX_DIM; }

int launch_fold_in(const float* V, int64_t n_cat, int D, int implicit, const int64_t* off, const int64_t* ids,
                   const float* scores, int64_t b, double l2, int max_iter, float* out, int32_t* iters,
                   cudaStream_t stream) {
    FoldArgs a;
    a.V = V; a.n_cat = n_cat; a.off = off; a.ids = ids; a.scores = scores; a.b = b; a.l2 = l2;
    a.D = D; a.max_iter = max_iter; a.out = out; a.iters = iters;
    a.vec16 = (D % 4 == 0 && ((uintptr_t)V & 15) == 0) ? 1 : 0;
    return implicit ? launch_fold_in_impl<true>(a, stream) : launch_fold_in_impl<false>(a, stream);
}

}  // namespace invpref
