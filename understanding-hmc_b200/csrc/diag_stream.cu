// Streamed diagnostics: the partial sums of hmc_diag_moments and hmc_diag_variogram, folded in block by block from a ring of the
// last R stored samples per chain (hmc_random_args.store_ring = R), so that a run never needs its whole sample stream on the device.
//
// Stored indices 1 .. 2n are used (index 0 is dropped as samplers.py:61 does; with L_chain - 1 odd the last sample is dropped too,
// utils.py:96-99): split chain 2m is indices [1, n] of chain m, split chain 2m+1 is [n+1, 2n] (utils.py:102).  Stored index j of chain
// c lives in ring row j % R: q_ring[(c * R + j % R) * D + d].
//
// Workspace (float64 throughout), caller-allocated, zeroed by the call with j0 = 0:
//   rows  [4][D]           sum_j std_j, sum_j (mean_j - c), sum_j (mean_j - c)^2, c  (the layout hmc_diag_moments writes)
//   lags  [T][D]           lag t at row t - 1: sum over split chains and i of (x[i+t] - x[i])^2, pairs inside one split chain
//   state [3][Nchain][D]   per chain and dimension, for the split chain being filled: its first sample (the shift), and the
//                          shifted sum and sum of squares of its samples so far
//
// hmc_diag_stream_update(j0, j1) adds every stored index in [j0, j1) to the moments (closing a split chain at index n or 2n folds its
// mean and ddof = 1 std into `rows`, and the state starts over for the next one), and adds to `lags` every pair (i - t, i) with i in
// [j0, j1), 1 <= t <= T and i - t in i's own split chain.  The earlier element comes from the ring, so rows [j0 - T, j1) must all
// still be there: R >= T + (j1 - j0).
//
// The lag kernel tiles like the windowed kernel of diag.cu: one block takes a 32-dimension tile of one chain at a time, copies the
// new rows and the rows they pair with (at most 128 lags per launch) into shared memory once, and each warp forms the pairs of 16
// consecutive lags from a register window that slides along the new samples (the window of diag_variogram_kernel: one new value per
// step, compile-time slot indices), so a pair costs a subtraction and a fused multiply-add.  Per-chain sums are kept in the stream's
// precision over at most 64 new samples and widened into float64 per chain, then added to `lags` with one float64 atomic per
// (block, lag, dimension).
#include "hmc_common.cuh"
#ifdef HMC_DIAG_STREAM_DEBUG
#include <cassert>
#define DS_ASSERT(c) assert(c)
#else
#define DS_ASSERT(c) ((void)0)
#endif

namespace {

constexpr int kTile = 32;        // dimensions per block (one warp-wide row segment)
constexpr int kWarps = 8;
constexpr int kLT = 16;          // lags per warp
constexpr int kLagsPerLaunch = kWarps * kLT;
constexpr int kNewPerLaunch = 64;
constexpr int kMaxD = 8192;

// Per chain and dimension: walk the new stored indices [ilo, ihi) (already clipped to [1, 2n]); at the first index of a split chain
// the state restarts from that sample, at its last one the split chain's mean and ddof = 1 std (utils.py:107-118) are folded into
// rows[0..2] relative to the device shift c = the first used sample of local chain 0 (rows[3]).
template <typename T>
__global__ void __launch_bounds__(kTile * kWarps) stream_moments_kernel(const T* __restrict__ ring, long Nchain, int D, int R, long n,
                                                                        long ilo, long ihi, long j0, long j1, double* __restrict__ rows,
                                                                        double* __restrict__ state) {
    __shared__ double red[3][kWarps][kTile];
    const int lane = threadIdx.x % kTile, w = threadIdx.x / kTile;
    const int d = blockIdx.x * kTile + lane;
    double s_std = 0.0, s_mean = 0.0, s_mean2 = 0.0;
    if (d < D) {
        // c is read from the ring in the call that hands over index 1 (and recorded in rows[3]), from rows[3] afterwards
        const bool have1 = j0 <= 1 && 1 < j1;
        const double c = have1 ? (double)ring[(size_t)(1 % R) * D + d] : rows[3 * (size_t)D + d];
        if (have1 && blockIdx.y == 0 && w == 0) rows[3 * (size_t)D + d] = c;
        const size_t plane = (size_t)Nchain * D;
        for (long ch = (long)blockIdx.y * kWarps + w; ch < Nchain; ch += (long)gridDim.y * kWarps) {
            double* st = state + (size_t)ch * D + d;
            double x0 = st[0], a = st[plane], b = st[2 * plane];
            for (long i = ilo; i < ihi; ++i) {
                DS_ASSERT(i >= j1 - R && i < j1);
                const double x = (double)ring[((size_t)ch * R + (size_t)(i % R)) * D + d];
                if (i == 1 || i == n + 1) { x0 = x; a = 0.0; b = 0.0; }
                const double v = x - x0;
                a += v;
                b += v * v;
                if (i == n || i == 2 * n) {
                    const double mean_s = a / (double)n;
                    double var = (b - (double)n * mean_s * mean_s) / (double)(n - 1);   // ddof = 1 (utils.py:111)
                    if (var < 0.0) var = 0.0;
                    const double mean = mean_s + (x0 - c);
                    s_std += sqrt(var);
                    s_mean += mean;
                    s_mean2 += mean * mean;
                }
            }
            st[0] = x0; st[plane] = a; st[2 * plane] = b;
        }
    }
    red[0][w][lane] = s_std; red[1][w][lane] = s_mean; red[2][w][lane] = s_mean2;
    __syncthreads();
    if (w < 3 && d < D) {
        double s = 0.0;
        for (int k = 0; k < kWarps; ++k) s += red[w][k][lane];
        if (s != 0.0) atomicAdd(rows + (size_t)w * D + d, s);
    }
}

// Pairs (i - t, i) for new indices i in [lo, hi) of ONE split chain starting at s0, lags t in [tl, th) (th - tl <= 128).
// Shared memory per chain: the new rows [lo, hi) and the earlier rows [elo, ehi] they pair with, 32 dimensions each.
// Warp w owns lags t0 + k, t0 = tl + 16 w, k < 16 (nl of them valid); step i pairs x[i] with the window slot of x[i - t0 - k].
template <typename T>
__global__ void __launch_bounds__(kTile * kWarps, sizeof(T) == 4 ? 2 : 1) stream_lags_kernel(const T* __restrict__ ring, long Nchain, int D, int R, long s0,
                                                                        long lo, long hi, int tl, int th, long j1, double* __restrict__ lags) {
    extern __shared__ __align__(16) unsigned char smraw[];
    T* nw = reinterpret_cast<T*>(smraw);                   // [hi - lo][32]
    const int lane = threadIdx.x % kTile, w = threadIdx.x / kTile;
    const int d = blockIdx.x * kTile + lane;
    const bool dok = d < D;
    const long elo = (s0 > lo - th + 1) ? s0 : lo - th + 1;
    const long ehi = hi - 1 - tl;                           // inclusive
    const int nnew = (int)(hi - lo);
    const int nold = ehi >= elo ? (int)(ehi - elo + 1) : 0;
    T* ow = nw + (size_t)nnew * kTile;                     // [nold][32]
    const int t0 = tl + w * kLT;
    const int nl = (th - t0 < kLT) ? th - t0 : kLT;        // lags of this warp (<= 0: idle)
    double dacc[kLT];
#pragma unroll
    for (int k = 0; k < kLT; ++k) dacc[k] = 0.0;
    for (long ch = blockIdx.y; ch < Nchain; ch += gridDim.y) {
        DS_ASSERT(ch >= 0 && ch < Nchain);
        const T* base = ring + (size_t)ch * R * D + d;
        __syncthreads();
        for (int r = w; r < nnew + nold; r += kWarps) {
            const long j = r < nnew ? lo + r : elo + (r - nnew);
            DS_ASSERT(j >= 1 && j >= j1 - R && j < j1);
            nw[(size_t)r * kTile + lane] = dok ? base[(size_t)(j % R) * D] : T(0);
        }
        __syncthreads();
        if (nl <= 0) continue;
        T acc[kLT], win[kLT];
#pragma unroll
        for (int k = 0; k < kLT; ++k) acc[k] = T(0);
        // slot (r mod 16) holds x[lo + r - t0]; preload the slots of steps r = -1 .. -15
#pragma unroll
        for (int k = 1; k < kLT; ++k) {
            const long e = lo - t0 - k;
            DS_ASSERT(e < elo || e - elo < nold);
            win[kLT - k] = (e >= elo) ? ow[(size_t)(e - elo) * kTile + lane] : T(0);
        }
        for (int rb = 0; rb < nnew; rb += kLT) {
#pragma unroll
            for (int r = 0; r < kLT; ++r) {
                if (rb + r < nnew) {
                    const long i = lo + rb + r;
                    const long e = i - t0;
                    DS_ASSERT(e < elo || e - elo < nold);
                    win[r] = (e >= elo) ? ow[(size_t)(e - elo) * kTile + lane] : T(0);
                    const T xi = nw[(size_t)(rb + r) * kTile + lane];
                    const long lim = (e - s0 < (long)nl - 1) ? e - s0 : (long)nl - 1;   // pair k valid iff k <= lim
                    if (lim >= kLT - 1) {
#pragma unroll
                        for (int k = 0; k < kLT; ++k) { const T df = xi - win[(r - k + kLT) % kLT]; acc[k] = fma(df, df, acc[k]); }
                    } else {
#pragma unroll
                        for (int k = 0; k < kLT; ++k) {
                            if (k <= lim) { const T df = xi - win[(r - k + kLT) % kLT]; acc[k] = fma(df, df, acc[k]); }
                        }
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < kLT; ++k) dacc[k] += (double)acc[k];
    }
    if (dok) {
#pragma unroll
        for (int k = 0; k < kLT; ++k) {
            if (k < nl) { DS_ASSERT(t0 + k >= 1 && t0 + k < th); atomicAdd(lags + (size_t)(t0 + k - 1) * D + d, dacc[k]); }
        }
    }
}

int sm_count() {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

int chain_groups(long want, int gx, int per_sm) {
    long g = (long)sm_count() * per_sm / gx;
    if (g < 1) g = 1;
    if (g > want) g = want;
    if (g > 65535) g = 65535;
    return (int)g;
}

}  // namespace

#define HMC_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            hmc_set_error(__VA_ARGS__);   \
            return HMC_E_BADARG;          \
        }                                 \
    } while (0)

static const int64_t kMaxT = 1 << 20;

extern "C" int64_t hmc_diag_stream_workspace_bytes(int64_t Nchain, int32_t D, int32_t T) {
    if (Nchain < 1 || Nchain > (int64_t(1) << 31) || D < 1 || D > kMaxD || T < 1 || T > kMaxT) return 0;
    return (int64_t)sizeof(double) * D * (4 + (int64_t)T + 3 * Nchain);
}

template <typename T>
static int stream_update(const T* ring, int64_t Nchain, int32_t D, int32_t R, int64_t n, int32_t Tl, int64_t j0, int64_t j1, double* ws,
                         cudaStream_t stream) {
    double* rows = ws;
    double* lags = ws + 4 * (size_t)D;
    double* state = lags + (size_t)Tl * D;
    const long ilo = j0 > 1 ? j0 : 1, ihi = j1 < 2 * n + 1 ? j1 : 2 * n + 1;
    if (ilo >= ihi) return HMC_OK;
    const int gx = (D + kTile - 1) / kTile;
    stream_moments_kernel<T><<<dim3(gx, chain_groups((Nchain + kWarps - 1) / kWarps, gx, 8)), kTile * kWarps, 0, stream>>>(
        ring, Nchain, D, R, n, ilo, ihi, j0, j1, rows, state);
    HMC_CUDA_CHECK(cudaGetLastError());
    const size_t smem_max = sizeof(T) * kTile * (2 * kNewPerLaunch + kLagsPerLaunch);
    HMC_CUDA_CHECK(cudaFuncSetAttribute(stream_lags_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
    const dim3 grid(gx, chain_groups(Nchain, gx, 4));
    // pieces of at most 64 new indices inside one split chain, lags in launches of 128
    for (long lo = ilo; lo < ihi;) {
        const long s0 = lo <= n ? 1 : n + 1;
        const long send = lo <= n ? n + 1 : 2 * n + 1;
        long hi = lo + kNewPerLaunch;
        if (hi > send) hi = send;
        if (hi > ihi) hi = ihi;
        for (int tl = 1; tl <= Tl; tl += kLagsPerLaunch) {
            const int th = (Tl + 1 - tl < kLagsPerLaunch) ? Tl + 1 : tl + kLagsPerLaunch;
            if (hi - 1 - tl < s0) break;                      // no pair of these (or larger) lags stays inside the split chain
            const long elo = (s0 > lo - th + 1) ? s0 : lo - th + 1;
            const long nold = hi - tl - elo;
            const size_t smem = sizeof(T) * kTile * (size_t)((hi - lo) + (nold > 0 ? nold : 0));
            stream_lags_kernel<T><<<grid, kTile * kWarps, smem, stream>>>(ring, Nchain, D, R, s0, lo, hi, tl, th, j1, lags);
        }
        lo = hi;
    }
    HMC_CUDA_CHECK(cudaGetLastError());
    return HMC_OK;
}

extern "C" int hmc_diag_stream_update(int32_t dtype, const void* q_ring, int64_t Nchain, int32_t D, int32_t R, int64_t L_chain, int32_t T,
                                      int64_t j0, int64_t j1, void* workspace, int64_t workspace_bytes, void* cuda_stream) {
    HMC_REQUIRE(dtype == HMC_F32 || dtype == HMC_F64, "dtype must be HMC_F32 or HMC_F64");
    HMC_REQUIRE(q_ring != nullptr, "NULL q_ring");
    HMC_REQUIRE(Nchain >= 1 && D >= 1 && D <= kMaxD, "need Nchain >= 1 and 1 <= D <= %d", kMaxD);
    HMC_REQUIRE(L_chain >= 1, "need L_chain >= 1");
    const int64_t n = (L_chain - 1) / 2;                     // utils.py:96-102 (an odd number of used samples drops the last)
    HMC_REQUIRE(T >= 1 && T <= n - 1, "need 1 <= T <= n - 1 = %lld (L_chain = %lld), got T = %d", (long long)(n - 1), (long long)L_chain, T);
    HMC_REQUIRE(0 <= j0 && j0 <= j1 && j1 <= L_chain, "need 0 <= j0 <= j1 <= L_chain = %lld, got [%lld, %lld)", (long long)L_chain,
                (long long)j0, (long long)j1);
    HMC_REQUIRE(R >= 1 && (int64_t)R >= (int64_t)T + (j1 - j0), "the ring must hold T + (j1 - j0) = %lld rows, has R = %d",
                (long long)T + (j1 - j0), R);
    const int64_t need = hmc_diag_stream_workspace_bytes(Nchain, D, T);
    HMC_REQUIRE(workspace != nullptr && workspace_bytes >= need, "needs a workspace of %lld bytes (hmc_diag_stream_workspace_bytes)",
                (long long)need);
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    if (j0 == 0) HMC_CUDA_CHECK(cudaMemsetAsync(workspace, 0, sizeof(double) * D * (4 + (size_t)T), stream));
    if (dtype == HMC_F32) return stream_update<float>((const float*)q_ring, Nchain, D, R, n, T, j0, j1, (double*)workspace, stream);
    return stream_update<double>((const double*)q_ring, Nchain, D, R, n, T, j0, j1, (double*)workspace, stream);
}

extern "C" int hmc_diag_stream_finish(const void* workspace, int64_t workspace_bytes, int32_t D, int32_t T, double* out4xD,
                                      double* out_lags, void* cuda_stream) {
    HMC_REQUIRE(D >= 1 && D <= kMaxD && T >= 1 && T <= kMaxT, "need 1 <= D <= %d and T >= 1", kMaxD);
    HMC_REQUIRE(workspace != nullptr && workspace_bytes >= (int64_t)sizeof(double) * D * (4 + (int64_t)T),
                "needs the workspace hmc_diag_stream_update filled");
    HMC_REQUIRE(out4xD && out_lags, "NULL buffer");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const double* ws = (const double*)workspace;
    HMC_CUDA_CHECK(cudaMemcpyAsync(out4xD, ws, sizeof(double) * 4 * D, cudaMemcpyDeviceToDevice, stream));
    HMC_CUDA_CHECK(cudaMemcpyAsync(out_lags, ws + 4 * (size_t)D, sizeof(double) * (size_t)T * D, cudaMemcpyDeviceToDevice, stream));
    return HMC_OK;
}
