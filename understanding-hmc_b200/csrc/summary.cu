// Start points and sample summaries on the device (SURVEY 8f rows 2 and 4):
//   hmc_start_pts        -- utils.start_pts (/root/reference/utils.py:204-209): q_m = q0 + Lc z_m, z ~ N(0, I)
//   hmc_summary_moments  -- per-dimension sum and sum of squares over all chains and samples
//                           (plot_samples' inferred mean / variance per dimension, samplers.py:209-216, 244-250)
//   hmc_summary_hist     -- histogram of one strided series on explicit bin edges (np.histogram semantics;
//                           plot_samples' q1 / q2 / E / dE histograms, samplers.py:95-113, 160-186)
//   hmc_summary_select   -- one radix-select pass (11-bit digit histogram of the order-preserving integer keys under a
//                           key prefix): the host walks the digits to the k-th smallest value, which gives np.percentile
//                           exactly (samplers.py:95-113, 177-180 use the 2.5 / 97.5 percentiles for the plot ranges)
// All of them are HBM-bound passes over device-resident outputs: at 65,536 chains the host never sees q_chain (26 GB).
#include "hmc_common.cuh"

namespace {

// one warp per chain: z staged in shared memory, lane j computes rows j, j+32, ... of q0 + Lc z (Lc lower triangular,
// row-major) or q0 + sd .* z
template <typename T>
__global__ void __launch_bounds__(128) start_pts_kernel(uint64_t seed, int64_t chain_id0, long Nchain, int D, const double* __restrict__ q0,
                                                       const double* __restrict__ Lc, const double* __restrict__ sd, T* __restrict__ out) {
    extern __shared__ float zs_all[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int Dp = (D + 3) & ~3;
    float* zs = zs_all + (size_t)warp * Dp;
    for (long m = (long)blockIdx.x * (blockDim.x >> 5) + warp; m < Nchain; m += (long)gridDim.x * (blockDim.x >> 5)) {
        const uint64_t gid = (uint64_t)(chain_id0 + m);
        for (int s = lane; s < Dp / 4; s += 32) *reinterpret_cast<float4*>(zs + 4 * s) = hmc_start_normal4(seed, gid, (uint32_t)s);
        __syncwarp();
        for (int j = lane; j < D; j += 32) {
            double v = q0[j];
            if (Lc) {
                const double* row = Lc + (size_t)j * D;
                for (int k = 0; k <= j; ++k) v = fma(row[k], (double)zs[k], v);
            } else {
                v = fma(sd[j], (double)zs[j], v);
            }
            out[(size_t)m * D + j] = (T)v;
        }
        __syncwarp();
    }
}

// per-dimension sum / sum of squares of rows [Nchain][nsamp] x D (row pitch `pitch`); thread = (series, dimension)
template <typename T>
__global__ void __launch_bounds__(256) summary_moments_kernel(const T* __restrict__ q, long Nchain, long nsamp, int D, long pitch,
                                                              long stride_chain, int d0, int Dt, int spb, double* __restrict__ out) {
    extern __shared__ double sm[];   // [2][Dt]
    for (int t = threadIdx.x; t < 2 * Dt; t += blockDim.x) sm[t] = 0.0;
    __syncthreads();
    const int d = threadIdx.x % Dt, sl = threadIdx.x / Dt;
    if (sl < spb) {
        double a = 0.0, b = 0.0;
        for (long s = (long)blockIdx.x * spb + sl; s < Nchain; s += (long)gridDim.x * spb) {
            const T* x = q + s * stride_chain + d0 + d;
            long i = 0;
            for (; i + 8 <= nsamp; i += 8) {
                T v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = x[(i + u) * pitch];
#pragma unroll
                for (int u = 0; u < 8; ++u) { a += (double)v[u]; b = fma((double)v[u], (double)v[u], b); }
            }
            for (; i < nsamp; ++i) { const double v = (double)x[i * pitch]; a += v; b = fma(v, v, b); }
        }
        atomicAdd(&sm[d], a);
        atomicAdd(&sm[Dt + d], b);
    }
    __syncthreads();
    for (int t = threadIdx.x; t < Dt; t += blockDim.x) { atomicAdd(out + d0 + t, sm[t]); atomicAdd(out + D + d0 + t, sm[Dt + t]); }
}

// float32 rows, D % 4 == 0: thread = (series, four adjacent dimensions), 128-bit loads, eight rows in flight
__global__ void __launch_bounds__(256) summary_moments_f32x4_kernel(const float* __restrict__ q, long Nchain, long nsamp, int D, long pitch,
                                                                    long stride_chain, int spb, double* __restrict__ out) {
    extern __shared__ double sm[];   // [2][D]
    for (int t = threadIdx.x; t < 2 * D; t += blockDim.x) sm[t] = 0.0;
    __syncthreads();
    const int D4 = D >> 2, dq = threadIdx.x % D4, sl = threadIdx.x / D4;
    if (sl < spb) {
        double a[4] = {0, 0, 0, 0}, b[4] = {0, 0, 0, 0};
        for (long s = (long)blockIdx.x * spb + sl; s < Nchain; s += (long)gridDim.x * spb) {
            const float* x = q + s * stride_chain + 4 * dq;
            const float4 x0 = *reinterpret_cast<const float4*>(x);      // shift: float partial sums stay small and accurate
            double sa[4] = {0, 0, 0, 0}, sb[4] = {0, 0, 0, 0};
            long i = 0;
            for (; i + 8 <= nsamp; i += 8) {
                float4 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = *reinterpret_cast<const float4*>(x + (i + u) * pitch);
                float pa[4] = {0.f, 0.f, 0.f, 0.f}, pb[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const float e0 = v[u].x - x0.x, e1 = v[u].y - x0.y, e2 = v[u].z - x0.z, e3 = v[u].w - x0.w;
                    pa[0] += e0; pa[1] += e1; pa[2] += e2; pa[3] += e3;
                    pb[0] = fmaf(e0, e0, pb[0]); pb[1] = fmaf(e1, e1, pb[1]); pb[2] = fmaf(e2, e2, pb[2]); pb[3] = fmaf(e3, e3, pb[3]);
                }
#pragma unroll
                for (int c = 0; c < 4; ++c) { sa[c] += (double)pa[c]; sb[c] += (double)pb[c]; }
            }
            for (; i < nsamp; ++i) {
                const float4 v = *reinterpret_cast<const float4*>(x + i * pitch);
                const double e[4] = {(double)v.x - x0.x, (double)v.y - x0.y, (double)v.z - x0.z, (double)v.w - x0.w};
#pragma unroll
                for (int c = 0; c < 4; ++c) { sa[c] += e[c]; sb[c] += e[c] * e[c]; }
            }
            // un-shift: sum x = sum e + n x0, sum x^2 = sum e^2 + 2 x0 sum e + n x0^2
            const double xs[4] = {(double)x0.x, (double)x0.y, (double)x0.z, (double)x0.w};
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                a[c] += sa[c] + (double)nsamp * xs[c];
                b[c] += sb[c] + 2.0 * xs[c] * sa[c] + (double)nsamp * xs[c] * xs[c];
            }
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) { atomicAdd(&sm[4 * dq + c], a[c]); atomicAdd(&sm[D + 4 * dq + c], b[c]); }
    }
    __syncthreads();
    for (int t = threadIdx.x; t < 2 * D; t += blockDim.x) atomicAdd(out + t, sm[t]);
}

// order-preserving integer keys
__device__ __forceinline__ unsigned long long key_of(float v) {
    const unsigned int u = __float_as_uint(v);
    return (unsigned long long)((u & 0x80000000u) ? ~u : (u | 0x80000000u));
}
__device__ __forceinline__ unsigned long long key_of(double v) {
    const unsigned long long u = (unsigned long long)__double_as_longlong(v);
    return (u & 0x8000000000000000ull) ? ~u : (u | 0x8000000000000000ull);
}

constexpr int kSelBins = 2048;

template <typename T>
__global__ void __launch_bounds__(256) summary_select_kernel(const T* __restrict__ x, long Nchain, long nsamp, long stride_sample,
                                                             long stride_chain, unsigned long long prefix, int prefix_shift,
                                                             int digit_shift, int digit_bits, unsigned long long* __restrict__ out) {
    __shared__ unsigned int h[kSelBins];
    for (int t = threadIdx.x; t < kSelBins; t += blockDim.x) h[t] = 0u;
    __syncthreads();
    const long total = Nchain * nsamp;
    const unsigned int mask = (1u << digit_bits) - 1u;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const long c = t / nsamp, s = t - c * nsamp;
        const unsigned long long k = key_of(x[c * stride_chain + s * stride_sample]);
        if (prefix_shift >= 64 || (k >> prefix_shift) == prefix) atomicAdd(&h[(unsigned int)(k >> digit_shift) & mask], 1u);
    }
    __syncthreads();
    for (int t = threadIdx.x; t < kSelBins; t += blockDim.x) if (h[t]) atomicAdd(out + t, (unsigned long long)h[t]);
}

constexpr int kHistMaxBins = 4096;

// counts[i] = #{ edges[i] <= v < edges[i+1] } (last bin closed on the right, np.histogram), v = x - shift;
// counts[nbins] = below the first edge, counts[nbins + 1] = above the last edge (NaN counts as above)
template <typename T>
__global__ void __launch_bounds__(256) summary_hist_kernel(const T* __restrict__ x, long Nchain, long nsamp, long stride_sample,
                                                           long stride_chain, double shift, const double* __restrict__ edges, int nbins,
                                                           unsigned long long* __restrict__ out) {
    extern __shared__ unsigned char raw[];
    double* e = reinterpret_cast<double*>(raw);                  // [nbins + 1]
    unsigned int* h = reinterpret_cast<unsigned int*>(e + nbins + 1);   // [nbins + 2]
    for (int t = threadIdx.x; t <= nbins; t += blockDim.x) e[t] = edges[t];
    for (int t = threadIdx.x; t < nbins + 2; t += blockDim.x) h[t] = 0u;
    __syncthreads();
    const double e0 = e[0], eN = e[nbins], inv = (double)nbins / (eN - e0);
    const long total = Nchain * nsamp;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const long c = t / nsamp, s = t - c * nsamp;
        const double v = (double)x[c * stride_chain + s * stride_sample] - shift;
        int b;
        if (v < e0) b = nbins;
        else if (!(v <= eN)) b = nbins + 1;
        else {
            b = (int)((v - e0) * inv);
            b = b < 0 ? 0 : (b > nbins - 1 ? nbins - 1 : b);
            while (b > 0 && v < e[b]) --b;                      // exact with respect to the given edges
            while (b < nbins - 1 && v >= e[b + 1]) ++b;
        }
        atomicAdd(&h[b], 1u);
    }
    __syncthreads();
    for (int t = threadIdx.x; t < nbins + 2; t += blockDim.x) if (h[t]) atomicAdd(out + t, (unsigned long long)h[t]);
}

int sm_count() {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    return sms;
}

}  // namespace

#define HMC_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            hmc_set_error(__VA_ARGS__);   \
            return HMC_E_BADARG;          \
        }                                 \
    } while (0)

extern "C" int hmc_start_pts(int32_t dtype, uint64_t seed, int64_t chain_id0, int64_t Nchain, int32_t D, const double* q0,
                             const double* Lc, const double* sd, void* out, void* cuda_stream) {
    HMC_REQUIRE(dtype == HMC_F32 || dtype == HMC_F64, "dtype must be HMC_F32 or HMC_F64");
    HMC_REQUIRE(Nchain >= 1 && D >= 1 && D <= 4096 && q0 && out && (Lc || sd), "need Nchain >= 1, 1 <= D <= 4096, q0, out and Lc or sd");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    const int warps = 4;
    const size_t smem = sizeof(float) * warps * ((D + 3) & ~3);
    long blocks = (Nchain + warps - 1) / warps;
    const long cap = (long)sm_count() * 16;
    if (blocks > cap) blocks = cap;
    if (smem > 48 * 1024) {                          // (above D = 3072 the z rows need the opt-in to more than 48 KB)
        HMC_CUDA_CHECK(cudaFuncSetAttribute(start_pts_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        HMC_CUDA_CHECK(cudaFuncSetAttribute(start_pts_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    if (dtype == HMC_F32) start_pts_kernel<float><<<(int)blocks, warps * 32, smem, stream>>>(seed, chain_id0, Nchain, D, q0, Lc, sd, (float*)out);
    else start_pts_kernel<double><<<(int)blocks, warps * 32, smem, stream>>>(seed, chain_id0, Nchain, D, q0, Lc, sd, (double*)out);
    HMC_CUDA_CHECK(cudaGetLastError());
    return HMC_OK;
}

extern "C" int hmc_summary_moments(int32_t dtype, const void* q, int64_t Nchain, int64_t nsamp, int32_t D, int64_t pitch,
                                   int64_t stride_chain, double* out2xD, void* cuda_stream) {
    HMC_REQUIRE(dtype == HMC_F32 || dtype == HMC_F64, "dtype must be HMC_F32 or HMC_F64");
    HMC_REQUIRE(q && out2xD && Nchain >= 1 && nsamp >= 1 && D >= 1 && pitch >= D, "bad arguments");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    HMC_CUDA_CHECK(cudaMemsetAsync(out2xD, 0, sizeof(double) * 2 * D, stream));
    const int sms = sm_count();
    if (dtype == HMC_F32 && D % 4 == 0 && D <= 1024 && pitch % 4 == 0 && stride_chain % 4 == 0 && (reinterpret_cast<uintptr_t>(q) % 16) == 0) {
        const int spb = 256 / (D / 4);
        long grid = (Nchain + spb - 1) / spb;
        if (grid > (long)sms * 8) grid = (long)sms * 8;
        summary_moments_f32x4_kernel<<<(int)grid, 256, sizeof(double) * 2 * D, stream>>>((const float*)q, Nchain, nsamp, D, pitch, stride_chain, spb, out2xD);
    } else {
        for (int d0 = 0; d0 < D; d0 += 256) {               // tiles of at most 256 dimensions
            const int Dt = (D - d0 < 256) ? D - d0 : 256;
            const int spb = 256 / Dt;
            long grid = (Nchain + spb - 1) / spb;
            if (grid > (long)sms * 8) grid = (long)sms * 8;
            if (dtype == HMC_F32)
                summary_moments_kernel<float><<<(int)grid, 256, sizeof(double) * 2 * Dt, stream>>>((const float*)q, Nchain, nsamp, D, pitch, stride_chain, d0, Dt, spb, out2xD);
            else
                summary_moments_kernel<double><<<(int)grid, 256, sizeof(double) * 2 * Dt, stream>>>((const double*)q, Nchain, nsamp, D, pitch, stride_chain, d0, Dt, spb, out2xD);
        }
    }
    HMC_CUDA_CHECK(cudaGetLastError());
    return HMC_OK;
}

extern "C" int hmc_summary_select(int32_t dtype, const void* x, int64_t Nchain, int64_t nsamp, int64_t stride_sample,
                                  int64_t stride_chain, uint64_t prefix, int32_t prefix_shift, int32_t digit_shift,
                                  int32_t digit_bits, unsigned long long* out_hist2048, void* cuda_stream) {
    HMC_REQUIRE(dtype == HMC_F32 || dtype == HMC_F64, "dtype must be HMC_F32 or HMC_F64");
    HMC_REQUIRE(x && out_hist2048 && Nchain >= 1 && nsamp >= 1, "bad arguments");
    HMC_REQUIRE(digit_bits >= 1 && digit_bits <= 11 && digit_shift >= 0 && digit_shift < 64 && prefix_shift >= 1 && prefix_shift <= 64,
                "need 1 <= digit_bits <= 11, 0 <= digit_shift < 64, 1 <= prefix_shift <= 64");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    HMC_CUDA_CHECK(cudaMemsetAsync(out_hist2048, 0, sizeof(unsigned long long) * kSelBins, stream));
    long grid = (Nchain * nsamp + 255) / 256;
    const long cap = (long)sm_count() * 8;
    if (grid > cap) grid = cap;
    if (dtype == HMC_F32)
        summary_select_kernel<float><<<(int)grid, 256, 0, stream>>>((const float*)x, Nchain, nsamp, stride_sample, stride_chain, prefix, prefix_shift, digit_shift, digit_bits, out_hist2048);
    else
        summary_select_kernel<double><<<(int)grid, 256, 0, stream>>>((const double*)x, Nchain, nsamp, stride_sample, stride_chain, prefix, prefix_shift, digit_shift, digit_bits, out_hist2048);
    HMC_CUDA_CHECK(cudaGetLastError());
    return HMC_OK;
}

extern "C" int hmc_summary_hist(int32_t dtype, const void* x, int64_t Nchain, int64_t nsamp, int64_t stride_sample,
                                int64_t stride_chain, double shift, const double* edges, int32_t nbins,
                                unsigned long long* out_counts, void* cuda_stream) {
    HMC_REQUIRE(dtype == HMC_F32 || dtype == HMC_F64, "dtype must be HMC_F32 or HMC_F64");
    HMC_REQUIRE(x && edges && out_counts && Nchain >= 1 && nsamp >= 1, "bad arguments");
    HMC_REQUIRE(nbins >= 1 && nbins <= kHistMaxBins, "need 1 <= nbins <= %d", kHistMaxBins);
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    HMC_CUDA_CHECK(cudaMemsetAsync(out_counts, 0, sizeof(unsigned long long) * (nbins + 2), stream));
    long grid = (Nchain * nsamp + 255) / 256;
    const long cap = (long)sm_count() * 8;
    if (grid > cap) grid = cap;
    const size_t smem = sizeof(double) * (nbins + 1) + sizeof(unsigned int) * (nbins + 2);
    if (dtype == HMC_F32) {
        HMC_CUDA_CHECK(cudaFuncSetAttribute(summary_hist_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        summary_hist_kernel<float><<<(int)grid, 256, smem, stream>>>((const float*)x, Nchain, nsamp, stride_sample, stride_chain, shift, edges, nbins, out_counts);
    } else {
        HMC_CUDA_CHECK(cudaFuncSetAttribute(summary_hist_kernel<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        summary_hist_kernel<double><<<(int)grid, 256, smem, stream>>>((const double*)x, Nchain, nsamp, stride_sample, stride_chain, shift, edges, nbins, out_counts);
    }
    HMC_CUDA_CHECK(cudaGetLastError());
    return HMC_OK;
}
