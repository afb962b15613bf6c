// Shared device helpers: Philox4x32-10, Box-Muller, draw keying, error plumbing.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include "../../include/hmc_b200.h"

#define HMC_FULL_MASK 0xffffffffu

void hmc_set_error(const char* fmt, ...);
#define HMC_CUDA_CHECK(expr)                                                                   \
    do {                                                                                       \
        cudaError_t _e = (expr);                                                               \
        if (_e != cudaSuccess) {                                                               \
            hmc_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return HMC_E_CUDA;                                                                 \
        }                                                                                      \
    } while (0)

// ---------------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011), counter-based: every draw is a pure function of
// (seed, global chain id, iteration, slot, stream) so chains can be sharded over any number of GPUs.
// ---------------------------------------------------------------------------------------------------------
struct Philox4 {
    uint32_t x, y, z, w;
};

__host__ __device__ __forceinline__ Philox4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                                                          uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * c0;
        uint64_t p1 = (uint64_t)M1 * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    Philox4 o; o.x = c0; o.y = c1; o.z = c2; o.w = c3;
    return o;
}

// stored-sample index of iteration `it` (samplers.py:436, 468: (i - warm_up_num) // thin_rate); below L_chain by construction, so
// only a ring of the last `store_ring` samples wraps.  32-bit on purpose: a 64-bit `% Lrow` is a software division in the middle
// of the per-trajectory service code (measured in the tensor-core kernel: 400 cycles of its 1,800-cycle bookkeeping phase).
__device__ __forceinline__ long hmc_store_index(int it, int warm_up_num, int thin_rate, long Lrow, bool ring) {
    int idx = (thin_rate == 1) ? it - warm_up_num : (it - warm_up_num) / thin_rate;
    if (ring) idx = (int)((unsigned int)idx % (unsigned int)Lrow);
    return (long)idx;
}

enum { HMC_STREAM_MOMENTUM = 0, HMC_STREAM_SCALAR = 1, HMC_STREAM_NUTS = 2, HMC_STREAM_START = 4 };

// 4 standard normals for dims 4*slot .. 4*slot+3 of a start point (hmc_start_pts, hmc_start_pts_bigd: both draw the same z)
__device__ __forceinline__ float4 hmc_start_normal4(uint64_t seed, uint64_t gid, uint32_t slot) {
    const Philox4 r = philox4x32_10((uint32_t)gid, 0u, slot, HMC_STREAM_START | ((uint32_t)(gid >> 32) << 8),
                                    (uint32_t)seed, (uint32_t)(seed >> 32));
    // Box-Muller, full-precision logf / sincosf (not on a hot path)
    const float u1 = ((float)(r.x >> 8) + 0.5f) * 5.9604644775390625e-08f, u2 = ((float)(r.z >> 8) + 0.5f) * 5.9604644775390625e-08f;
    const float r1 = sqrtf(-2.0f * logf(u1)), r2 = sqrtf(-2.0f * logf(u2));
    const float a1 = ((float)(r.y >> 8) * 5.9604644775390625e-08f - 0.5f) * 6.283185307179586f;
    const float a2 = ((float)(r.w >> 8) * 5.9604644775390625e-08f - 0.5f) * 6.283185307179586f;
    float s1, c1, s2, c2;
    sincosf(a1, &s1, &c1);
    sincosf(a2, &s2, &c2);
    return make_float4(r1 * c1, r1 * s1, r2 * c2, r2 * s2);
}

// 4 standard normals for dims 4*slot .. 4*slot+3 of (chain, iteration): float32 Box-Muller.
__device__ __forceinline__ float4 hmc_normal4(uint64_t seed, uint64_t chain, uint32_t iter, uint32_t slot) {
    Philox4 r = philox4x32_10((uint32_t)chain, iter, slot, HMC_STREAM_MOMENTUM | ((uint32_t)(chain >> 32) << 8),
                              (uint32_t)seed, (uint32_t)(seed >> 32));
    // Box-Muller on the SFU (MUFU.LG2 / MUFU.SIN / MUFU.COS, abs. error ~2^-21): the refresh is on the hot path
    // of the fused kernel; every kernel and hmc_philox_draws share this function, so all see identical draws.
    const float u1 = ((float)(r.x >> 8) + 0.5f) * 5.9604644775390625e-08f;  // (0,1), 24 bits
    const float u2 = ((float)(r.z >> 8) + 0.5f) * 5.9604644775390625e-08f;
    const float r1 = sqrtf(-2.0f * __logf(u1));
    const float r2 = sqrtf(-2.0f * __logf(u2));
    const float a1 = ((float)(r.y >> 8) * 5.9604644775390625e-08f - 0.5f) * 6.283185307179586f;   // [-pi, pi)
    const float a2 = ((float)(r.w >> 8) * 5.9604644775390625e-08f - 0.5f) * 6.283185307179586f;
    const float s1 = __sinf(a1), c1 = __cosf(a1), s2 = __sinf(a2), c2 = __cosf(a2);
    return make_float4(r1 * c1, r1 * s1, r2 * c2, r2 * s2);
}

// Trajectory length in {L_low .. L_high-1} and acceptance uniform in (0,1) for (chain, iteration).
__device__ __forceinline__ void hmc_scalar_draws(uint64_t seed, uint64_t chain, uint32_t iter, int L_low, int L_high,
                                                 int* L, double* u) {
    Philox4 r = philox4x32_10((uint32_t)chain, iter, 0u, HMC_STREAM_SCALAR | ((uint32_t)(chain >> 32) << 8),
                              (uint32_t)seed, (uint32_t)(seed >> 32));
    *L = L_low + (int)__umulhi(r.x, (uint32_t)(L_high - L_low));
    *u = ((double)(r.y >> 8) + 0.5) * 5.9604644775390625e-08;   // 24-bit uniform in (0,1): exact in float and double
}

// NUTS per-chain stream: draw number n of iteration iter -> (coin, uniform).
__device__ __forceinline__ void hmc_nuts_draw(uint64_t seed, uint64_t chain, uint32_t iter, uint32_t n, int* coin,
                                              double* u) {
    Philox4 r = philox4x32_10((uint32_t)chain, iter, n, HMC_STREAM_NUTS | ((uint32_t)(chain >> 32) << 8),
                              (uint32_t)seed, (uint32_t)(seed >> 32));
    *coin = (int)(r.x >> 31);
    *u = ((double)r.y + 0.5) * 2.3283064365386963e-10;
}

template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(HMC_FULL_MASK, v, o);
    return v;
}

// ---------------------------------------------------------------------------------------------------------
// Warp-distributed vectors used by the one-warp-per-chain kernels: register i of lane l holds dimension
// hmc_dim<NJ>(l, i).  NJ % 4 == 0: blocks of 4 adjacent dimensions per lane (128-bit shared/global accesses, one
// Philox call per block); NJ < 4 (D <= 32): strided, so that small D still spreads over the lanes.
// ---------------------------------------------------------------------------------------------------------
template <int NJ>
__device__ __forceinline__ int hmc_dim(int lane, int i) {
    if constexpr (NJ % 4 == 0) return (i >> 2) * 128 + 4 * lane + (i & 3);
    else return lane + 32 * i;
}

__device__ __forceinline__ void hmc_load4(const float* p, float (&v)[4]) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
}
__device__ __forceinline__ void hmc_load4(const double* p, double (&v)[4]) {
    const double2 t0 = *reinterpret_cast<const double2*>(p), t1 = *reinterpret_cast<const double2*>(p + 2);
    v[0] = t0.x; v[1] = t0.y; v[2] = t1.x; v[3] = t1.y;
}

// explicit shared-space loads (the matrix pointer is chosen at run time, so the compiler would otherwise emit
// generic-address LD.E instead of LDS)
__device__ __forceinline__ void hmc_lds4(uint32_t addr, float (&v)[4]) {
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[0]), "=f"(v[1]), "=f"(v[2]), "=f"(v[3]) : "r"(addr));
}
__device__ __forceinline__ void hmc_lds4(uint32_t addr, double (&v)[4]) {
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v[0]), "=d"(v[1]) : "r"(addr));
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v[2]), "=d"(v[3]) : "r"(addr + 16));
}

// y = M x for a D x D matrix given by its transpose Mt[k][j] (row pitch Dp, a multiple of 4, columns >= D zero);
// x, y distributed over the warp.  x is staged in a per-warp shared buffer (Dp entries) and read back as a
// broadcast, four k at a time.  SM = the matrix sits in shared memory with Dp zero-padded ROWS as well, so the
// k loop needs no bounds checks.
template <typename T, int NJ, bool SM>
__device__ __forceinline__ void matvec_t(const T* __restrict__ Mt, int D, int Dp, const T (&x)[NJ], T (&y)[NJ],
                                         int lane, T* __restrict__ xs) {
#pragma unroll
    for (int i = 0; i < NJ; ++i) { y[i] = T(0); const int j = hmc_dim<NJ>(lane, i); if (j < Dp) xs[j] = (j < D) ? x[i] : T(0); }
    __syncwarp();
    if constexpr (NJ % 4 == 0 && SM) {
        const uint32_t xs_a = (uint32_t)__cvta_generic_to_shared(xs);
        const uint32_t m_a = (uint32_t)__cvta_generic_to_shared(Mt) + (uint32_t)(4 * lane * sizeof(T));
        const uint32_t pitch = (uint32_t)(Dp * sizeof(T));
        const bool on = 4 * lane < Dp;
#pragma unroll 2
        for (int kb = 0; kb < Dp; kb += 4) {
            T xk[4];
            hmc_lds4(xs_a + (uint32_t)(kb * sizeof(T)), xk);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
                for (int i4 = 0; i4 < NJ / 4; ++i4) {
                    if (i4 == 0 ? on : (i4 * 128 + 4 * lane < Dp)) {
                        T v[4];
                        hmc_lds4(m_a + (uint32_t)(kb + kk) * pitch + (uint32_t)(i4 * 128 * sizeof(T)), v);
#pragma unroll
                        for (int c = 0; c < 4; ++c) y[4 * i4 + c] = fma(v[c], xk[kk], y[4 * i4 + c]);
                    }
                }
            }
        }
    } else if constexpr (NJ % 4 == 0) {
        for (int kb = 0; kb < D; kb += 4) {
            T xk[4];
            hmc_load4(xs + kb, xk);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                if (kb + kk < D) {
                    const T* row = Mt + (size_t)(kb + kk) * Dp;
#pragma unroll
                    for (int i4 = 0; i4 < NJ / 4; ++i4) {
                        const int j0 = i4 * 128 + 4 * lane;
                        if (j0 < Dp) {
                            T v[4];
                            hmc_load4(row + j0, v);
#pragma unroll
                            for (int c = 0; c < 4; ++c) y[4 * i4 + c] = fma(v[c], xk[kk], y[4 * i4 + c]);
                        }
                    }
                }
            }
        }
    } else {
#pragma unroll 2
        for (int k = 0; k < D; ++k) {
            const T xk = xs[k];
            const T* row = Mt + (size_t)k * Dp;
#pragma unroll
            for (int i2 = 0; i2 < NJ; ++i2) {
                const int j = hmc_dim<NJ>(lane, i2);
                if (j < D) y[i2] = fma(row[j], xk, y[i2]);
            }
        }
    }
    __syncwarp();
}

template <typename T, int NJ>
__device__ __forceinline__ double dot_warp(const T (&a)[NJ], const T (&b)[NJ]) {
    T s = T(0);
#pragma unroll
    for (int i = 0; i < NJ; ++i) s = fma(a[i], b[i], s);
    return warp_sum<double>((double)s);
}

