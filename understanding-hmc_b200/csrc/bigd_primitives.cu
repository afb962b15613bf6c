// Large-D primitives on the tcgen05 GEMM of bigd_gemm.cuh, for every 128 <= D <= 8192 (float32).  Both are dense products of a
// batch of rows with one D x D matrix, the shape the samplers' GEMM already runs:
//
//   hmc_start_pts_bigd   utils.start_pts (reference utils.py:204-209): Q = q0 + Z Lc^T.
//                        start_draw         one warp per row: the Philox normals z of hmc_start_pts (hmc_start_normal4, same keying,
//                                           so the two entry points draw the same z), zero from D on and in the padding rows,
//                                           written straight as the three bf16 parts of the A operand (a float32 z splits exactly)
//                        start_split_lc     Lc (float64, row-major, lower triangle read) rounded to float32 and split into three
//                                           bf16 parts = the B operand (fp32-grade: the rounding to float32 is the only error of
//                                           the operands; the GEMM drops the part products below 2^-24 and accumulates in fp32)
//                        bigd_gemm_step<EPI_GRAD>  the fp32 rows Z Lc^T, Dp wide
//                        start_finish       q0 + (Z Lc^T) in float64, rounded to float32, into the D-wide caller rows
//                        With sd (diagonal cov0) the whole call is start_diag, elementwise, no GEMM, and gives hmc_start_pts's rows bit
//                        for bit.  The all-zero K blocks above the diagonal of Lc are multiplied like the others.
//
//   hmc_leap_frog_bigd   HMC_sampler.leap_frog (samplers.py:831-839) for B rows: the Random path's fused EPI_LEAPFROG epilogue run as a
//                        trajectory of fixed length nsteps with no accept step, every row in the same phase: pass 0 MD_FIRST (half
//                        kick + drift), passes 1 .. nsteps - 1 MD_MID (the closing half kick of a step and the opening one of the
//                        next merged into one full kick, + drift), pass nsteps MD_LAST (half kick): nsteps + 1 GEMMs.  The per-pass
//                        phase is one of three constant mode rows the by-value workspace struct points at.  Only target.Ft, mu and dt
//                        enter, so any metric runs (Ft = (M^-1 P)^T).
#include "bigd_gemm.cuh"

namespace {

// ---------------------------------------------------------------------------------------------------------------------------
// start points
// ---------------------------------------------------------------------------------------------------------------------------
struct StartWs {
    uint16_t* xp;        // [3][Ncp][Dp] split normals (A operand), zero from D on and in the padding rows
    uint16_t* bp;        // [3][Dp][Dp]  split Lc (B operand): bp[part][n][k] = part(Lc[n][k]), zero above the diagonal and outside D x D
    float* g;            // [Ncp][Dp]    Z Lc^T
    int* mode;           // [Ncp] MD_FIRST for a chain, MD_IDLE for a padding row (the gradient epilogue stores rows of live warps)
    int* tile_active;    // [Ncp / 128]
    float binv;          // 1: the bf16 split is not scaled
    int Ncp, NT, Dp;
};

size_t carve_start(StartWs& w, unsigned char* ws, long Nchain, int D) {
    BigdCarve c(ws, Nchain, D, 128);
    w.Ncp = (int)c.Ncp; w.NT = c.NT; w.Dp = c.Dp; w.binv = 1.f;
    w.xp = (uint16_t*)c.take((size_t)3 * c.Ncp * c.Dp * 2);
    w.bp = (uint16_t*)c.take((size_t)3 * c.Dp * c.Dp * 2);
    w.g = (float*)c.take((size_t)c.Ncp * c.Dp * 4);
    w.mode = (int*)c.take(c.Ncp * 4);
    w.tile_active = (int*)c.take((c.Ncp / BM) * 4);
    return c.off;
}

__global__ void __launch_bounds__(256) start_draw(uint64_t seed, int64_t chain_id0, long Nchain, int D, StartWs w) {
    const int lane = threadIdx.x & 31, Dp = w.Dp;
    const long m = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (m >= w.Ncp) return;
    const uint64_t gid = (uint64_t)(chain_id0 + m);
    for (int s = lane; s < Dp / 4; s += 32) {
        float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m < Nchain && 4 * s < D) {
            z = hmc_start_normal4(seed, gid, (uint32_t)s);
            if (4 * s + 3 >= D) z.w = 0.f;
            if (4 * s + 2 >= D) z.z = 0.f;
            if (4 * s + 1 >= D) z.y = 0.f;
        }
        uint32_t h0[3], h1[3];
        split_pair<3>(z.x, z.y, h0);
        split_pair<3>(z.z, z.w, h1);
#pragma unroll
        for (int pt = 0; pt < 3; ++pt) reinterpret_cast<uint2*>(w.xp + ((size_t)pt * w.Ncp + m) * Dp)[s] = make_uint2(h0[pt], h1[pt]);
    }
    if (lane == 0) {
        w.mode[m] = m < Nchain ? MD_FIRST : MD_IDLE;
        if (m % BM == 0) w.tile_active[m / BM] = m < Nchain;
    }
}

__global__ void start_split_lc(const double* __restrict__ Lc, int D, int Dp, uint16_t* __restrict__ bp) {
    const long total = (long)Dp * (Dp / 2);
    for (long t = blockIdx.x * (long)blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const int n = (int)(t / (Dp / 2)), k = 2 * (int)(t % (Dp / 2));
        const float f0 = (n < D && k <= n) ? (float)Lc[(size_t)n * D + k] : 0.f;
        const float f1 = (n < D && k + 1 <= n) ? (float)Lc[(size_t)n * D + k + 1] : 0.f;
        uint32_t h[3];
        split_pair<3>(f0, f1, h);
#pragma unroll
        for (int pt = 0; pt < 3; ++pt) reinterpret_cast<uint32_t*>(bp + ((size_t)pt * Dp + n) * Dp)[k >> 1] = h[pt];
    }
}

// the caller's rows are D wide (not 16-byte aligned when D % 4 != 0): plain 4-byte accesses, one block per row
__global__ void __launch_bounds__(256) start_finish(const float* __restrict__ g, int Dp, long Nchain, int D, const double* __restrict__ q0,
                                                    float* __restrict__ out) {
    for (long m = blockIdx.x; m < Nchain; m += gridDim.x)
        for (int j = threadIdx.x; j < D; j += blockDim.x) out[(size_t)m * D + j] = (float)(q0[j] + (double)g[(size_t)m * Dp + j]);
}

// diagonal cov0: q = q0 + sd .* z, one warp per chain, the arithmetic of start_pts_kernel (summary.cu)
__global__ void __launch_bounds__(256) start_diag(uint64_t seed, int64_t chain_id0, long Nchain, int D, const double* __restrict__ q0,
                                                  const double* __restrict__ sd, float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    for (long m = (long)blockIdx.x * 8 + (threadIdx.x >> 5); m < Nchain; m += (long)gridDim.x * 8) {
        const uint64_t gid = (uint64_t)(chain_id0 + m);
        for (int s = lane; 4 * s < D; s += 32) {
            const float4 z4 = hmc_start_normal4(seed, gid, (uint32_t)s);
            const float z[4] = {z4.x, z4.y, z4.z, z4.w};
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const int j = 4 * s + c;
                if (j < D) out[(size_t)m * D + j] = (float)fma(sd[j], (double)z[c], q0[j]);
            }
        }
    }
}

constexpr const char* kStartName = "hmc_start_pts_bigd";

int run_start_pts(uint64_t seed, int64_t chain_id0, long Nchain, int D, const double* q0, const double* Lc, float* out, void* ws,
                  int64_t ws_bytes, cudaStream_t stream) {
    constexpr int NPART = 3, BN = 128, CL = 2, BK = 32, STAGES = 2;
    StartWs w;
    const size_t need = carve_start(w, (unsigned char*)ws, Nchain, D);
    if (int rc = bigd_check_workspace(ws, ws_bytes, need, kStartName, "hmc_start_pts_workspace_bytes")) return rc;
    int dev = 0, sms = 0;
    HMC_CUDA_CHECK(cudaGetDevice(&dev));
    HMC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int Dp = w.Dp;
    CUtensorMap mapA, mapB, mapG;
    if (int rc = make_map(&mapA, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, w.xp, (uint64_t)NPART * w.Ncp, Dp, BK, BM)) return rc;
    if (int rc = make_map(&mapB, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, w.bp, (uint64_t)NPART * Dp, Dp, BK, BN / CL)) return rc;
    if (int rc = make_map(&mapG, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, w.g, (uint64_t)w.Ncp, Dp, CW, 32)) return rc;
    start_draw<<<(w.Ncp + 7) / 8, 256, 0, stream>>>(seed, chain_id0, Nchain, D, w);
    start_split_lc<<<sms * 8, 256, 0, stream>>>(Lc, D, Dp, w.bp);
    auto kern = bigd_gemm_step<StartWs, EPI_GRAD, NPART, BN, CL, BK, STAGES>;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr;
    if (int rc = bigd_launch_config(cfg, attr, kern, CL, (w.Ncp / BM / CL) * w.NT, gemm_smem_bytes<NPART, BN, BK, STAGES>(), sms, stream,
                                    kStartName)) return rc;
    HMC_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, mapA, mapB, mapG, mapG, mapG, w, (int)Nchain, Dp, (const float*)nullptr));
    const long blocks = Nchain < (long)sms * 16 ? Nchain : (long)sms * 16;
    start_finish<<<(int)blocks, 256, 0, stream>>>(w.g, Dp, Nchain, D, q0, out);
    HMC_CUDA_CHECK(cudaGetLastError());
    return HMC_OK;
}

// ---------------------------------------------------------------------------------------------------------------------------
// leap frog
// ---------------------------------------------------------------------------------------------------------------------------
struct LfWs {
    uint16_t* xp;        // [2][NPART][Ncp][Dp] split position = A operand: pass n reads buffer n & 1, its epilogue writes the other one
    uint16_t* bp;        // [NPART][Dp][Dp] split force matrix (x 2^s for the fp16 split) = B operand, zero outside D x D
    float* x;            // [Ncp][Dp] q - mu
    float* p;            // [Ncp][Dp] momentum
    float* mu;           // [Dp] zero from D on
    float* dt;           // [Dp] zero from D on (the padded dimensions never move)
    float* red;          // [Ncp][NT][2][2] partial (q.g, p.p) the epilogue writes (no energies are needed here)
    int* modes;          // [3][Ncp] phase of every row in the first, an interior and the last pass; MD_IDLE in the padding rows
    int* mode;           // the row of `modes` of the pass being launched
    int* tile_active;    // [Ncp / 128]
    int* counters;       // [16] cleared by bigd_target_operands; word 8: abs-max scratch of the fp16 split
    float binv;          // 2^-s
    int Ncp, NT, Dp;
};

size_t carve_lf(LfWs& w, unsigned char* ws, long B, int D, int npart, int bn) {
    BigdCarve c(ws, B, D, bn);
    const long Ncp = c.Ncp;
    const int Dp = c.Dp;
    w.Ncp = (int)Ncp; w.NT = c.NT; w.Dp = Dp;
    w.xp = (uint16_t*)c.take((size_t)2 * npart * Ncp * Dp * 2);
    w.bp = (uint16_t*)c.take((size_t)npart * Dp * Dp * 2);
    w.x = (float*)c.take((size_t)Ncp * Dp * 4);
    w.p = (float*)c.take((size_t)Ncp * Dp * 4);
    w.mu = (float*)c.take((size_t)Dp * 4);
    w.dt = (float*)c.take((size_t)Dp * 4);
    w.red = (float*)c.take((size_t)Ncp * c.NT * 2 * 2 * 4);
    w.modes = (int*)c.take((size_t)3 * Ncp * 4);
    w.mode = w.modes;
    w.tile_active = (int*)c.take((Ncp / BM) * 4);
    w.counters = (int*)c.take(64);
    return c.off;
}

// rows of (p, q - mu), Dp wide and zero in the padding, the split position into operand buffer 0, the mode rows: one warp per row
template <int NPART>
__global__ void __launch_bounds__(256) lf_init(const float* __restrict__ p_old, const float* __restrict__ q_old, long B, int D, LfWs w) {
    const int lane = threadIdx.x & 31, Dp = w.Dp;
    const long m = (long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (m >= w.Ncp) return;
    float* xr = w.x + (size_t)m * Dp;
    float* pr = w.p + (size_t)m * Dp;
    const bool row = m < B;
    for (int j = lane; j < Dp; j += 32) {
        const bool in = row && j < D;
        xr[j] = in ? q_old[(size_t)m * D + j] - w.mu[j] : 0.f;
        pr[j] = in ? p_old[(size_t)m * D + j] : 0.f;
    }
    bigd_write_parts<NPART>(w.xp, w.Ncp, Dp, m, lane, xr);
    if (lane == 0) {
        w.modes[m] = row ? MD_FIRST : MD_IDLE;
        w.modes[w.Ncp + m] = row ? MD_MID : MD_IDLE;
        w.modes[2 * (size_t)w.Ncp + m] = row ? MD_LAST : MD_IDLE;
        if (m % BM == 0) w.tile_active[m / BM] = row;
    }
}

// (p, x + mu) back into the D-wide caller rows: plain 4-byte accesses (not 16-byte aligned when D % 4 != 0), one block per row
__global__ void __launch_bounds__(256) lf_end(const LfWs w, long B, int D, float* __restrict__ p_new, float* __restrict__ q_new) {
    const int Dp = w.Dp;
    for (long m = blockIdx.x; m < B; m += gridDim.x)
        for (int j = threadIdx.x; j < D; j += blockDim.x) {
            q_new[(size_t)m * D + j] = w.x[(size_t)m * Dp + j] + w.mu[j];
            p_new[(size_t)m * D + j] = w.p[(size_t)m * Dp + j];
        }
}

constexpr const char* kLfName = "hmc_leap_frog_bigd";

template <int NPART, int BN, int CL, int BK, int STAGES>
int run_leap_frog(const hmc_target& t, long B, const float* p_old, const float* q_old, float* p_new, float* q_new, int nsteps, void* ws,
                  int64_t ws_bytes, cudaStream_t stream) {
    LfWs w;
    const size_t need = carve_lf(w, (unsigned char*)ws, B, t.D, NPART, BN);
    if (int rc = bigd_check_workspace(ws, ws_bytes, need, kLfName, "hmc_leap_frog_workspace_bytes")) return rc;
    int dev = 0, sms = 0;
    HMC_CUDA_CHECK(cudaGetDevice(&dev));
    HMC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int Dp = w.Dp;
    CUtensorMap mapA[2], mapS[2], mapB, mapP, mapX;
    if (int rc = bigd_target_operands<NPART, BN, CL, BK>(t, w, sms, stream, &mapB)) return rc;
    for (int b = 0; b < 2; ++b) {
        uint16_t* xb = w.xp + (size_t)b * NPART * w.Ncp * Dp;
        if (int rc = make_map(&mapA[b], bigd_dt16<NPART>(), 2, xb, (uint64_t)NPART * w.Ncp, Dp, BK, BM)) return rc;      // operand loads
        if (int rc = make_map(&mapS[b], bigd_dt16<NPART>(), 2, xb, (uint64_t)NPART * w.Ncp, Dp, CW, 32)) return rc;      // epilogue stores
    }
    if (int rc = make_map(&mapP, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, w.p, (uint64_t)w.Ncp, Dp, CW, 32)) return rc;
    if (int rc = make_map(&mapX, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, w.x, (uint64_t)w.Ncp, Dp, CW, 32)) return rc;
    lf_init<NPART><<<(w.Ncp + 7) / 8, 256, 0, stream>>>(p_old, q_old, B, t.D, w);
    auto kern = bigd_gemm_step<LfWs, EPI_LEAPFROG, NPART, BN, CL, BK, STAGES>;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr;
    if (int rc = bigd_launch_config(cfg, attr, kern, CL, (w.Ncp / BM / CL) * w.NT, gemm_smem_bytes<NPART, BN, BK, STAGES>(), sms, stream,
                                    kLfName)) return rc;
    int rc = HMC_OK;
    for (int pass = 0; pass <= nsteps; ++pass) {       // pass n: operands from buffer n & 1, the epilogue writes buffer (n + 1) & 1
        w.mode = w.modes + (size_t)(pass == 0 ? 0 : (pass < nsteps ? 1 : 2)) * w.Ncp;
        if (cudaLaunchKernelEx(&cfg, kern, mapA[pass & 1], mapB, mapP, mapX, mapS[(pass + 1) & 1], w, (int)B, Dp, (const float*)w.dt) !=
            cudaSuccess) { rc = HMC_E_CUDA; break; }
    }
    if (rc != HMC_OK) return bigd_loop_result(rc, kLfName);
    const long blocks = B < (long)sms * 16 ? B : (long)sms * 16;
    lf_end<<<(int)blocks, 256, 0, stream>>>(w, B, t.D, p_new, q_new);
    HMC_CUDA_CHECK(cudaGetLastError());
    return HMC_OK;
}

}  // namespace

bool hmc_start_pts_bigd_supported(int dtype, int D, const char** why) { return bigd_covers_gemm(dtype, D, why); }

size_t hmc_start_pts_bigd_workspace(long Nchain, int D) {
    StartWs w;
    return carve_start(w, nullptr, Nchain, D);
}

int hmc_start_pts_bigd_run(uint64_t seed, int64_t chain_id0, long Nchain, int D, const double* q0, const double* Lc, const double* sd,
                           float* out, void* ws, int64_t ws_bytes, cudaStream_t stream) {
    if (!Lc) {
        int sms = 0, dev = 0;
        HMC_CUDA_CHECK(cudaGetDevice(&dev));
        HMC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        const long need = (Nchain + 7) / 8, cap = (long)sms * 16;
        start_diag<<<(int)(need < cap ? need : cap), 256, 0, stream>>>(seed, chain_id0, Nchain, D, q0, sd, out);
        HMC_CUDA_CHECK(cudaGetLastError());
        return HMC_OK;
    }
    return run_start_pts(seed, chain_id0, Nchain, D, q0, Lc, out, ws, ws_bytes, stream);
}

bool hmc_leap_frog_bigd_supported(int dtype, int D, const char** why) { return bigd_covers_gemm(dtype, D, why); }

size_t hmc_leap_frog_bigd_workspace(long B, int D) {
    LfWs w;                                       // sized for the larger of the two splits
    return carve_lf(w, nullptr, B, D, 3, 128);
}

int hmc_leap_frog_bigd_run(const hmc_target& t, long B, const float* p_old, const float* q_old, float* p_new, float* q_new, int nsteps,
                           int flags, void* ws, int64_t ws_bytes, cudaStream_t stream) {
    return bigd_run_variant(flags, [&](auto v) {
        using V = decltype(v);
        return run_leap_frog<V::NPART, V::BN, V::CL, V::BK, V::STAGES>(t, B, p_old, q_old, p_new, q_new, nsteps, ws, ws_bytes, stream);
    });
}
