// C-ABI entry points of libhmc_b200.so (see include/hmc_b200.h): argument checks, kernel selection, error string.
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include "hmc_common.cuh"

static thread_local char g_err[512] = "";

void hmc_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int hmc_random_run_generic(const hmc_random_args& a, cudaStream_t stream);
int hmc_random_run_fast(const hmc_random_args& a, cudaStream_t stream);
bool hmc_random_fast_supported(const hmc_random_args& a, const char** why);
int hmc_random_run_tc(const hmc_random_args& a, cudaStream_t stream);
bool hmc_random_tc_supported(const hmc_random_args& a, const char** why);
int hmc_random_run_bigd(const hmc_random_args& a, cudaStream_t stream);
bool hmc_random_bigd_supported(const hmc_random_args& a, const char** why);
size_t hmc_random_bigd_workspace(const hmc_random_args& a);
int hmc_nuts_run_generic(const hmc_nuts_args& a, cudaStream_t stream);
int hmc_nuts_run_tc(const hmc_nuts_args& a, cudaStream_t stream);
bool hmc_nuts_tc_supported(const hmc_nuts_args& a, const char** why);
int hmc_nuts_run_bigd(const hmc_nuts_args& a, cudaStream_t stream);
bool hmc_nuts_bigd_supported(const hmc_nuts_args& a, const char** why);
size_t hmc_nuts_bigd_workspace(const hmc_nuts_args& a);
bool hmc_start_pts_bigd_supported(int dtype, int D, const char** why);
size_t hmc_start_pts_bigd_workspace(long Nchain, int D);
int hmc_start_pts_bigd_run(uint64_t seed, int64_t chain_id0, long Nchain, int D, const double* q0, const double* Lc, const double* sd,
                           float* out, void* ws, int64_t ws_bytes, cudaStream_t stream);
bool hmc_leap_frog_bigd_supported(int dtype, int D, const char** why);
size_t hmc_leap_frog_bigd_workspace(long B, int D);
int hmc_leap_frog_bigd_run(const hmc_target& t, long B, const float* p_old, const float* q_old, float* p_new, float* q_new, int nsteps,
                           int flags, void* ws, int64_t ws_bytes, cudaStream_t stream);

extern "C" int hmc_version(void) { return HMC_B200_VERSION; }
extern "C" const char* hmc_last_error_string(void) { return g_err; }

#define HMC_REQUIRE(cond, ...)            \
    do {                                  \
        if (!(cond)) {                    \
            hmc_set_error(__VA_ARGS__);   \
            return HMC_E_BADARG;          \
        }                                 \
    } while (0)

static int check_target(const hmc_target& t) {
    HMC_REQUIRE(t.D >= 1, "D must be >= 1 (got %d)", t.D);
    HMC_REQUIRE(t.D_pad >= t.D && (t.D_pad % 4) == 0, "D_pad must be a multiple of 4 and >= D");
    HMC_REQUIRE(t.Ft && t.mu && t.dt, "target.Ft/mu/dt must be device pointers");
    return HMC_OK;
}

extern "C" int hmc_random_run(const hmc_random_args* args, void* cuda_stream) {
    HMC_REQUIRE(args != nullptr, "args is NULL");
    const hmc_random_args& a = *args;
    HMC_REQUIRE(a.dtype == HMC_F32 || a.dtype == HMC_F64, "dtype must be HMC_F32 or HMC_F64");
    if (int rc = check_target(a.target)) return rc;
    HMC_REQUIRE(a.Nchain >= 1, "Nchain must be >= 1");
    HMC_REQUIRE(a.Niter >= 0 && a.iter_begin >= 0 && a.iter_begin <= a.iter_end && a.iter_end <= a.Niter,
                "need 0 <= iter_begin <= iter_end <= Niter");
    HMC_REQUIRE(a.thin_rate >= 1 && a.warm_up_num >= 0, "thin_rate >= 1 and warm_up_num >= 0 required");
    HMC_REQUIRE(a.L_low >= 1 && a.L_high > a.L_low, "need 1 <= L_low < L_high (np.random.randint bounds, samplers.py:441)");
    HMC_REQUIRE(a.q_chain && a.E_chain && a.dE_chain && a.state_q && a.state_eprev, "output/state buffers must be set");
    HMC_REQUIRE(a.iter_begin > 0 || a.q_start, "q_start required when iter_begin == 0");
    HMC_REQUIRE((a.p_tape == nullptr) == (a.L_tape == nullptr) && (a.L_tape == nullptr) == (a.u_tape == nullptr),
                "p_tape, L_tape and u_tape must be given together");
    HMC_REQUIRE(a.N_save_chain0 == 0 || (a.phi_q && a.phi_len && a.decision_chain) || a.chain_id0 != 0,
                "trace buffers required when N_save_chain0 > 0 on the device owning chain 0");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    int kernel = a.kernel;
    const char* why = "";
    // tensor-core kernel where it applies and pays (its 100-wide tile does the work of D = 100 whatever D is: ~6.4e9
    // gradient-evals/s; the FFMA kernel's rate grows as 1/D^2 and overtakes it below D ~ 50), then the large-D GEMM path, then
    // the FFMA kernel, then the generic one.  The large-D path covers every 128 <= D <= 8192; AUTO takes it for D % 256 == 0
    // (unpadded tiles) and for D > 1024 (beyond the generic kernel), and leaves 128 < D <= 1024 otherwise to the generic kernel
    // (HMC_KERNEL_BIGD reaches the padded path there).  A dense momentum metric is covered for D > 1024 only, so AUTO keeps it on
    // the generic kernel up to D = 1024
    if (kernel == HMC_KERNEL_AUTO)
        kernel = (a.target.D >= 52 && hmc_random_tc_supported(a, &why)) ? HMC_KERNEL_TC
                 : (a.workspace && hmc_random_bigd_supported(a, &why) && (a.target.D % 256 == 0 || a.target.D > 1024)) ? HMC_KERNEL_BIGD
                 : hmc_random_fast_supported(a, &why) ? HMC_KERNEL_FAST : HMC_KERNEL_GENERIC;
    if (kernel == HMC_KERNEL_BIGD) {
        if (!hmc_random_bigd_supported(a, &why)) {
            hmc_set_error("large-D kernel does not cover this configuration: %s", why);
            return HMC_E_UNSUPPORTED;
        }
        return hmc_random_run_bigd(a, stream);
    }
    if (kernel == HMC_KERNEL_FAST) {
        if (!hmc_random_fast_supported(a, &why)) {
            hmc_set_error("fast kernel does not cover this configuration: %s", why);
            return HMC_E_UNSUPPORTED;
        }
        return hmc_random_run_fast(a, stream);
    }
    if (kernel == HMC_KERNEL_TC) {
        if (!hmc_random_tc_supported(a, &why)) {
            hmc_set_error("tensor-core kernel does not cover this configuration: %s", why);
            return HMC_E_UNSUPPORTED;
        }
        return hmc_random_run_tc(a, stream);
    }
    if (kernel == HMC_KERNEL_GENERIC) return hmc_random_run_generic(a, stream);
    hmc_set_error("unknown kernel id %d", a.kernel);
    return HMC_E_BADARG;
}

extern "C" int64_t hmc_random_workspace_bytes(const hmc_random_args* args) {
    const char* why = "";
    if (!args) return 0;
    hmc_random_args a = *args;                      // (the iteration range of the launch does not matter for the size)
    a.iter_begin = 0; a.iter_end = 1;
    if (!hmc_random_bigd_supported(a, &why)) return 0;
    return (int64_t)hmc_random_bigd_workspace(a);
}

extern "C" int hmc_nuts_run(const hmc_nuts_args* args, void* cuda_stream) {
    HMC_REQUIRE(args != nullptr, "args is NULL");
    const hmc_nuts_args& a = *args;
    HMC_REQUIRE(a.dtype == HMC_F32 || a.dtype == HMC_F64, "dtype must be HMC_F32 or HMC_F64");
    if (int rc = check_target(a.target)) return rc;
    HMC_REQUIRE(a.Nchain >= 1, "Nchain must be >= 1");
    HMC_REQUIRE(a.d_max >= 1 && a.d_max <= 24, "d_max must be in [1, 24]");
    HMC_REQUIRE(a.Niter >= 0 && a.iter_begin >= 0 && a.iter_begin <= a.iter_end && a.iter_end <= a.Niter,
                "need 0 <= iter_begin <= iter_end <= Niter");
    HMC_REQUIRE(a.thin_rate >= 1 && a.warm_up_num >= 0, "thin_rate >= 1 and warm_up_num >= 0 required");
    HMC_REQUIRE(a.q_chain && a.E_chain && a.dE_chain && a.state_q && a.state_eprev && a.scratch && a.counters,
                "output/state/scratch buffers must be set");
    HMC_REQUIRE(a.iter_begin > 0 || a.q_start, "q_start required when iter_begin == 0");
    HMC_REQUIRE((a.p_tape == nullptr) == (a.dir_tape == nullptr) && (a.dir_tape == nullptr) == (a.u_tape == nullptr),
                "p_tape, dir_tape and u_tape must be given together");
    HMC_REQUIRE((a.target.Mit == nullptr) == (a.target.Pt == nullptr) && (a.target.Pt == nullptr) == (a.target.Lct == nullptr),
                "dense momentum metric: target.Pt, Mit and Lct must be given together");
    HMC_REQUIRE(a.store_ring >= 0, "store_ring must be >= 0 (got %d)", a.store_ring);
    const char* why = "";
    int kernel = a.kernel;
    // a ring of stored samples is written by the large-D path only: AUTO takes it wherever it covers the run, from D = 128
    if (a.store_ring > 0 && (kernel == HMC_KERNEL_AUTO || kernel == HMC_KERNEL_GENERIC || kernel == HMC_KERNEL_TC)) {
        if (kernel == HMC_KERNEL_AUTO && a.workspace && hmc_nuts_bigd_supported(a, &why)) {
            kernel = HMC_KERNEL_BIGD;
        } else {
            hmc_set_error("NUTS with store_ring > 0 runs on the large-D path only (float32, identity momentum metric, 128 <= D <= 8192, "
                          "hmc_nuts_args.workspace given): %s",
                          kernel != HMC_KERNEL_AUTO ? "the generic and tensor-core kernels keep the full stream"
                          : !a.workspace ? "no workspace given" : why);
            return HMC_E_UNSUPPORTED;
        }
    }
    // tensor-core kernel where it applies, else the large-D GEMM path above the generic kernel's D <= 256, else the generic kernel
    if (kernel == HMC_KERNEL_AUTO)
        kernel = hmc_nuts_tc_supported(a, &why) ? HMC_KERNEL_TC
                 : (a.target.D > 256 && a.workspace && hmc_nuts_bigd_supported(a, &why)) ? HMC_KERNEL_BIGD : HMC_KERNEL_GENERIC;
    if (kernel == HMC_KERNEL_BIGD) {
        if (!hmc_nuts_bigd_supported(a, &why)) {
            hmc_set_error("large-D NUTS kernel does not cover this configuration: %s", why);
            return HMC_E_UNSUPPORTED;
        }
        return hmc_nuts_run_bigd(a, (cudaStream_t)cuda_stream);
    }
    if (kernel == HMC_KERNEL_GENERIC && a.target.D > 256) {
        // (the generic kernel stops at D = 256; above it only the large-D path runs NUTS)
        if (!hmc_nuts_bigd_supported(a, &why)) {
            hmc_set_error("NUTS above D = 256 runs on the large-D path only, which does not cover this configuration: %s (got D = %d)",
                          why, a.target.D);
            return HMC_E_UNSUPPORTED;
        }
        hmc_set_error("NUTS above D = 256 runs on the large-D path only: it needs hmc_nuts_args.workspace (hmc_nuts_workspace_bytes)");
        return HMC_E_UNSUPPORTED;
    }
    if (kernel == HMC_KERNEL_TC) {
        if (!hmc_nuts_tc_supported(a, &why)) {
            hmc_set_error("tensor-core NUTS kernel does not cover this configuration: %s", why);
            return HMC_E_UNSUPPORTED;
        }
        return hmc_nuts_run_tc(a, (cudaStream_t)cuda_stream);
    }
    if (kernel != HMC_KERNEL_GENERIC) {
        hmc_set_error("NUTS: kernel must be auto, generic, tc or bigd");
        return HMC_E_BADARG;
    }
    return hmc_nuts_run_generic(a, (cudaStream_t)cuda_stream);
}

extern "C" int64_t hmc_nuts_workspace_bytes(const hmc_nuts_args* args) {
    const char* why = "";
    if (!args) return 0;
    hmc_nuts_args a = *args;                        // (the iteration range of the launch does not matter for the size)
    a.iter_begin = 0; a.iter_end = 1;
    if (!hmc_nuts_bigd_supported(a, &why)) return 0;
    return (int64_t)hmc_nuts_bigd_workspace(a);
}

// ---------------------------------------------------------------------------------------------------------
// Large-D primitives (csrc/bigd_primitives.cu): start points and leap_frog on the tcgen05 GEMM, 128 <= D <= 8192, float32
// ---------------------------------------------------------------------------------------------------------
static constexpr int64_t kBigdMaxRows = (int64_t)1 << 30;       // chains / rows of one call (the GEMM indexes rows with int)

extern "C" int64_t hmc_start_pts_workspace_bytes(int64_t Nchain, int32_t D) {
    const char* why = "";
    if (Nchain < 1 || Nchain > kBigdMaxRows || !hmc_start_pts_bigd_supported(HMC_F32, D, &why)) return 0;
    return (int64_t)hmc_start_pts_bigd_workspace((long)Nchain, D);
}

extern "C" int hmc_start_pts_bigd(int32_t dtype, uint64_t seed, int64_t chain_id0, int64_t Nchain, int32_t D, const double* q0,
                                  const double* Lc, const double* sd, void* out, void* workspace, int64_t workspace_bytes,
                                  void* cuda_stream) {
    HMC_REQUIRE(Nchain >= 1 && Nchain <= kBigdMaxRows && q0 && out && (Lc || sd),
                "hmc_start_pts_bigd: need 1 <= Nchain <= 2^30, q0, out and Lc or sd");
    const char* why = "";
    if (!hmc_start_pts_bigd_supported(dtype, D, &why)) {
        hmc_set_error("hmc_start_pts_bigd does not cover this configuration: %s", why);
        return HMC_E_UNSUPPORTED;
    }
    return hmc_start_pts_bigd_run(seed, chain_id0, (long)Nchain, D, q0, Lc, sd, (float*)out, workspace, workspace_bytes,
                                  (cudaStream_t)cuda_stream);
}

extern "C" int64_t hmc_leap_frog_workspace_bytes(const hmc_target* target, int64_t B, int32_t flags) {
    (void)flags;                                    // (sized for the larger of the two splits)
    const char* why = "";
    if (!target || B < 1 || B > kBigdMaxRows || !hmc_leap_frog_bigd_supported(HMC_F32, target->D, &why)) return 0;
    return (int64_t)hmc_leap_frog_bigd_workspace((long)B, target->D);
}

extern "C" int hmc_leap_frog_bigd(int32_t dtype, const hmc_target* target, int64_t B, const void* p_old, const void* q_old, void* p_new,
                                  void* q_new, int32_t nsteps, int32_t flags, void* workspace, int64_t workspace_bytes, void* cuda_stream) {
    HMC_REQUIRE(target && p_old && q_old && p_new && q_new, "hmc_leap_frog_bigd: NULL buffer");
    if (int rc = check_target(*target)) return rc;
    HMC_REQUIRE(B >= 1 && B <= kBigdMaxRows && nsteps >= 1, "hmc_leap_frog_bigd: need 1 <= B <= 2^30 and nsteps >= 1");
    const char* why = "";
    if (!hmc_leap_frog_bigd_supported(dtype, target->D, &why)) {
        hmc_set_error("hmc_leap_frog_bigd does not cover this configuration: %s", why);
        return HMC_E_UNSUPPORTED;
    }
    return hmc_leap_frog_bigd_run(*target, (long)B, (const float*)p_old, (const float*)q_old, (float*)p_new, (float*)q_new, nsteps, flags,
                                  workspace, workspace_bytes, (cudaStream_t)cuda_stream);
}

// ---------------------------------------------------------------------------------------------------------
// hmc_philox_draws: dump the device's own draws (test aid)
// ---------------------------------------------------------------------------------------------------------
__global__ void philox_draws_kernel(uint64_t seed, int64_t chain_id0, int Nchain, int Niter, int D, int L_low, int L_high,
                                    double* out_p, int32_t* out_L, double* out_u) {
    const int nslot = (D + 3) / 4;
    const long total = (long)Nchain * (Niter + 1) * nslot;
    for (long t = blockIdx.x * (long)blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const int slot = (int)(t % nslot);
        const long r = t / nslot;
        const int it = (int)(r % (Niter + 1));
        const long m = r / (Niter + 1);
        float4 z = hmc_normal4(seed, (uint64_t)(chain_id0 + m), (uint32_t)it, (uint32_t)slot);
        double* dst = out_p + ((size_t)m * (Niter + 1) + it) * D + 4 * slot;
        const float zz[4] = {z.x, z.y, z.z, z.w};
        for (int c = 0; c < 4; ++c) if (4 * slot + c < D) dst[c] = (double)zz[c];
        if (slot == 0 && it >= 1) {
            int L; double u;
            hmc_scalar_draws(seed, (uint64_t)(chain_id0 + m), (uint32_t)it, L_low, L_high, &L, &u);
            out_L[(size_t)m * Niter + it - 1] = L;
            out_u[(size_t)m * Niter + it - 1] = u;
        }
    }
}

extern "C" int hmc_philox_draws(uint64_t seed, int64_t chain_id0, int32_t Nchain, int32_t Niter, int32_t D,
                                int32_t L_low, int32_t L_high, double* out_p, int32_t* out_L, double* out_u,
                                void* cuda_stream) {
    HMC_REQUIRE(Nchain >= 1 && Niter >= 0 && D >= 1 && out_p && out_L && out_u, "bad arguments");
    philox_draws_kernel<<<256, 256, 0, (cudaStream_t)cuda_stream>>>(seed, chain_id0, Nchain, Niter, D, L_low, L_high,
                                                                    out_p, out_L, out_u);
    HMC_CUDA_CHECK(cudaGetLastError());
    return HMC_OK;
}

// ---------------------------------------------------------------------------------------------------------
// hmc_ffma_peak: FP32 FMA roofline probe
// ---------------------------------------------------------------------------------------------------------
template <bool kPacked>
__global__ void __launch_bounds__(512) ffma_peak_kernel(float* out, int iters) {
    // 32 independent FMA chains per thread, multiplier and addend as compile-time constants: the immediate-operand
    // FFMA form issues every cycle, which is what the 2*128*SMs*clock nominal peak assumes (a three-register FFMA
    // stream measured 63 % of it on B200 because of register-bank reads; FFMA2 needs register pairs anyway).
    float acc[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = threadIdx.x * 1e-3f + i;
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            if (kPacked) {
                float2 v = make_float2(acc[i], acc[(i + 1) & 31]);
                unsigned long long B = *reinterpret_cast<unsigned long long*>(&v);
                const float2 ca = make_float2(0.999f, 0.998f), cb = make_float2(0.001f, 0.002f);
                asm volatile("fma.rn.f32x2 %0, %1, %0, %2;" : "+l"(B) : "l"(*reinterpret_cast<const unsigned long long*>(&ca)),
                             "l"(*reinterpret_cast<const unsigned long long*>(&cb)));
                acc[i] = reinterpret_cast<float2*>(&B)->x;
            } else {
                acc[i] = fmaf(0.999f, acc[i], 0.001f);
            }
        }
    }
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < 32; ++i) s += acc[i];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
}

extern "C" int hmc_ffma_peak(double* out_flops_host, int32_t use_ffma2, void* cuda_stream) {
    HMC_REQUIRE(out_flops_host != nullptr, "out pointer is NULL");
    cudaStream_t stream = (cudaStream_t)cuda_stream;
    int dev = 0, sms = 0;
    HMC_CUDA_CHECK(cudaGetDevice(&dev));
    HMC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int blocks = sms * 4, threads = 512, iters = 20000;
    float* buf = nullptr;
    HMC_CUDA_CHECK(cudaMalloc(&buf, sizeof(float) * blocks * threads));
    cudaEvent_t e0, e1;
    HMC_CUDA_CHECK(cudaEventCreate(&e0));
    HMC_CUDA_CHECK(cudaEventCreate(&e1));
    double best = 0.0;
    for (int rep = 0; rep < 4; ++rep) {
        HMC_CUDA_CHECK(cudaEventRecord(e0, stream));
        if (use_ffma2) ffma_peak_kernel<true><<<blocks, threads, 0, stream>>>(buf, iters);
        else ffma_peak_kernel<false><<<blocks, threads, 0, stream>>>(buf, iters);
        HMC_CUDA_CHECK(cudaEventRecord(e1, stream));
        HMC_CUDA_CHECK(cudaEventSynchronize(e1));
        float ms = 0.f;
        HMC_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
        const double flops = 2.0 * 32.0 * (use_ffma2 ? 2.0 : 1.0) * iters * (double)blocks * threads / (ms * 1e-3);
        if (rep > 0 && flops > best) best = flops;
    }
    HMC_CUDA_CHECK(cudaGetLastError());
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(buf);
    *out_flops_host = best;
    return HMC_OK;
}
