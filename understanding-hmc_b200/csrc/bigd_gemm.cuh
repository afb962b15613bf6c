// The large-D tcgen05 GEMM shared by the large-D samplers (random_bigd.cu, nuts_bigd.cu) and primitives (bigd_primitives.cu:
// start points, leap_frog): G = X F^T for all chains of a pass,
// X = the split positions [Ncp][Dp] (A operand, by TMA), F = the split force matrix [Dp][Dp] (B operand, by TMA, multicast to a
// cluster of row blocks), fp32 accumulators in tensor memory.  The epilogue is a template parameter:
//   EPI_LEAPFROG  the leapfrog update of the random-trajectory sampler fused into the epilogue (random_bigd.cu explains it)
//   EPI_GRAD      the gradient rows themselves, G[Ncp][Dp] float32 by TMA store (the NUTS step runs as its own kernel)
// W is the caller's workspace: it provides tile_active (row blocks with a chain that takes part), mode (per row: MD_IDLE rows
// need no gradient), Ncp, NT and binv (2^-s of the fp16 split's matrix scaling); the leapfrog epilogue also uses red.
// Also here: the split of a pair of floats into 16-bit parts, the split of the force matrix, the tensor-map helper, and what the
// two samplers do alike around the GEMM (bottom of the file): coverage, workspace geometry and carving, the target as GEMM
// operands, the launch configuration, the choice of split and cluster, the look at the running chains, and the momentum-row and
// split-position helpers of their own kernels.
#pragma once
#include "hmc_common.cuh"
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <cstdlib>

namespace {

constexpr int BM = 128;            // chains per tile (UMMA M)
// dimensions per tile (UMMA N; fp32 accumulator columns) is a template parameter BN: 256 for the two-part split, 128 for the
// three-part one (shared memory)
// K per stage is a template parameter BK in {64, 32, 16} (one swizzle row of 128 / 64 / 32 bytes) with 128 / BK stages: the bytes
// of operand memory are the same, the pipeline is finer -- a stage can only be refilled after its MMAs are done, so with two
// 96 KB stages one load is in flight while the other stage is consumed and the tensor pipe waits for most of a load's latency.
constexpr int kStageK = 128;       // stages x BK
constexpr int kMaxCluster = 4;     // largest cluster of row blocks (the chain count is padded to whole clusters)
constexpr int CW = 16;             // epilogue chunk: 16 columns of a warp's 32 chains
#ifndef BIGD_NEPI
#define BIGD_NEPI 4
#endif
constexpr int NEPI = BIGD_NEPI;    // epilogue warps: one (4) or two (8, alternating chunks) per TMEM lane quarter
constexpr int NBUF = NEPI == 4 ? 3 : 2;   // chunk buffers per epilogue warp (one in arithmetic, one being stored, one loading)
constexpr int NHALF = NEPI / 4;
constexpr int NTHREADS = 64 + 32 * NEPI;      // warp 0 TMA, warp 1 MMA, warps 2..5 epilogue
constexpr int EPB_PX = 32 * CW * 4;           // one float32 array of a chunk: 32 rows x 64 bytes, SWIZZLE_64B
constexpr int EPB_PART = 32 * CW * 2;         // one 16-bit part of a chunk: 32 rows x 32 bytes, SWIZZLE_32B
enum : int { MD_IDLE = 0, MD_FIRST = 1, MD_MID = 2, MD_LAST = 3, MD_PENDING = 4 };

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* b, int count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(b)), "r"(count)); }
// (a wait that lasts longer than ~4 s of SM clocks means a lost TMA / MMA completion: abort the kernel instead of hanging the GPU)
__device__ __forceinline__ void mbar_wait(uint64_t* b, uint32_t parity) {
    uint32_t done = 0;
    const long long t0 = clock64();
    while (!done) {
        asm volatile("{\n\t.reg .pred pw;\n\tmbarrier.try_wait.parity.shared::cta.b64 pw, [%1], %2;\n\tselp.u32 %0, 1, 0, pw;\n\t}"
                     : "=r"(done) : "r"(smem_u32(b)), "r"(parity) : "memory");
        if (!done && clock64() - t0 > 8000000000ll) __trap();
    }
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* b, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* b) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(b)) : "memory"); }
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
// the same load delivered to the same shared-memory offset (data and mbarrier signal) of every CTA of the cluster named in `mask`
__device__ __forceinline__ void tma_load_2d_mc(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar, uint16_t mask) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
                 ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask) : "memory");
}
// MMA completion signalled on the mbarrier at this offset in every CTA of `mask` (a stage is shared by the cluster's producers)
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// K-major operand tile [rows][BK x 16 bit] written by TMA with the swizzle of its row length (128 / 64 / 32 bytes): 8-row groups
// 8 x row bytes apart; layout type 2 = SWIZZLE_128B, 4 = SWIZZLE_64B, 6 = SWIZZLE_32B
template <int BK>
__device__ __forceinline__ uint64_t make_desc_sw(uint32_t saddr) {
    constexpr uint32_t row_bytes = BK * 2;
    constexpr uint64_t layout = (BK == 64) ? 2 : (BK == 32 ? 4 : 6);
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3fff);
    d |= (uint64_t)1 << 16;                              // leading byte offset: unused for swizzled K-major (set to 1)
    d |= (uint64_t)(((8u * row_bytes) >> 4) & 0x3fff) << 32;   // stride byte offset: 8 rows
    d |= (uint64_t)1 << 46;                              // descriptor version (Blackwell)
    d |= layout << 61;
    return d;
}
__device__ __forceinline__ void umma_ss(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t addr, uint32_t* v) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                   "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(addr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// split of a pair of float32 values into 16-bit parts (true signs), NPART = 2: fp16, NPART = 3: bf16
template <int NPART>
__device__ __forceinline__ void split_pair(float x0, float x1, uint32_t (&h)[3]) {
    if constexpr (NPART == 2) {
        const __half2 a = __floats2half2_rn(x0, x1);
        const float2 af = __half22float2(a);
        const __half2 b = __floats2half2_rn(x0 - af.x, x1 - af.y);
        h[0] = *reinterpret_cast<const uint32_t*>(&a); h[1] = *reinterpret_cast<const uint32_t*>(&b); h[2] = 0u;
    } else {
        const __nv_bfloat162 a = __floats2bfloat162_rn(x0, x1);
        float r0 = x0 - __low2float(a), r1 = x1 - __high2float(a);
        const __nv_bfloat162 b = __floats2bfloat162_rn(r0, r1);
        r0 -= __low2float(b); r1 -= __high2float(b);
        const __nv_bfloat162 c = __floats2bfloat162_rn(r0, r1);
        h[0] = *reinterpret_cast<const uint32_t*>(&a); h[1] = *reinterpret_cast<const uint32_t*>(&b); h[2] = *reinterpret_cast<const uint32_t*>(&c);
    }
}

enum : int { EPI_LEAPFROG = 0, EPI_GRAD = 1 };

// CL = CTAs per cluster (launch attribute): the CL row blocks of a cluster work on the SAME column block at the same time, each
// CTA loads 1 / CL of the B tile and multicasts it to the others -- the L2 -> SM traffic of a tile drops from A + B to A + B / CL
// (the kernel was bound by exactly that traffic: 4.0 TB/s of L2 reads at 23 % tensor-pipe activity with CL = 1).
// The epilogue moves its rows by TMA as well: mapP / mapX are the momentum and position arrays [Ncp][D] float32 (box 16 columns x
// 32 rows, 64-byte swizzle; loaded and stored through the same map), mapS the 16-bit parts of the NEXT pass's A operand (box 16 x 32,
// 32-byte swizzle; mapA reads the parts of THIS pass: the two live in different buffers, alternating by pass, because the row blocks
// of a chain tile are read in full by every column tile while one of them already writes its columns).
template <class W, int EPI, int NPART, int BN, int CL, int BK, int STAGES>
__global__ void __launch_bounds__(NTHREADS, 1) bigd_gemm_step(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                                                              const __grid_constant__ CUtensorMap mapP, const __grid_constant__ CUtensorMap mapX,
                                                              const __grid_constant__ CUtensorMap mapS,
                                                              W w, int Nchain, int Dp, const float* __restrict__ dtv) {
    extern __shared__ __align__(1024) unsigned char smem[];
    constexpr int A_BYTES = BM * BK * 2, B_BYTES = BN * BK * 2;                 // one part of one stage
    constexpr int STAGE_BYTES = NPART * (A_BYTES + B_BYTES);
    unsigned char* stage_base = smem;
    unsigned char* epi = smem + STAGES * STAGE_BYTES;                           // epilogue chunk buffers, per warp
    constexpr int EPI_BUF_BYTES = 2 * EPB_PX + NPART * EPB_PART;               // momentum | position | parts of one chunk
    constexpr int EPI_WARP_BYTES = NBUF * EPI_BUF_BYTES;
    uint64_t* bars = reinterpret_cast<uint64_t*>(epi + NEPI * EPI_WARP_BYTES);
    uint64_t* full = bars;                 // [STAGES]
    uint64_t* empty = bars + STAGES;       // [STAGES]
    uint64_t* tfull = bars + 2 * STAGES;   // [2]
    uint64_t* tempty = bars + 2 * STAGES + 2;   // [2]
    uint64_t* efull = bars + 2 * STAGES + 4;    // [NEPI][NBUF] chunk loaded
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4 + NEPI * NBUF);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) { mbar_init(full + s, 1); mbar_init(empty + s, CL); }   // a stage is refilled by all CL producers
        for (int s = 0; s < 2; ++s) { mbar_init(tfull + s, 1); mbar_init(tempty + s, NEPI); }
        for (int s = 0; s < NEPI * NBUF; ++s) mbar_init(efull + s, 1);
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(tmem_slot)));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if constexpr (CL > 1) cluster_sync_all();              // barriers of every CTA initialised before anybody signals them
    asm volatile("tcgen05.fence::after_thread_sync;");
    const uint32_t tmem = *tmem_slot;
    const int NT = w.NT, KB = Dp / BK;
    // the last column tile is narrow when BN does not divide Dp: its MMAs run at N = n_last (a multiple of 32) and its epilogue
    // takes n_last / CW chunks.  Its B loads keep the full box: the rows past n_last are loaded (the next part's first rows, or
    // the TMA's zero fill past the last part) but no MMA reads them, so the stage's transaction bytes stay STAGE_BYTES
    const int n_last = Dp - (NT - 1) * BN;
    const int ntiles = (w.Ncp / (BM * CL)) * NT;            // work items of a cluster: (CL row blocks, one column block)
    const size_t part_rows_a = (size_t)w.Ncp, part_rows_b = (size_t)Dp;
    const int crank = (CL > 1) ? (int)cluster_ctarank() : 0;
    const int cid = blockIdx.x / CL, ncl = gridDim.x / CL;
    constexpr uint16_t cmask = (uint16_t)((1u << CL) - 1u);
    // the same decision in every CTA of the cluster (their loops must stay in step): skip a work item only if all its row blocks are idle
    auto item_active = [&](int mtc) { int any = 0;
#pragma unroll
        for (int r = 0; r < CL; ++r) any |= w.tile_active[mtc * CL + r];
        return any != 0; };

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            uint32_t n = 0;
            for (int t = cid; t < ntiles; t += ncl) {
                const int mtc = t / NT, nt = t % NT;
                if (!item_active(mtc)) continue;
                const int mt = mtc * CL + crank;
                for (int kb = 0; kb < KB; ++kb, ++n) {
                    const int s = n % STAGES;
                    mbar_wait(empty + s, ((n / STAGES) & 1) ^ 1);           // released by the MMA warps of all CL CTAs
                    unsigned char* sb = stage_base + s * STAGE_BYTES;
                    mbar_expect_tx(full + s, STAGE_BYTES);                   // my A parts + the whole B tile (1 / CL of it from each CTA)
#pragma unroll
                    for (int pt = 0; pt < NPART; ++pt) {
                        tma_load_2d(sb + pt * A_BYTES, &mapA, kb * BK, (int)(pt * part_rows_a) + mt * BM, full + s);
                        if constexpr (CL == 1)
                            tma_load_2d(sb + NPART * A_BYTES + pt * B_BYTES, &mapB, kb * BK, (int)(pt * part_rows_b) + nt * BN, full + s);
                        else
                            tma_load_2d_mc(sb + NPART * A_BYTES + pt * B_BYTES + crank * (B_BYTES / CL), &mapB, kb * BK,
                                           (int)(pt * part_rows_b) + nt * BN + crank * (BN / CL), full + s, cmask);
                    }
                }
            }
            if constexpr (CL > 1) {                                          // every release aimed at this CTA has arrived before it may exit
                for (uint32_t k = 0; k < STAGES && k < n; ++k) {
                    const uint32_t m = n - 1 - k;
                    mbar_wait(empty + (m % STAGES), (m / STAGES) & 1);
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (lane == 0) {
            constexpr uint32_t fmt = (NPART == 2) ? 0u : 1u;       // 0 = f16, 1 = bf16
            const uint32_t idesc0 = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(BM >> 4) << 24);
            const uint32_t idesc_full = idesc0 | ((uint32_t)(BN >> 3) << 17), idesc_last = idesc0 | ((uint32_t)(n_last >> 3) << 17);
            uint32_t n = 0, nt_done = 0;
            for (int t = cid; t < ntiles; t += ncl) {
                if (!item_active(t / NT)) continue;
                const uint32_t idesc = (t % NT == NT - 1) ? idesc_last : idesc_full;
                const int as = nt_done & 1;
                mbar_wait(tempty + as, ((nt_done >> 1) & 1) ^ 1);
                asm volatile("tcgen05.fence::after_thread_sync;");
                const uint32_t tacc = tmem + (uint32_t)(as * BN);
                for (int kb = 0; kb < KB; ++kb, ++n) {
                    const int s = n % STAGES;
                    mbar_wait(full + s, (n / STAGES) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;");
                    const uint32_t sa = smem_u32(stage_base + s * STAGE_BYTES), sbb = sa + NPART * A_BYTES;
                    // part products of this K block, small terms first: fp16x2 (1,2) (2,1) (1,1); bf16x3 (1,3) (3,1) (2,2) (1,2) (2,1) (1,1)
                    constexpr int NPROD = (NPART == 2) ? 3 : 6;
                    constexpr int pa2[3] = {0, 1, 0}, pb2[3] = {1, 0, 0};
                    constexpr int pa3[6] = {0, 2, 1, 0, 1, 0}, pb3[6] = {2, 0, 1, 1, 0, 0};
#pragma unroll
                    for (int pr = 0; pr < NPROD; ++pr) {
                        const int pa = (NPART == 2) ? pa2[pr % 3] : pa3[pr], pb = (NPART == 2) ? pb2[pr % 3] : pb3[pr];
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) {
                            const uint64_t ad = make_desc_sw<BK>(sa + pa * A_BYTES + k * 32);
                            const uint64_t bd = make_desc_sw<BK>(sbb + pb * B_BYTES + k * 32);
                            umma_ss(tacc, ad, bd, idesc, (kb | pr | k) ? 1u : 0u);
                        }
                    }
                    if constexpr (CL == 1) umma_commit(empty + s);           // frees the stage when these MMAs are done
                    else umma_commit_mc(empty + s, cmask);                    // ... in every CTA of the cluster (all of them refill it)
                }
                umma_commit(tfull + as);                      // accumulator complete
                ++nt_done;
            }
        }
    } else if constexpr (EPI == EPI_GRAD) {
        // ===== gradient epilogue: the fp32 gradient rows G[chain][Dp] (the accumulator x 2^-s) go to global memory by TMA
        //       (mapP is the map of G; 64-byte swizzle, a chunk = 16 columns of the warp's 32 chains).  Chunk g uses buffer
        //       g % NBUF, which the store of chunk g - NBUF has left when the storing lane's read wait below returns. ==========
        const int quarter = warp & 3, ew = warp - 2, half = ew >> 2;
        unsigned char* ebase = epi + ew * EPI_WARP_BYTES;
        const int swz = (lane >> 1) & 3;
        uint32_t nt_done = 0, g = 0;
        for (int t = cid; t < ntiles; t += ncl) {
            const int mtc = t / NT, nt = t % NT;
            if (!item_active(mtc)) continue;
            const int as = nt_done & 1;
            const long row0 = (long)(mtc * CL + crank) * BM + quarter * 32;
            const long chain = row0 + lane;
            const int md = (chain < Nchain) ? w.mode[chain] : (int)MD_IDLE;
            const bool live = __any_sync(HMC_FULL_MASK, md != MD_IDLE) != 0;
            mbar_wait(tfull + as, (nt_done >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;");
            if (live) {
                const int NCH = (nt == NT - 1 ? n_last : BN) / CW;
                for (int c = half; c < NCH; c += NHALF, ++g) {
                    unsigned char* bp = ebase + (g % NBUF) * EPI_BUF_BYTES;
                    uint32_t gv[16];
                    tmem_ld16(tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(as * BN + c * CW), gv);
                    float4* grow = reinterpret_cast<float4*>(bp + lane * 64);
#pragma unroll
                    for (int i = 0; i < CW / 4; ++i)
                        grow[i ^ swz] = make_float4(__uint_as_float(gv[4 * i]) * w.binv, __uint_as_float(gv[4 * i + 1]) * w.binv,
                                                    __uint_as_float(gv[4 * i + 2]) * w.binv, __uint_as_float(gv[4 * i + 3]) * w.binv);
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) {
                        tma_store_2d(&mapP, bp, nt * BN + c * CW, (int)row0);
                        bulk_commit();
                        bulk_wait_read<NBUF - 1>();
                    }
                    __syncwarp();
                }
            }
            asm volatile("tcgen05.fence::before_thread_sync;");
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty + as);
            ++nt_done;
        }
        if (lane == 0) bulk_wait_all();
    } else {
        // ===== epilogue warps: TMEM lanes 32 (warp % 4) .. + 31 = 32 chains of the tile, one thread per chain (the layout
        //       tcgen05.ld delivers).  The momentum and position rows of a 16-column chunk arrive by TMA (64-byte swizzle: a thread's
        //       16-byte pieces of its row fall on distinct banks), are updated in place, go back by TMA together with the split
        //       position; NBUF chunk buffers per warp, the load of chunk g + 2 is issued when the store of chunk g - 1 has left its
        //       buffer.  (The first version moved every element through registers -> padded tile -> registers twice: ~150 LSU
        //       instructions per 256 elements, and ran at 26 % tensor-pipe activity whatever the operand pipeline did.) ==========
        const int quarter = warp & 3, ew = warp - 2, half = ew >> 2;    // (two warps of a quarter take alternating chunks)
        unsigned char* ebase = epi + ew * EPI_WARP_BYTES;
        uint64_t* ef = efull + ew * NBUF;
        auto nch = [&](int tt) { return ((tt % NT) == NT - 1 ? n_last : BN) / CW; };    // chunks of a tile
        // a tile is LIVE for this warp when one of its 32 chains takes part in the pass; only live tiles enter the chunk stream
        auto tile_md = [&](int tt) { const long ch = (long)((tt / NT) * CL + crank) * BM + quarter * 32 + lane;
                                     return (ch < Nchain) ? w.mode[ch] : (int)MD_IDLE; };
        auto is_live = [&](int md) { return __any_sync(HMC_FULL_MASK, md == MD_FIRST || md == MD_MID || md == MD_LAST) != 0; };
        auto next_live = [&](int tt) { for (tt += ncl; tt < ntiles; tt += ncl) if (item_active(tt / NT) && is_live(tile_md(tt))) break; return tt; };
        // chunk c of tile tt is the g-th chunk of this warp's stream; lanes 0 and 1 issue the two loads in ONE warp instruction (a
        // lane-serial sequence of TMA instructions was 30 % of the epilogue warps' stall samples)
        auto issue_chunk = [&](int tt, int c, uint32_t g) {
            const int buf = g % NBUF;
            unsigned char* bp = ebase + buf * EPI_BUF_BYTES;
            const int col0 = (tt % NT) * BN + c * CW, row0 = ((tt / NT) * CL + crank) * BM + quarter * 32;
            if (lane == 0) mbar_expect_tx(ef + buf, 2 * EPB_PX);
            __syncwarp();
            if (lane < 2) tma_load_2d(bp + lane * EPB_PX, lane == 0 ? &mapP : &mapX, col0, row0, ef + buf);
        };
        // prefetch cursor: (pf_t, pf_c) = the next chunk to request, pf_g its number in the stream
        int pf_t = cid - ncl;
        pf_t = next_live(pf_t);
        int pf_c = half;
        uint32_t pf_g = 0, g = 0;
        auto prefetch_one = [&]() {
            if (pf_t >= ntiles) return;
            issue_chunk(pf_t, pf_c, pf_g);
            ++pf_g;
            if ((pf_c += NHALF) >= nch(pf_t)) { pf_c = half; pf_t = next_live(pf_t); }
        };
        prefetch_one();
        prefetch_one();
        uint32_t nt_done = 0;
        const int swz = (lane >> 1) & 3;                        // 64-byte swizzle of my row: 16-byte piece c sits at piece c ^ swz
        const int swz2 = (lane >> 2) & 1;                       // 32-byte swizzle of my row
        for (int t = cid; t < ntiles; t += ncl) {
            const int mtc = t / NT, nt = t % NT;
            if (!item_active(mtc)) continue;
            const int mt = mtc * CL + crank;
            const int as = nt_done & 1;
            const long row0 = (long)mt * BM + quarter * 32;          // first chain of this warp
            const long chain = row0 + lane;
            const int md = tile_md(t);
            const float kw = (md == MD_MID) ? -w.binv : ((md == MD_FIRST || md == MD_LAST) ? -0.5f * w.binv : 0.f);
            const float dw = (md == MD_FIRST || md == MD_MID) ? 1.f : 0.f;
            const bool live = is_live(md);
            mbar_wait(tfull + as, (nt_done >> 1) & 1);
            asm volatile("tcgen05.fence::after_thread_sync;");
            float hv = 0.f, hk = 0.f;
            if (live) {
                const int NCH = nch(t);
                for (int c = half; c < NCH; c += NHALF, ++g) {
                    const int buf = g % NBUF;
                    unsigned char* bp = ebase + buf * EPI_BUF_BYTES;
                    const int c0 = nt * BN + c * CW;
                    float dts[CW];
#pragma unroll
                    for (int i = 0; i < CW / 4; ++i) {
                        const float4 d4 = __ldg(reinterpret_cast<const float4*>(dtv + c0) + i);
                        dts[4 * i] = d4.x; dts[4 * i + 1] = d4.y; dts[4 * i + 2] = d4.z; dts[4 * i + 3] = d4.w;
                    }
                    uint32_t gv[16];
                    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
                                 : "=r"(gv[0]), "=r"(gv[1]), "=r"(gv[2]), "=r"(gv[3]), "=r"(gv[4]), "=r"(gv[5]), "=r"(gv[6]), "=r"(gv[7]),
                                   "=r"(gv[8]), "=r"(gv[9]), "=r"(gv[10]), "=r"(gv[11]), "=r"(gv[12]), "=r"(gv[13]), "=r"(gv[14]), "=r"(gv[15])
                                 : "r"(tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(as * BN + c * CW)));
                    mbar_wait(ef + buf, (g / NBUF) & 1);                 // momentum and position rows of the chunk have landed
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    float4* prow = reinterpret_cast<float4*>(bp + lane * 64);
                    float4* xrow = reinterpret_cast<float4*>(bp + EPB_PX + lane * 64);
                    uint4* hrow = reinterpret_cast<uint4*>(bp + 2 * EPB_PX + lane * 32);
#pragma unroll
                    for (int i = 0; i < CW / 4; ++i) {
                        float4 p4 = prow[i ^ swz], x4 = xrow[i ^ swz];
                        float pv[4] = {p4.x, p4.y, p4.z, p4.w}, xv[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float gj = __uint_as_float(gv[4 * i + e]);
                            const float dtj = dts[4 * i + e];
                            hv = fmaf(xv[e], gj, hv);
                            const float pn = fmaf(gj, kw * dtj, pv[e]);                       // samplers.py:835, 837
                            hk = fmaf(pn, pn, hk);
                            xv[e] = fmaf(pn, dw * dtj, xv[e]);                                // samplers.py:836
                            pv[e] = pn;
                        }
                        prow[i ^ swz] = make_float4(pv[0], pv[1], pv[2], pv[3]);
                        xrow[i ^ swz] = make_float4(xv[0], xv[1], xv[2], xv[3]);
                        uint32_t h0[3], h1[3];
                        split_pair<NPART>(xv[0], xv[1], h0);
                        split_pair<NPART>(xv[2], xv[3], h1);
                        // the 8 bytes of columns 4 i .. 4 i + 3 of part pt: half of 16-byte piece i / 2 of the part's 32-byte row
#pragma unroll
                        for (int pt = 0; pt < NPART; ++pt) {
                            uint2* piece = reinterpret_cast<uint2*>(reinterpret_cast<unsigned char*>(hrow) + pt * EPB_PART + (((i >> 1) ^ swz2) << 4));
                            piece[i & 1] = make_uint2(h0[pt], h1[pt]);
                        }
                    }
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // my generic-proxy writes -> visible to the TMA store
                    __syncwarp();
                    if (lane < 2 + NPART) {                              // lanes 0, 1: momentum, position; lanes 2..: the parts -- one instruction
                        const CUtensorMap* mp = lane == 0 ? &mapP : (lane == 1 ? &mapX : &mapS);
                        const unsigned char* src = bp + (lane < 2 ? lane * EPB_PX : 2 * EPB_PX + (lane - 2) * EPB_PART);
                        const int r = (int)row0 + (lane < 2 ? 0 : (lane - 2) * (int)part_rows_a);
                        tma_store_2d(mp, src, c0, r);
                        bulk_commit();                                   // (bulk groups are per thread: each storing lane tracks its own)
                        bulk_wait_read<NBUF - 2>();                      // the stores of chunk g + 2 - NBUF have left their buffer: chunk g + 2 goes there
                    }
                    __syncwarp();
                    prefetch_one();
                }
            }
            if (chain < Nchain) {
                float* rd = w.red + ((size_t)chain * NT + nt) * 4 + half * 2;
                rd[0] = hv; rd[1] = hk;
                if (NHALF == 1) { rd[2] = 0.f; rd[3] = 0.f; }
            }
            asm volatile("tcgen05.fence::before_thread_sync;");
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty + as);
            ++nt_done;
        }
        if (lane < 2 + NPART) bulk_wait_all();                           // every store complete before the buffers go away
    }
    asm volatile("tcgen05.fence::before_thread_sync;");
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem));
    if constexpr (CL > 1) cluster_sync_all();              // nobody leaves while a peer may still write into its shared memory
}

// force matrix -> split 16-bit parts, K-major rows: bp[part][n][k] = part(F[n][k] * scale) for n, k < D, zero up to Dp;
// Ft[k][n] = F[n][k] (row stride Dpad)
template <int NPART>
__global__ void bigd_split_matrix(const float* __restrict__ Ft, int D, int Dpad, int Dp, float scale, uint16_t* __restrict__ bp) {
    const long total = (long)Dp * (Dp / 2);
    for (long t = blockIdx.x * (long)blockDim.x + threadIdx.x; t < total; t += (long)gridDim.x * blockDim.x) {
        const int n = (int)(t / (Dp / 2)), k = 2 * (int)(t % (Dp / 2));
        const float f0 = (n < D && k < D) ? Ft[(size_t)k * Dpad + n] * scale : 0.f;
        const float f1 = (n < D && k + 1 < D) ? Ft[(size_t)(k + 1) * Dpad + n] * scale : 0.f;
        uint32_t h[3];
        split_pair<NPART>(f0, f1, h);
#pragma unroll
        for (int pt = 0; pt < NPART; ++pt) reinterpret_cast<uint32_t*>(bp + ((size_t)pt * Dp + n) * Dp)[k >> 1] = h[pt];
    }
}

__global__ void bigd_absmax(const float* __restrict__ Ft, int D, int Dpad, unsigned int* out) {
    unsigned int mx = 0u;
    for (long t = blockIdx.x * (long)blockDim.x + threadIdx.x; t < (long)D * D; t += (long)gridDim.x * blockDim.x)
        mx = max(mx, __float_as_uint(fabsf(Ft[(size_t)(t / D) * Dpad + (t % D)])));
    mx = __reduce_max_sync(HMC_FULL_MASK, mx);
    if ((threadIdx.x & 31) == 0) atomicMax(out, mx);
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess && qres == cudaDriverEntryPointSuccess)
            fn = (EncodeTiledFn)p;
    }
    return fn;
}

// 2-D map over a row-major [rows][D] matrix: box = box_cols x box_rows elements, swizzle = the box's row length in bytes
// (128 / 64 / 32)
int make_map(CUtensorMap* map, CUtensorMapDataType dt, int elem_bytes, void* base, uint64_t rows, uint64_t D, uint32_t box_cols, uint32_t box_rows) {
    EncodeTiledFn enc = get_encode();
    if (!enc) { hmc_set_error("cuTensorMapEncodeTiled is not available from the driver"); return HMC_E_CUDA; }
    const cuuint64_t dims[2] = {D, rows};
    const cuuint64_t strides[1] = {D * (uint64_t)elem_bytes};
    const cuuint32_t box[2] = {box_cols, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    const uint32_t row_bytes = box_cols * (uint32_t)elem_bytes;
    const CUtensorMapSwizzle swz = row_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : (row_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
    const CUresult r = enc(map, dt, 2, base, dims, strides, box, estr,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { hmc_set_error("cuTensorMapEncodeTiled failed (%d)", (int)r); return HMC_E_CUDA; }
    return HMC_OK;
}

size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

template <int NPART, int BN, int BK, int STAGES>
constexpr size_t gemm_smem_bytes() {
    return (size_t)STAGES * NPART * (BM * BK * 2 + BN * BK * 2) + (size_t)NEPI * NBUF * (2 * EPB_PX + NPART * EPB_PART) + (2 * STAGES + 4 + NEPI * NBUF) * 8 + 64;
}
static_assert(gemm_smem_bytes<2, 256, 32, (NEPI == 4 ? 3 : 2)>() <= 232448 && gemm_smem_bytes<3, 128, 32, 2>() <= 232448,
              "shared memory of the large-D GEMM exceeds 227 KB");

// =====================================================================================================================
// What the two samplers do alike around the GEMM.  Each keeps its own workspace struct (the fields the GEMM reads are named
// alike), kernels and pass loop; `name` is the path's name in error messages.
// =====================================================================================================================

// the runs the large-D path covers (the `why` strings end up in error messages).  A dense momentum metric (target.Pt, Mit and
// Lct, all three) only where the caller has it (`dense`: the Random sampler) and only for D > 1024: up to D = 1024 the generic
// kernel runs it, and that stays so
bool bigd_covers(int dtype, const hmc_target& t, int iter_begin, int iter_end, const char** why, bool dense = false) {
    if (dtype != HMC_F32) { *why = "float32 only"; return false; }
    const bool metric = t.Mit || t.Pt || t.Lct;
    if (metric && !dense) { *why = "identity momentum metric only"; return false; }
    if (metric && t.D <= 1024) {
        *why = "identity momentum metric only for D <= 1024 (the generic kernel runs a dense metric there)";
        return false;
    }
    if (metric && !(t.Mit && t.Pt && t.Lct)) { *why = "a dense momentum metric needs target.Pt, Mit and Lct together"; return false; }
    if (t.D < 128 || t.D > 8192) { *why = "D must be in [128, 8192]"; return false; }
    if (iter_end <= iter_begin) { *why = "needs at least one iteration"; return false; }
    return true;
}

// the dtype and sizes the GEMM itself covers, whatever the metric: the large-D primitives (bigd_primitives.cu) take any metric,
// their caller having folded it into the one matrix they multiply by
bool bigd_covers_gemm(int dtype, int D, const char** why) {
    if (dtype != HMC_F32) { *why = "float32 only"; return false; }
    if (D < 128 || D > 8192) { *why = "D must be in [128, 8192]"; return false; }
    return true;
}

// Workspace geometry and carving: Ncp rows (the chains padded to whole clusters of row blocks), Dp = D rounded up to whole K
// stages (32) columns in NT column tiles of width bn; take() hands out the arrays one after the other, 1024-byte aligned (with a
// NULL base it only sizes them)
struct BigdCarve {
    unsigned char* base;
    long Ncp;
    int Dp, NT;
    size_t off = 0;
    BigdCarve(unsigned char* ws, long Nchain, int D, int bn)
        : base(ws), Ncp((Nchain + BM * kMaxCluster - 1) / (BM * kMaxCluster) * (BM * kMaxCluster)), Dp((D + 31) / 32 * 32),
          NT((Dp + bn - 1) / bn) {}
    void* take(size_t bytes) { unsigned char* p = base ? base + off : nullptr; off = align_up(off + bytes, 1024); return p; }
};

int bigd_check_workspace(const void* ws, int64_t bytes, size_t need, const char* name, const char* sizer) {
    if (ws && (size_t)bytes >= need) return HMC_OK;
    hmc_set_error("%s needs a workspace of %zu bytes (%s)", name, need, sizer);
    return HMC_E_BADARG;
}

template <int NPART>
constexpr CUtensorMapDataType bigd_dt16() { return NPART == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16; }

// The target as the GEMM's inputs: clears w.counters (word 8 is the abs-max scratch), mu and dt zero-padded to Dp (the caller's
// arrays are D_pad <= Dp long), the force matrix split into w.bp -- for the fp16 split scaled by 2^s to the top of the fp16 range,
// which needs the matrix's abs-max on the host (the one wait for the device here) -- w.binv = 2^-s, and the map of the B operand
// (each CTA of a cluster loads 1 / CL of a B tile)
template <int NPART, int BN, int CL, int BK, class W>
int bigd_target_operands(const hmc_target& t, W& w, int sms, cudaStream_t stream, CUtensorMap* mapB) {
    const int D = t.D, Dp = w.Dp;
    HMC_CUDA_CHECK(cudaMemsetAsync(w.counters, 0, 64, stream));
    HMC_CUDA_CHECK(cudaMemsetAsync(w.mu, 0, (size_t)Dp * 4, stream));
    HMC_CUDA_CHECK(cudaMemsetAsync(w.dt, 0, (size_t)Dp * 4, stream));
    HMC_CUDA_CHECK(cudaMemcpyAsync(w.mu, t.mu, (size_t)D * 4, cudaMemcpyDeviceToDevice, stream));
    HMC_CUDA_CHECK(cudaMemcpyAsync(w.dt, t.dt, (size_t)D * 4, cudaMemcpyDeviceToDevice, stream));
    float scale = 1.f;
    if (NPART == 2) {
        unsigned int* mxd = (unsigned int*)(w.counters + 8);
        bigd_absmax<<<sms * 4, 256, 0, stream>>>((const float*)t.Ft, D, t.D_pad, mxd);
        unsigned int mx = 0;
        HMC_CUDA_CHECK(cudaMemcpyAsync(&mx, mxd, 4, cudaMemcpyDeviceToHost, stream));
        HMC_CUDA_CHECK(cudaStreamSynchronize(stream));
        const int e = (int)(mx >> 23) - 127;
        int sft = (mx == 0u || e < -100) ? 0 : 14 - e;
        sft = sft > 100 ? 100 : (sft < -100 ? -100 : sft);
        scale = ldexpf(1.f, sft);
    }
    w.binv = 1.f / scale;
    bigd_split_matrix<NPART><<<sms * 8, 256, 0, stream>>>((const float*)t.Ft, D, t.D_pad, Dp, scale, w.bp);
    return make_map(mapB, bigd_dt16<NPART>(), 2, w.bp, (uint64_t)NPART * Dp, Dp, BK, BN / CL);
}

// Launch configuration of the GEMM kernel: persistent clusters of CL CTAs, as many as are resident at once (a GPC holds whole
// clusters only), never more than the nwork work items.  cfg points to attr for the cluster attribute.
template <class K>
int bigd_launch_config(cudaLaunchConfig_t& cfg, cudaLaunchAttribute& attr, K kern, int CL, int nwork, size_t smem, int sms,
                       cudaStream_t stream, const char* name) {
    HMC_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr.id = cudaLaunchAttributeClusterDimension;
    attr.val.clusterDim.x = CL; attr.val.clusterDim.y = 1; attr.val.clusterDim.z = 1;
    cfg = {};
    cfg.gridDim = dim3(sms / CL * CL); cfg.blockDim = dim3(NTHREADS); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cfg.attrs = &attr; cfg.numAttrs = 1;
    int max_clusters = sms / CL;
    if (CL > 1) {
        int nc = 0;
        HMC_CUDA_CHECK(cudaOccupancyMaxActiveClusters(&nc, kern, &cfg));
        if (nc < 1) { hmc_set_error("%s: no cluster of %d CTAs fits on this device", name, CL); return HMC_E_CUDA; }
        if (nc < max_clusters) max_clusters = nc;
    }
    cfg.gridDim = dim3((nwork < max_clusters ? nwork : max_clusters) * CL);
    return HMC_OK;
}

template <int NPART_, int BN_, int CL_, int BK_, int STAGES_>
struct BigdVariant { static constexpr int NPART = NPART_, BN = BN_, CL = CL_, BK = BK_, STAGES = STAGES_; };

// The GEMM variant of a run, handed to the path's runner as run(BigdVariant<...>{}): the two-part fp16 split on 256-column tiles
// when the caller sets HMC_FLAG_TC_FP16X2, else the three-part bf16 split on 128-column tiles (shared memory); HMC_B200_TC_PREC
// overrides the flag ('f...': fp16x2, else bf16x3).  Clusters of two row blocks share the column block's B tile by TMA multicast
// (HMC_B200_BIGD_CLUSTER=1: plain CTAs).  With the first epilogue the cluster changed nothing (the kernel was bound by its
// epilogue); with the TMA epilogue it is worth 8 % of a full pass at fp16x2 and 19 % of a bf16x3 run (DESIGN 4.5).
template <class Run>
int bigd_run_variant(int flags, Run run) {
    bool fp16 = (flags & HMC_FLAG_TC_FP16X2) != 0;
    if (const char* e = getenv("HMC_B200_TC_PREC")) fp16 = (e[0] == 'f');
    int cl = 2;
    if (const char* e = getenv("HMC_B200_BIGD_CLUSTER")) cl = atoi(e);
    constexpr int ST2 = NEPI == 4 ? 3 : 2;           // operand stages that fit beside the epilogue buffers
    if (fp16) return cl == 2 ? run(BigdVariant<2, 256, 2, 32, ST2>{}) : run(BigdVariant<2, 256, 1, 32, ST2>{});
    return cl == 2 ? run(BigdVariant<3, 128, 2, 32, 2>{}) : run(BigdVariant<3, 128, 1, 32, 2>{});
}

// The host's look at the running chains: counters[2] (running chains after the last pass) read through a pinned word
struct BigdRunning {
    int* h = nullptr;
    int alloc() { HMC_CUDA_CHECK(cudaMallocHost(&h, 4)); return HMC_OK; }
    ~BigdRunning() { if (h) cudaFreeHost(h); }
    int read(const int* counters, cudaStream_t stream) {          // -1 on a CUDA error
        if (cudaMemcpyAsync(h, counters + 2, 4, cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
            cudaStreamSynchronize(stream) != cudaSuccess) return -1;
        return *h;
    }
};

// the result of a pass loop: rc as the loop left it (HMC_E_CUDA: a launch or a look failed), else a launch error since
int bigd_loop_result(int rc, const char* name) {
    if (rc == HMC_OK) HMC_CUDA_CHECK(cudaGetLastError());
    else hmc_set_error("%s: CUDA error in the pass loop: %s", name, cudaGetErrorString(cudaGetLastError()));
    return rc;
}

// Momentum row of one chain and iteration, by one warp: normal j is component j & 3 of hmc_normal4(seed, gid, iter, j >> 2) -- or
// element j of the injected tape row when one is given -- for j < D, zero from D on; stored to the Dp-wide row prow when one is
// given.  Returns this lane's sum of the squares.  Lane l takes the tape elements l, l + 32, ..., and the Philox slots l, l + 32,
// ... below `wrap`, then from `wrap` on (the partly used last slot when D % 4 != 0, then the padding) wrap + l, wrap + l + 32, ...
// That order decides the last bit of the float sums: Random passes wrap = D / 4, NUTS 0, as their results have always had it.
__device__ __forceinline__ float bigd_momentum(const double* tape, uint64_t seed, uint64_t gid, int iter, int D, int Dp, int lane,
                                               float* prow, int wrap) {
    float s = 0.f;
    if (tape) {
        for (int j = lane; j < Dp; j += 32) { const float v = j < D ? (float)tape[j] : 0.f; if (prow) prow[j] = v; s = fmaf(v, v, s); }
    } else {
        for (int sl = lane; sl < wrap; sl += 32) {
            const float4 z = hmc_normal4(seed, gid, (uint32_t)iter, (uint32_t)sl);
            if (prow) *reinterpret_cast<float4*>(prow + 4 * sl) = z;
            s += z.x * z.x + z.y * z.y + z.z * z.z + z.w * z.w;
        }
        for (int sl = wrap + lane; sl < Dp / 4; sl += 32) {
            float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
            if (4 * sl < D) {
                z = hmc_normal4(seed, gid, (uint32_t)iter, (uint32_t)sl);
                if (4 * sl + 3 >= D) z.w = 0.f;
                if (4 * sl + 2 >= D) z.z = 0.f;
                if (4 * sl + 1 >= D) z.y = 0.f;
            }
            if (prow) *reinterpret_cast<float4*>(prow + 4 * sl) = z;
            s += z.x * z.x + z.y * z.y + z.z * z.z + z.w * z.w;
        }
    }
    __syncwarp();                              // (the row is read with other lane-to-element maps afterwards)
    return s;
}

// the split position of row m (Dp wide) as the NPART 16-bit parts of the A operand: xp[part][Ncp][Dp] from the buffer base xp
template <int NPART>
__device__ __forceinline__ void bigd_write_parts(uint16_t* xp, int Ncp, int Dp, long m, int lane, const float* xr) {
    __syncwarp();                              // xr was written with another lane-to-element map
    for (int j = 2 * lane; j < Dp; j += 64) {
        uint32_t h[3];
        split_pair<NPART>(xr[j], xr[j + 1], h);
#pragma unroll
        for (int pt = 0; pt < NPART; ++pt) reinterpret_cast<uint32_t*>(xp + ((size_t)pt * Ncp + m) * Dp)[j >> 1] = h[pt];
    }
}

}  // namespace
