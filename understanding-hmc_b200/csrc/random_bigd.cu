// Large-D random-trajectory HMC path (BASELINE config 5: dense-covariance MVN, D = 1024, 131,072 chains per GPU):
// the gradient of ALL chains, G[Nchain x D] = X[Nchain x D] * F[D x D]^T, is a real dense contraction and runs as a
// tcgen05 GEMM with TMA-fed operands; the leapfrog update is fused into its epilogue.
//
// Follows HMC_sampler.gen_sample_random + leap_frog (/root/reference/samplers.py:387-491, 831-839).
//
// Any 128 <= D <= 8192: the GEMM works on Dp = D rounded up to 32 (one K stage).  Every operand, state row and the force matrix
// are Dp wide and zero in the padded dimensions (no force, no momentum, dt = 0 there), so those stay zero and add nothing to the
// energies; K = Dp, and the last column tile is Dp - (NT - 1) BN wide when BN does not divide Dp.  For D % 256 == 0, Dp = D
// and nothing changes.  Only the caller's rows (start points, stored samples, state_q, the chain-0 trace) are exactly D wide.
//
// One PASS = one gradient evaluation for every chain (SURVEY H9: per-step GEMM with the leapfrog update fused in):
//   bigd_gemm_step   persistent CTAs (clusters of two row blocks) over (128 chains x 256 dimensions) tiles, K = D.  Warp 0 issues
//                    the TMA loads (cp.async.bulk.tensor, 64-byte swizzle, 3 stages of K = 32; the B tile multicast to the
//                    cluster), warp 1 issues the tcgen05.mma (cta_group::1, kind::f16, M = 128, N = 256, fp32 accumulators
//                    double-buffered in the 512 TMEM columns), warps 2..5 are the epilogue: tcgen05.ld of a 16-column chunk, the
//                    chunk's momentum and position rows brought in by TMA, per-chain kick / drift weights by trajectory phase
//                    (first point: half kick + drift, interior: full kick + drift, last: half kick), momentum and position
//                    updated in shared memory and stored by TMA, the NEXT pass's A operand (the split position) stored by TMA
//                    into the other operand buffer, partial sums of q.g and p.p per (chain, column tile) for the energies.
//                    FP32-grade product from a two-part fp16 split (x = h1 + h2, F 2^s = f1 + f2; products (1,2) (2,1) (1,1)
//                    per K step) -- or the three-part bf16 split with six products (flags bit 1 clear).
//   bigd_events      one thread per chain: trajectory bookkeeping (energies, Metropolis accept on the Philox uniform, step
//                    counters, samplers.py:434-462); chains whose trajectory ended go on a list.
//   bigd_trajectory_end  one warp per listed chain: accept (start point <- proposal) or reject (position and operand rows <-
//                    start point), stored sample row, momentum refresh / new length / new uniform (samplers.py:431, 441,
//                    461-472), next iteration or chain end.
// Chains advance asynchronously (SURVEY H3): every chain has its own phase, the GEMM never waits for a trajectory end.
// All three kernels of a pass are enqueued back to back; the host looks at the number of running chains every 8 passes.
//
// HBM per chain and pass: p and q read + written (16 B / dimension), split position written (4 or 6 B) and read by TMA
// (4 or 6 B; the four column tiles of a row block re-read it from L2): ~24 B x D vs 2 D^2 x 3 tensor flop.
#include "hmc_common.cuh"
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <cstdlib>
#include <cstdio>
#include <vector>
#include <algorithm>
#include <exception>

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

struct BigdWs {                      // workspace carved by the host (all device pointers)
    uint16_t* xp;                    // [2][NPART][Ncp][Dp]  split position = A operand: pass n reads buffer n & 1 and writes the other one
                                     // (the column tiles of a row block read ALL its columns while one of them already writes its own)
    int wr;                          // buffer the parts of the next pass go to (set per launch)
    int* perm;                       // [Ncp] row -> local chain index (-1: padding row).  Rows are chains SORTED by the number of passes
                                     // their run needs (the trajectory lengths are a pure function of (seed, chain, iteration)), so the
                                     // 128 chains of a row block end together and finished blocks drop out of the GEMM early
    int* plan;                       // [Ncp] passes a chain needs: sum over its iterations of L + 1
    uint16_t* bp;                    // [NPART][Dp][Dp]  split force matrix (x 2^s for the fp16 split) = B operand, zero outside D x D
    float* x;                        // [Ncp][Dp] shifted position q - mu
    float* x0;                       // [Ncp][Dp] position at the start of the running trajectory
    float* p;                        // [Ncp][Dp] momentum
    float* mu;                       // [Dp] target mean, zero from D on
    float* dt;                       // [Dp] step sizes, zero from D on (the padded dimensions never move)
    float* red;                      // [Ncp][NT][2][2] partial (q.g, p.p) per column tile and epilogue warp of the last pass
    int* mode;                       // [Ncp] MD_*
    int* l;                          // [Ncp] leapfrog steps done in the running trajectory
    int* L;                          // [Ncp] its length
    int* it;                         // [Ncp] running iteration
    int* init;                       // [Ncp] chain start: E_chain[., 0] still to be recorded
    float* K_new;                    // [Ncp] 0.5 |p|^2 of the momentum of the running iteration
    float* K0;                       // [Ncp] 0.5 |p|^2 of the chain-start momentum (samplers.py:415)
    float* lnu;                      // [Ncp] log of the acceptance uniform
    float* E_init;                   // [Ncp]
    float* E_prev;                   // [Ncp]
    int* tile_active;                // [Ncp / 128]
    int* list;                       // [Ncp] chains whose trajectory ended in this pass (bit 31: accepted)
    int* counters;                   // [0..1] list length by pass parity, [2] running chains after the last events kernel
    float binv;                      // 2^-s
    int Ncp, NT, npart;
    int Dp;                          // D rounded up to whole K stages (32): the width of every row and matrix above.  The padded
                                     // dimensions hold zeros throughout: no force, no momentum, no step
};

// CL = CTAs per cluster (launch attribute): the CL row blocks of a cluster work on the SAME column block at the same time, each
// CTA loads 1 / CL of the B tile and multicasts it to the others -- the L2 -> SM traffic of a tile drops from A + B to A + B / CL
// (the kernel was bound by exactly that traffic: 4.0 TB/s of L2 reads at 23 % tensor-pipe activity with CL = 1).
// The epilogue moves its rows by TMA as well: mapP / mapX are the momentum and position arrays [Ncp][D] float32 (box 16 columns x
// 32 rows, 64-byte swizzle; loaded and stored through the same map), mapS the 16-bit parts of the NEXT pass's A operand (box 16 x 32,
// 32-byte swizzle; mapA reads the parts of THIS pass: the two live in different buffers, alternating by pass, because the row blocks
// of a chain tile are read in full by every column tile while one of them already writes its columns).
template <int NPART, int BN, int CL, int BK, int STAGES>
__global__ void __launch_bounds__(NTHREADS, 1) bigd_gemm_step(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapB,
                                                              const __grid_constant__ CUtensorMap mapP, const __grid_constant__ CUtensorMap mapX,
                                                              const __grid_constant__ CUtensorMap mapS,
                                                              BigdWs w, int Nchain, int Dp, const float* __restrict__ dtv) {
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

// ---------------------------------------------------------------------------------------------------------------------
// momentum draw for one chain by one warp: p row (Dp wide, zero from D on), 0.5 |p|^2 of the D real dimensions, and
// (iteration >= 1) trajectory length and log-uniform (same Philox keying as every other kernel: hmc_normal4 / hmc_scalar_draws;
// when D % 4 != 0 only the first D % 4 normals of the last slot are used)
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float bigd_draw(const hmc_random_args& a, int Dp, long m, int iter, int lane, float* prow, int* L, float* lnu) {
    const int D = a.target.D;
    const uint64_t gid = (uint64_t)(a.chain_id0 + m);
    float s = 0.f;
    if (a.p_tape) {
        const double* src = a.p_tape + ((size_t)m * (a.Niter + 1) + iter) * D;
        for (int j = lane; j < D; j += 32) { const float v = (float)src[j]; if (prow) prow[j] = v; s = fmaf(v, v, s); }
        if (prow) for (int j = D + lane; j < Dp; j += 32) prow[j] = 0.f;
        if (iter >= 1) { *L = a.L_tape[(size_t)m * a.Niter + iter - 1]; *lnu = (float)log(a.u_tape[(size_t)m * a.Niter + iter - 1]); }
    } else {
        for (int sl = lane; sl < D / 4; sl += 32) {
            const float4 z = hmc_normal4(a.seed, gid, (uint32_t)iter, (uint32_t)sl);
            if (prow) *reinterpret_cast<float4*>(prow + 4 * sl) = z;
            s += z.x * z.x + z.y * z.y + z.z * z.z + z.w * z.w;
        }
        for (int sl = D / 4 + lane; sl < Dp / 4; sl += 32) {             // the partly used last slot, then the padding
            float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
            if (4 * sl < D) {
                z = hmc_normal4(a.seed, gid, (uint32_t)iter, (uint32_t)sl);
                z.w = 0.f;
                if (4 * sl + 2 >= D) z.z = 0.f;
                if (4 * sl + 1 >= D) z.y = 0.f;
            }
            if (prow) *reinterpret_cast<float4*>(prow + 4 * sl) = z;
            s += z.x * z.x + z.y * z.y + z.z * z.z + z.w * z.w;
        }
        if (iter >= 1) { double u; hmc_scalar_draws(a.seed, gid, (uint32_t)iter, a.L_low, a.L_high, L, &u); *lnu = (float)log(u); }
    }
    return 0.5f * warp_sum<float>(s);
}

template <int NPART>
__device__ __forceinline__ void bigd_write_parts(const BigdWs& w, long m, int lane, const float* xrow) {
    const int Dp = w.Dp;
    for (int j = 2 * lane; j < Dp; j += 64) {
        uint32_t h[3];
        split_pair<NPART>(xrow[j], xrow[j + 1], h);
#pragma unroll
        for (int pt = 0; pt < NPART; ++pt) reinterpret_cast<uint32_t*>(w.xp + (((size_t)w.wr * NPART + pt) * w.Ncp + m) * Dp)[j >> 1] = h[pt];
    }
}

// passes the run of a chain needs (one per leapfrog point: L + 1 per iteration; rejections add a few): the key the rows are sorted by
__global__ void __launch_bounds__(256) bigd_plan(hmc_random_args a, int* __restrict__ plan) {
    const long c = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= a.Nchain) return;
    const uint64_t gid = (uint64_t)(a.chain_id0 + c);
    int total = 0;
    for (int it = a.iter_begin + 1; it <= a.iter_end; ++it) {
        int L; double u;
        if (a.L_tape) L = a.L_tape[(size_t)c * a.Niter + it - 1];
        else hmc_scalar_draws(a.seed, gid, (uint32_t)it, a.L_low, a.L_high, &L, &u);
        total += L + 1;
    }
    plan[c] = total;
}

// chain start (samplers.py:411-420) or resume from state_q: one warp per chain
template <int NPART>
__global__ void __launch_bounds__(128) bigd_init(hmc_random_args a, BigdWs w) {
    const int lane = threadIdx.x & 31, D = a.target.D, Dp = w.Dp;
    const long m = (long)blockIdx.x * 4 + (threadIdx.x >> 5);            // row of the workspace
    if (m >= w.Ncp) return;
    float* xr = w.x + (size_t)m * Dp;
    float* x0r = w.x0 + (size_t)m * Dp;
    float* pr = w.p + (size_t)m * Dp;
    const long c = w.perm[m];                                            // the chain that lives in this row
    if (c < 0) {                                             // padding rows of the last tile
        for (int j = lane; j < Dp; j += 32) { xr[j] = 0.f; x0r[j] = 0.f; pr[j] = 0.f; }
        bigd_write_parts<NPART>(w, m, lane, xr);
        if (lane == 0) { w.mode[m] = MD_IDLE; w.it[m] = a.iter_end + 1; }
        return;
    }
    const bool fresh = a.iter_begin == 0;
    const float* src = (fresh ? (const float*)a.q_start : (const float*)a.state_q) + (size_t)c * D;
    const float* mu = w.mu;
    const long Lc = 1 + (a.Niter - a.warm_up_num) / a.thin_rate;
    const long Lrow = a.store_ring > 0 ? a.store_ring : Lc;
    for (int j = lane; j < D; j += 32) {
        const float v = src[j];
        if (fresh) ((float*)a.q_chain)[(size_t)c * Lrow * D + j] = v;              // samplers.py:413
        xr[j] = v - mu[j]; x0r[j] = v - mu[j];
    }
    for (int j = D + lane; j < Dp; j += 32) { xr[j] = 0.f; x0r[j] = 0.f; }
    __syncwarp();
    bigd_write_parts<NPART>(w, m, lane, xr);
    int L = 1; float lnu = 0.f;
    float K0 = 0.f;
    if (fresh) K0 = bigd_draw(a, Dp, c, 0, lane, nullptr, &L, &lnu);               // samplers.py:415 (K only)
    const int it = a.iter_begin + 1;
    const float Kn = bigd_draw(a, Dp, c, it, lane, pr, &L, &lnu);                  // samplers.py:431, 441, 461
    if (lane == 0) {
        w.mode[m] = (it <= a.iter_end) ? MD_FIRST : MD_IDLE;
        w.l[m] = 0; w.L[m] = L; w.it[m] = it; w.init[m] = fresh ? 1 : 0;
        w.K_new[m] = Kn; w.K0[m] = K0; w.lnu[m] = lnu;
        w.E_init[m] = 0.f; w.E_prev[m] = fresh ? 0.f : (float)a.state_eprev[c];
        if (fresh && a.decision_chain && a.chain_id0 + c == 0) a.decision_chain[a.N_save_chain0] = 0;
    }
}

// per-chain bookkeeping after a pass (one thread per chain, one block per 128-chain tile)
__global__ void __launch_bounds__(BM) bigd_events(hmc_random_args a, BigdWs w, int pass) {
    const long m = (long)blockIdx.x * BM + threadIdx.x;                              // row (the grid covers the Ncp rows exactly)
    const int Dp = w.Dp;
    const long Lc = 1 + (a.Niter - a.warm_up_num) / a.thin_rate;
    const long Lrow = a.store_ring > 0 ? a.store_ring : Lc;
    if (blockIdx.x == 0 && threadIdx.x == 0) w.counters[(pass + 1) & 1] = 0;       // list length of the NEXT pass
    int md = w.mode[m];                                                              // (padding rows are MD_IDLE from the start)
    const long c = w.perm[m];                                                        // chain of this row: indexes the outputs
    unsigned long long acc_warm = 0, acc_post = 0, sL = 0, sL2 = 0;
    if (md == MD_FIRST || md == MD_MID || md == MD_LAST) {
        float hv = 0.f, hk = 0.f;
        for (int t = 0; t < 2 * w.NT; ++t) { hv += w.red[((size_t)m * 2 * w.NT + t) * 2]; hk += w.red[((size_t)m * 2 * w.NT + t) * 2 + 1]; }
        const float V = fmaf(0.5f * w.binv, hv, (float)a.target.v_const);           // V(q) at the point the gradient was taken
        const int it = w.it[m];
        const bool tr = a.phi_q && (a.chain_id0 + c) == 0 && it <= a.N_save_chain0;
        const float* mu = w.mu;
        if (md == MD_FIRST) {
            const int L = w.L[m];
            sL = (unsigned long long)L; sL2 = (unsigned long long)L * L;
            if (w.init[m]) {                                                        // samplers.py:416-420
                const float E0 = V + w.K0[m];
                a.E_chain[(size_t)c * Lrow] = (double)E0; a.dE_chain[(size_t)c * Lrow] = 0.0;
                w.E_prev[m] = E0; w.init[m] = 0;
            }
            const float Ei = V + w.K_new[m];                                        // samplers.py:434-438
            w.E_init[m] = Ei;
            if (it >= a.warm_up_num) {
                const long idx = ((it - a.warm_up_num) / a.thin_rate) % Lrow;
                a.E_chain[(size_t)c * Lrow + idx] = (double)Ei;
                a.dE_chain[(size_t)c * Lrow + idx] = (double)(Ei - w.E_prev[m]);
            }
            if (tr) {                                                               // samplers.py:442-452
                a.phi_len[it - 1] = L + 1;
                double* phi = a.phi_q + (size_t)(it - 1) * a.L_high * 2;
                phi[0] = (double)(w.x0[(size_t)m * Dp] + mu[0]); phi[1] = (double)(w.x0[(size_t)m * Dp + 1] + mu[1]);
                phi[2] = (double)(w.x[(size_t)m * Dp] + mu[0]); phi[3] = (double)(w.x[(size_t)m * Dp + 1] + mu[1]);
            }
            w.l[m] = 1;
            md = (L == 1) ? MD_LAST : MD_MID;
        } else if (md == MD_MID) {
            const int l = w.l[m] + 1;
            if (tr) {
                double* phi = a.phi_q + (size_t)(it - 1) * a.L_high * 2;
                phi[2 * l] = (double)(w.x[(size_t)m * Dp] + mu[0]); phi[2 * l + 1] = (double)(w.x[(size_t)m * Dp + 1] + mu[1]);
            }
            w.l[m] = l;
            if (l == w.L[m]) md = MD_LAST;
        } else {                                                                    // Metropolis accept (samplers.py:455-472)
            const float Ei = w.E_init[m];
            const float dE = (V + 0.5f * hk) - Ei;
            w.E_prev[m] = Ei;                                                       // samplers.py:460
            const bool accepted = (dE < 0.f) || (w.lnu[m] < -dE);                   // samplers.py:462
            if (accepted) { if (it >= a.warm_up_num) acc_post = 1; else acc_warm = 1; }
            if (tr) a.decision_chain[it - 1] = accepted ? 1 : 0;
            const int slot = atomicAdd(&w.counters[pass & 1], 1);
            w.list[slot] = (int)m | (accepted ? (1 << 31) : 0);
            md = MD_PENDING;
        }
        w.mode[m] = md;
    }
    const int running = __syncthreads_count(md != MD_IDLE);
    if (threadIdx.x == 0) {
        w.tile_active[blockIdx.x] = running > 0;
        if (running) atomicAdd(&w.counters[2], running);
    }
    if (a.counters) {
        const unsigned long long c0 = warp_sum<unsigned long long>(acc_warm), c1 = warp_sum<unsigned long long>(acc_post);
        const unsigned long long c2 = warp_sum<unsigned long long>(sL), c3 = warp_sum<unsigned long long>(sL2);
        if ((threadIdx.x & 31) == 0 && (c0 | c1 | c2 | c3)) {
            if (c0) atomicAdd(a.counters + 0, c0);
            if (c1) atomicAdd(a.counters + 1, c1);
            atomicAdd(a.counters + 2, c2); atomicAdd(a.counters + 3, c3);
        }
    }
}

// trajectory ends: one warp per listed chain
template <int NPART>
__global__ void __launch_bounds__(256) bigd_trajectory_end(hmc_random_args a, BigdWs w, int pass) {
    const int lane = threadIdx.x & 31, D = a.target.D, Dp = w.Dp;
    const int n = w.counters[pass & 1];
    const long Lc = 1 + (a.Niter - a.warm_up_num) / a.thin_rate;
    const long Lrow = a.store_ring > 0 ? a.store_ring : Lc;
    const float* mu = w.mu;
    const bool ext4 = (D & 3) == 0;             // the external rows (stored samples, state_q) are D wide: 16-byte aligned only then
    for (int e = blockIdx.x * 8 + (threadIdx.x >> 5); e < n; e += gridDim.x * 8) {
        const int ent = w.list[e];
        const long m = ent & 0x7fffffff;                                            // row
        const long c = w.perm[m];                                                   // its chain
        const bool accepted = ent < 0;
        float* xr = w.x + (size_t)m * Dp;
        float* x0r = w.x0 + (size_t)m * Dp;
        int it = w.it[m];
        const bool keep = it >= a.warm_up_num;
        float* dst = keep ? (float*)a.q_chain + ((size_t)c * Lrow + ((it - a.warm_up_num) / a.thin_rate) % Lrow) * D : nullptr;
        const bool last = it >= a.iter_end;
        float* sq = last ? (float*)a.state_q + (size_t)c * D : nullptr;
        // accepted: start point <- proposal (samplers.py:463-469); rejected: proposal <- start point (samplers.py:470-472)
        const float* from = accepted ? xr : x0r;
        float* to = accepted ? x0r : xr;
        for (int j = 4 * lane; j < Dp; j += 128) {
            const float4 v = *reinterpret_cast<const float4*>(from + j);
            *reinterpret_cast<float4*>(to + j) = v;
            if (ext4 && j < D) {
                const float4 mu4 = *reinterpret_cast<const float4*>(mu + j);
                const float4 q = make_float4(v.x + mu4.x, v.y + mu4.y, v.z + mu4.z, v.w + mu4.w);
                if (dst) *reinterpret_cast<float4*>(dst + j) = q;
                if (sq) *reinterpret_cast<float4*>(sq + j) = q;
            }
        }
        if (!ext4) {
            for (int j = lane; j < D; j += 32) {
                const float q = from[j] + mu[j];
                if (dst) dst[j] = q;
                if (sq) sq[j] = q;
            }
        }
        if (!accepted) {
            __syncwarp();
            bigd_write_parts<NPART>(w, m, lane, x0r);
        }
        if (last) {
            if (lane == 0) { w.mode[m] = MD_IDLE; w.it[m] = it + 1; a.state_eprev[c] = (double)w.E_prev[m]; }
        } else {
            it += 1;
            int L = 1; float lnu = 0.f;
            const float Kn = bigd_draw(a, Dp, c, it, lane, w.p + (size_t)m * Dp, &L, &lnu);  // samplers.py:431, 441, 461
            if (lane == 0) { w.K_new[m] = Kn; w.L[m] = L; w.lnu[m] = lnu; w.l[m] = 0; w.it[m] = it; w.mode[m] = MD_FIRST; }
        }
    }
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

// carve the workspace; returns the bytes needed (ws may be NULL to only size it)
size_t carve(BigdWs& w, unsigned char* ws, long Nchain, int D, int npart, int bn) {
    const long Ncp = (Nchain + BM * kMaxCluster - 1) / (BM * kMaxCluster) * (BM * kMaxCluster);   // whole clusters of row blocks
    const int Dp = (D + 31) / 32 * 32;
    const int NT = (Dp + bn - 1) / bn;
    size_t off = 0;
    auto take = [&](size_t bytes) { unsigned char* p = ws ? ws + off : nullptr; off = align_up(off + bytes, 1024); return p; };
    w.Ncp = (int)Ncp; w.NT = NT; w.npart = npart; w.Dp = Dp;
    w.xp = (uint16_t*)take((size_t)2 * npart * Ncp * Dp * 2);
    w.bp = (uint16_t*)take((size_t)npart * Dp * Dp * 2);
    w.x = (float*)take((size_t)Ncp * Dp * 4);
    w.x0 = (float*)take((size_t)Ncp * Dp * 4);
    w.p = (float*)take((size_t)Ncp * Dp * 4);
    w.mu = (float*)take((size_t)Dp * 4);
    w.dt = (float*)take((size_t)Dp * 4);
    w.red = (float*)take((size_t)Ncp * NT * 2 * 2 * 4);
    w.mode = (int*)take(Ncp * 4); w.l = (int*)take(Ncp * 4); w.L = (int*)take(Ncp * 4); w.it = (int*)take(Ncp * 4); w.init = (int*)take(Ncp * 4);
    w.K_new = (float*)take(Ncp * 4); w.K0 = (float*)take(Ncp * 4); w.lnu = (float*)take(Ncp * 4); w.E_init = (float*)take(Ncp * 4);
    w.E_prev = (float*)take(Ncp * 4);
    w.tile_active = (int*)take((Ncp / BM) * 4);
    w.list = (int*)take(Ncp * 4);
    w.counters = (int*)take(64);
    w.perm = (int*)take(Ncp * 4);
    w.plan = (int*)take(Ncp * 4);
    return off;
}

template <int NPART, int BN, int BK, int STAGES>
constexpr size_t gemm_smem_bytes() {
    return (size_t)STAGES * NPART * (BM * BK * 2 + BN * BK * 2) + (size_t)NEPI * NBUF * (2 * EPB_PX + NPART * EPB_PART) + (2 * STAGES + 4 + NEPI * NBUF) * 8 + 64;
}
static_assert(gemm_smem_bytes<2, 256, 32, (NEPI == 4 ? 3 : 2)>() <= 232448 && gemm_smem_bytes<3, 128, 32, 2>() <= 232448,
              "shared memory of the large-D GEMM exceeds 227 KB");

template <int NPART, int BN, int CL, int BK, int STAGES>
int run_bigd(const hmc_random_args& a, cudaStream_t stream) {
    const int D = a.target.D;
    BigdWs w;
    const size_t need = carve(w, (unsigned char*)a.workspace, a.Nchain, D, NPART, BN);
    if (!a.workspace || (size_t)a.workspace_bytes < need) {
        hmc_set_error("large-D kernel needs a workspace of %zu bytes (hmc_random_workspace_bytes)", need);
        return HMC_E_BADARG;
    }
    int dev = 0, sms = 0;
    HMC_CUDA_CHECK(cudaGetDevice(&dev));
    HMC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    // force matrix parts (scaled to the top of the fp16 range for the fp16 split)
    const int Dp = w.Dp;
    float scale = 1.f;
    HMC_CUDA_CHECK(cudaMemsetAsync(w.counters, 0, 64, stream));
    // mean and step sizes, zero-padded to Dp (the caller's arrays are D_pad <= Dp long)
    HMC_CUDA_CHECK(cudaMemsetAsync(w.mu, 0, (size_t)Dp * 4, stream));
    HMC_CUDA_CHECK(cudaMemsetAsync(w.dt, 0, (size_t)Dp * 4, stream));
    HMC_CUDA_CHECK(cudaMemcpyAsync(w.mu, a.target.mu, (size_t)D * 4, cudaMemcpyDeviceToDevice, stream));
    HMC_CUDA_CHECK(cudaMemcpyAsync(w.dt, a.target.dt, (size_t)D * 4, cudaMemcpyDeviceToDevice, stream));
    if (NPART == 2) {
        unsigned int* mxd = (unsigned int*)(w.counters + 8);
        bigd_absmax<<<sms * 4, 256, 0, stream>>>((const float*)a.target.Ft, D, a.target.D_pad, mxd);
        unsigned int mx = 0;
        HMC_CUDA_CHECK(cudaMemcpyAsync(&mx, mxd, 4, cudaMemcpyDeviceToHost, stream));
        HMC_CUDA_CHECK(cudaStreamSynchronize(stream));
        const int e = (int)(mx >> 23) - 127;
        int sft = (mx == 0u || e < -100) ? 0 : 14 - e;
        sft = sft > 100 ? 100 : (sft < -100 ? -100 : sft);
        scale = ldexpf(1.f, sft);
    }
    w.binv = 1.f / scale;
    bigd_split_matrix<NPART><<<sms * 8, 256, 0, stream>>>((const float*)a.target.Ft, D, a.target.D_pad, Dp, scale, w.bp);
    CUtensorMap mapA[2], mapS[2], mapB, mapP, mapX;
    const CUtensorMapDataType dt16 = NPART == 2 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
    for (int b = 0; b < 2; ++b) {
        uint16_t* xb = w.xp + (size_t)b * NPART * w.Ncp * Dp;
        if (int rc = make_map(&mapA[b], dt16, 2, xb, (uint64_t)NPART * w.Ncp, Dp, BK, BM)) return rc;      // operand loads
        if (int rc = make_map(&mapS[b], dt16, 2, xb, (uint64_t)NPART * w.Ncp, Dp, CW, 32)) return rc;      // epilogue stores
    }
    if (int rc = make_map(&mapB, dt16, 2, w.bp, (uint64_t)NPART * Dp, Dp, BK, BN / CL)) return rc;         // each CTA of a cluster loads 1 / CL of a B tile
    if (int rc = make_map(&mapP, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, w.p, (uint64_t)w.Ncp, Dp, CW, 32)) return rc;
    if (int rc = make_map(&mapX, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, w.x, (uint64_t)w.Ncp, Dp, CW, 32)) return rc;
    w.wr = 0;                                                    // pass 0 reads buffer 0
    try {   // rows = chains sorted by planned passes, longest first (stable: equal plans keep the chain order); padding rows last
        bigd_plan<<<(a.Nchain + 255) / 256, 256, 0, stream>>>(a, w.plan);
        std::vector<int> plan_h(a.Nchain), perm_h(w.Ncp, -1);
        HMC_CUDA_CHECK(cudaMemcpyAsync(plan_h.data(), w.plan, sizeof(int) * a.Nchain, cudaMemcpyDeviceToHost, stream));
        HMC_CUDA_CHECK(cudaStreamSynchronize(stream));
        for (int i = 0; i < a.Nchain; ++i) perm_h[i] = i;
        if (getenv("HMC_B200_BIGD_NOSORT") == nullptr)
            std::stable_sort(perm_h.begin(), perm_h.begin() + a.Nchain, [&](int x, int y) { return plan_h[x] > plan_h[y]; });
        HMC_CUDA_CHECK(cudaMemcpyAsync(w.perm, perm_h.data(), sizeof(int) * w.Ncp, cudaMemcpyHostToDevice, stream));
        HMC_CUDA_CHECK(cudaStreamSynchronize(stream));                      // (perm_h leaves scope)
    } catch (const std::exception& e) {                    // (no exception crosses the C boundary)
        hmc_set_error("large-D kernel: host-side row plan failed: %s", e.what());
        return HMC_E_CUDA;
    }
    bigd_init<NPART><<<(w.Ncp + 3) / 4, 128, 0, stream>>>(a, w);
    const int ntile_rows = w.Ncp / BM;
    HMC_CUDA_CHECK(cudaMemsetAsync(w.tile_active, 0xff, (size_t)ntile_rows * 4, stream));
    const size_t smem = gemm_smem_bytes<NPART, BN, BK, STAGES>();
    auto kern = bigd_gemm_step<NPART, BN, CL, BK, STAGES>;
    HMC_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int ntiles = (ntile_rows / CL) * w.NT;                 // work items of a cluster
    // persistent clusters: as many as are resident at once (a GPC holds whole clusters only), never more than there is work
    cudaLaunchConfig_t cfg = {};
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = CL; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.gridDim = dim3(sms / CL * CL); cfg.blockDim = dim3(NTHREADS); cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cfg.attrs = attr; cfg.numAttrs = 1;
    int max_clusters = sms / CL;
    if (CL > 1) {
        int nc = 0;
        HMC_CUDA_CHECK(cudaOccupancyMaxActiveClusters(&nc, kern, &cfg));
        if (nc < 1) { hmc_set_error("large-D kernel: no cluster of %d CTAs fits on this device", CL); return HMC_E_CUDA; }
        if (nc < max_clusters) max_clusters = nc;
    }
    const int nclusters = ntiles < max_clusters ? ntiles : max_clusters;
    const int grid = nclusters * CL;
    cfg.gridDim = dim3(grid);
    const float* dtv = w.dt;
    const int Nch = a.Nchain;
    // pass n: operands from buffer n & 1, the epilogue (and the trajectory ends after it) write buffer (n + 1) & 1
    auto launch_gemm = [&](long pass) { w.wr = (int)((pass + 1) & 1);
                                        return cudaLaunchKernelEx(&cfg, kern, mapA[pass & 1], mapB, mapP, mapX, mapS[(pass + 1) & 1], w, Nch, Dp, dtv); };
    int* running_h = nullptr;
    HMC_CUDA_CHECK(cudaMallocHost(&running_h, 4));
    const long max_pass = (long)(a.iter_end - a.iter_begin) * (a.L_high + 1) + 8;
    int rc = HMC_OK;
    // HMC_B200_BIGD_TIMING=1: CUDA-event times of the three kernels of passes 4..11 on stderr (measurement aid)
    const bool timing = getenv("HMC_B200_BIGD_TIMING") != nullptr;
    cudaEvent_t ev[4];
    float tsum[3] = {0.f, 0.f, 0.f};
    if (timing) for (int i = 0; i < 4; ++i) cudaEventCreate(&ev[i]);
    for (long pass = 0; pass < max_pass; ++pass) {
        if (timing && pass >= 4 && pass < 12) {
            cudaEventRecord(ev[0], stream);
            launch_gemm(pass);
            cudaEventRecord(ev[1], stream);
            cudaMemsetAsync(w.counters + 2, 0, 4, stream);
            bigd_events<<<ntile_rows, BM, 0, stream>>>(a, w, (int)pass);
            cudaEventRecord(ev[2], stream);
            bigd_trajectory_end<NPART><<<sms * 2, 256, 0, stream>>>(a, w, (int)pass);
            cudaEventRecord(ev[3], stream);
            cudaEventSynchronize(ev[3]);
            for (int i = 0; i < 3; ++i) { float ms = 0.f; cudaEventElapsedTime(&ms, ev[i], ev[i + 1]); tsum[i] += ms; }
            if (pass == 11) fprintf(stderr, "[bigd timing] NPART=%d BN=%d BK=%d cluster=%d chains=%d D=%d: gemm_step %.3f ms, events %.3f ms, trajectory_end %.3f ms per pass (%d work items on %d CTAs)\n",
                                    NPART, BN, BK, CL, a.Nchain, D, tsum[0] / 8, tsum[1] / 8, tsum[2] / 8, ntiles, grid);
            continue;
        }
        if (launch_gemm(pass) != cudaSuccess) { rc = HMC_E_CUDA; break; }
        cudaMemsetAsync(w.counters + 2, 0, 4, stream);
        bigd_events<<<ntile_rows, BM, 0, stream>>>(a, w, (int)pass);
        bigd_trajectory_end<NPART><<<sms * 2, 256, 0, stream>>>(a, w, (int)pass);
        if ((pass & 7) == 7) {
            // chains that ended their last trajectory in this pass are still MD_PENDING for the events kernel's count: they are
            // counted as running and found idle at the next look
            if (cudaMemcpyAsync(running_h, w.counters + 2, 4, cudaMemcpyDeviceToHost, stream) != cudaSuccess ||
                cudaStreamSynchronize(stream) != cudaSuccess) { rc = HMC_E_CUDA; break; }
            if (*running_h == 0) break;
        }
    }
    if (timing) for (int i = 0; i < 4; ++i) cudaEventDestroy(ev[i]);
    cudaFreeHost(running_h);
    if (rc == HMC_OK) HMC_CUDA_CHECK(cudaGetLastError());
    else hmc_set_error("large-D kernel: CUDA error in the pass loop: %s", cudaGetErrorString(cudaGetLastError()));
    return rc;
}

}  // namespace

bool hmc_random_bigd_supported(const hmc_random_args& a, const char** why) {
    if (a.dtype != HMC_F32) { *why = "float32 only"; return false; }
    if (a.target.Mit || a.target.Pt || a.target.Lct) { *why = "identity momentum metric only"; return false; }
    if (a.target.D < 128 || a.target.D > 8192) { *why = "D must be in [128, 8192]"; return false; }
    if (a.iter_end <= a.iter_begin) { *why = "needs at least one iteration"; return false; }
    return true;
}

size_t hmc_random_bigd_workspace(const hmc_random_args& a) {
    BigdWs w;                                     // sized for the larger of the two variants
    return carve(w, nullptr, a.Nchain, a.target.D, 3, 128);
}

int hmc_random_run_bigd(const hmc_random_args& a, cudaStream_t stream) {
    bool fp16 = (a.flags & HMC_FLAG_TC_FP16X2) != 0;
    if (const char* e = getenv("HMC_B200_TC_PREC")) fp16 = (e[0] == 'f');
    // Clusters of two row blocks share the column block's B tile by TMA multicast (HMC_B200_BIGD_CLUSTER=1: plain CTAs).  With the
    // first epilogue the cluster changed nothing (the kernel was bound by its epilogue); with the TMA epilogue it is worth 8 % of a
    // full pass at fp16x2 and 19 % of a bf16x3 run (DESIGN 4.5).
    int cl = 2;
    if (const char* e = getenv("HMC_B200_BIGD_CLUSTER")) cl = atoi(e);
    constexpr int ST2 = NEPI == 4 ? 3 : 2;           // operand stages that fit beside the epilogue buffers
    if (fp16) return cl == 2 ? run_bigd<2, 256, 2, 32, ST2>(a, stream) : run_bigd<2, 256, 1, 32, ST2>(a, stream);
    return cl == 2 ? run_bigd<3, 128, 2, 32, 2>(a, stream) : run_bigd<3, 128, 1, 32, 2>(a, stream);
}
