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
//   bigd_gemm_step   (bigd_gemm.cuh, shared with the NUTS path nuts_bigd.cu; here with the EPI_LEAPFROG epilogue)
//                    persistent CTAs (clusters of two row blocks) over (128 chains x 256 dimensions) tiles, K = D.  Warp 0 issues
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
// The set-up around the GEMM and the momentum-row / split-position helpers are shared with nuts_bigd.cu (bigd_gemm.cuh).
//
// HBM per chain and pass: p and q read + written (16 B / dimension), split position written (4 or 6 B) and read by TMA
// (4 or 6 B; the four column tiles of a row block re-read it from L2): ~24 B x D vs 2 D^2 x 3 tensor flop.
#include "bigd_gemm.cuh"
#include <cstdlib>
#include <cstdio>
#include <vector>
#include <algorithm>
#include <exception>

namespace {

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


// momentum draw for one chain by one warp: p row (bigd_momentum; prow may be NULL), 0.5 |p|^2 of the D real dimensions, and
// (iteration >= 1) trajectory length and log-uniform (same Philox keying as every other kernel: hmc_scalar_draws)
__device__ __forceinline__ float bigd_draw(const hmc_random_args& a, int Dp, long m, int iter, int lane, float* prow, int* L, float* lnu) {
    const int D = a.target.D;
    const uint64_t gid = (uint64_t)(a.chain_id0 + m);
    const double* tape = a.p_tape ? a.p_tape + ((size_t)m * (a.Niter + 1) + iter) * D : nullptr;
    const float s = bigd_momentum(tape, a.seed, gid, iter, D, Dp, lane, prow, D / 4);
    if (iter >= 1) {
        if (a.p_tape) { *L = a.L_tape[(size_t)m * a.Niter + iter - 1]; *lnu = (float)log(a.u_tape[(size_t)m * a.Niter + iter - 1]); }
        else { double u; hmc_scalar_draws(a.seed, gid, (uint32_t)iter, a.L_low, a.L_high, L, &u); *lnu = (float)log(u); }
    }
    return 0.5f * warp_sum<float>(s);
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
    uint16_t* const xw = w.xp + (size_t)w.wr * NPART * w.Ncp * Dp;      // the operand buffer the next pass reads
    const long c = w.perm[m];                                            // the chain that lives in this row
    if (c < 0) {                                             // padding rows of the last tile
        for (int j = lane; j < Dp; j += 32) { xr[j] = 0.f; x0r[j] = 0.f; pr[j] = 0.f; }
        bigd_write_parts<NPART>(xw, w.Ncp, Dp, m, lane, xr);
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
    bigd_write_parts<NPART>(xw, w.Ncp, Dp, m, lane, xr);
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

// per-chain bookkeeping after a pass (one thread per chain, one block per 128-chain tile).  DENSE (a dense momentum metric): V at
// a trajectory start is the carried V0 (V(x) != x.(F x) / 2 there), and a chain that ends its trajectory only goes on the list --
// its energies need the metric products, and bigd_finish decides
template <bool DENSE>
__global__ void __launch_bounds__(BM) bigd_events(hmc_random_args a, BigdWs w, int pass, const float* __restrict__ V0) {
    const long m = (long)blockIdx.x * BM + threadIdx.x;                              // row (the grid covers the Ncp rows exactly)
    const int Dp = w.Dp;
    const long Lc = 1 + (a.Niter - a.warm_up_num) / a.thin_rate;
    const long Lrow = a.store_ring > 0 ? a.store_ring : Lc;
    if (blockIdx.x == 0 && threadIdx.x == 0) w.counters[(pass + 1) & 1] = 0;       // list length of the NEXT pass
    int md = w.mode[m];                                                              // (padding rows are MD_IDLE from the start)
    const long c = w.perm[m];                                                        // chain of this row: indexes the outputs
    unsigned long long acc_warm = 0, acc_post = 0, sL = 0, sL2 = 0;
    if (md == MD_FIRST || md == MD_MID || md == MD_LAST) {
        float hv = 0.f, hk = 0.f, V;
        if constexpr (DENSE) {
            V = md == MD_FIRST ? V0[m] : 0.f;
        } else {
            for (int t = 0; t < 2 * w.NT; ++t) { hv += w.red[((size_t)m * 2 * w.NT + t) * 2]; hk += w.red[((size_t)m * 2 * w.NT + t) * 2 + 1]; }
            V = fmaf(0.5f * w.binv, hv, (float)a.target.v_const);                   // V(q) at the point the gradient was taken
        }
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
        } else if constexpr (DENSE) {
            w.list[atomicAdd(&w.counters[pass & 1], 1)] = (int)m;
            md = MD_PENDING;
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
        if (!accepted) bigd_write_parts<NPART>(w.xp + (size_t)w.wr * NPART * w.Ncp * Dp, w.Ncp, Dp, m, lane, x0r);   // next pass's buffer
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

// ---------------------------------------------------------------------------------------------------------------------------
// Dense momentum metric (target.Pt, Mit, Lct; 1024 < D <= 8192).  The passes do not change: the main GEMM multiplies by the force
// matrix F = M^-1 P, which is all a leapfrog step needs (q moves by p: quirk Q9).  What a dense metric adds is at the ends of a
// trajectory: V(x) = x.(P x) / 2 + v_const, K(p) = p.(M^-1 p) / 2 and the momentum draw p = Lc z.  They are three batched products on
// the tensor cores (the EPI_GRAD GEMM, bf16x3 split whatever the pass split is: x, p and z are not bounded the way the fp16 split
// needs), over the chains that ended a trajectory in the pass, gathered into compact rows:
//   bigd_gather    one warp per listed chain: x = (x + mu) - mu (the x a resume from the stored float row sees, so that iteration
//                  blocks equal one launch), its split row (segment 0, times P), the split p_L (segment 1, times M^-1), the split
//                  next momentum (segment 2: z times Lc on Philox draws, the tape row times M^-1 on tapes); the row blocks below
//                  the list length for the products
//   3 x bigd_gemm_step<MetricWs, EPI_GRAD>  over the full capacity, idle row blocks skipped
//   bigd_finish    one warp per listed chain: V(x_L), K(p_L), the Metropolis test, then bigd_trajectory_end's work; the next momentum
//                  p0 = Lc z (or the tape row) with K(p0) = z.z / 2 on Philox draws (Lc Lc^T = cov_p = M, so p0.(M^-1 p0) = z.z
//                  exactly) and p0.(M^-1 p0) / 2 on tapes.  V(x0) is carried: V(x_L) after an accept, the old V0 after a reject.
// The chain start (or resume) runs the same three kernels once over every chain (`start`): V(x0), on tapes K of the iteration-0 row
// and of the first momentum, and p0 = Lc z of the first iteration (bigd_init has drawn z, L and the uniform).
// ---------------------------------------------------------------------------------------------------------------------------
struct MetricWs {                    // the products' workspace (the fields the GEMM reads are named as in BigdWs)
    uint16_t* xp;                    // [3 segments][3 parts][Ncp][Dp]  split rows, row e = list entry e (A operand)
    uint16_t* bp;                    // [3 segments][3 parts][Dp][Dp]   split P, M^-1 and Lc (tapes: M^-1 again) (B operand)
    float* g;                        // [3 segments][Ncp][Dp]           the products
    int* mode;                       // [Ncp] MD_FIRST: every row of an active row block is stored (rows past the list are not read)
    int* tile_active;                // [Ncp / 128] row blocks below the list length
    float* V0;                       // [Ncp] by workspace row: V(x0) of the running trajectory
    float binv;                      // 1: the bf16 split is not scaled
    int Ncp, NT, Dp;
};

size_t carve_metric(MetricWs& mw, unsigned char* ws, size_t off, long Nchain, int D) {
    BigdCarve c(ws, Nchain, D, 128);
    c.off = off;
    mw.Ncp = (int)c.Ncp; mw.NT = c.NT; mw.Dp = c.Dp; mw.binv = 1.f;
    mw.xp = (uint16_t*)c.take((size_t)9 * c.Ncp * c.Dp * 2);
    mw.bp = (uint16_t*)c.take((size_t)9 * c.Dp * c.Dp * 2);
    mw.g = (float*)c.take((size_t)3 * c.Ncp * c.Dp * 4);
    mw.mode = (int*)c.take(c.Ncp * 4);
    mw.tile_active = (int*)c.take((c.Ncp / BM) * 4);
    mw.V0 = (float*)c.take(c.Ncp * 4);
    return c.off;
}

__device__ __forceinline__ float row_dot(const float* u, const float* v, int Dp, int lane) {
    float s = 0.f;
    for (int j = lane; j < Dp; j += 32) s = fmaf(u[j], v[j], s);
    return warp_sum<float>(s);
}

__global__ void __launch_bounds__(256) bigd_gather(hmc_random_args a, BigdWs w, MetricWs mw, int pass, int start) {
    const int lane = threadIdx.x & 31, D = a.target.D, Dp = w.Dp;
    const int n = start ? a.Nchain : w.counters[pass & 1];
    const long nthr = (long)gridDim.x * blockDim.x;
    for (long t = (long)blockIdx.x * blockDim.x + threadIdx.x; t < mw.Ncp; t += nthr) {
        if (start) mw.mode[t] = MD_FIRST;
        if (t < mw.Ncp / BM) mw.tile_active[t] = t * BM < n;
    }
    const size_t seg = (size_t)3 * mw.Ncp * Dp;
    for (int e = blockIdx.x * 8 + (threadIdx.x >> 5); e < n; e += gridDim.x * 8) {
        const long m = start ? e : (w.list[e] & 0x7fffffff);
        const long c = w.perm[m];
        float* xr = w.x + (size_t)m * Dp;
        float* pr = w.p + (size_t)m * Dp;
        const int it = w.it[m];
        if (!start)
            for (int j = lane; j < Dp; j += 32) xr[j] = (xr[j] + w.mu[j]) - w.mu[j];
        bigd_write_parts<3>(mw.xp, mw.Ncp, Dp, e, lane, xr);
        // the momentum rows: at the start, the iteration-0 tape row (its K enters E_chain[., 0]) and p of the first iteration as
        // bigd_init drew it; at a trajectory end, p_L and the draw of the next iteration (none after the last).  A drawn row is
        // staged in the segment's product row, which the GEMM overwrites
        const bool fresh_tape = start && a.iter_begin == 0 && a.p_tape;
        if (!start || fresh_tape) {
            float* g1 = mw.g + ((size_t)mw.Ncp + e) * Dp;
            if (fresh_tape) bigd_momentum(a.p_tape + (size_t)c * (a.Niter + 1) * D, a.seed, 0, 0, D, Dp, lane, g1, D / 4);
            bigd_write_parts<3>(mw.xp + seg, mw.Ncp, Dp, e, lane, start ? g1 : pr);
        }
        if (start) {
            bigd_write_parts<3>(mw.xp + 2 * seg, mw.Ncp, Dp, e, lane, pr);
        } else if (it < a.iter_end) {
            float* g2 = mw.g + (2 * (size_t)mw.Ncp + e) * Dp;
            const double* tape = a.p_tape ? a.p_tape + ((size_t)c * (a.Niter + 1) + it + 1) * D : nullptr;
            bigd_momentum(tape, a.seed, (uint64_t)(a.chain_id0 + c), it + 1, D, Dp, lane, g2, D / 4);
            bigd_write_parts<3>(mw.xp + 2 * seg, mw.Ncp, Dp, e, lane, g2);
        }
    }
}

template <int NPART>
__global__ void __launch_bounds__(256) bigd_finish(hmc_random_args a, BigdWs w, MetricWs mw, int pass, int start) {
    const int lane = threadIdx.x & 31, D = a.target.D, Dp = w.Dp;
    const int n = start ? a.Nchain : w.counters[pass & 1];
    const long Lc = 1 + (a.Niter - a.warm_up_num) / a.thin_rate;
    const long Lrow = a.store_ring > 0 ? a.store_ring : Lc;
    const float* mu = w.mu;
    const float vc = (float)a.target.v_const;
    for (int e = blockIdx.x * 8 + (threadIdx.x >> 5); e < n; e += gridDim.x * 8) {
        const long m = start ? e : (w.list[e] & 0x7fffffff);
        const long c = w.perm[m];
        const float* gP = mw.g + (size_t)e * Dp;
        const float* gM = mw.g + ((size_t)mw.Ncp + e) * Dp;
        const float* gN = mw.g + (2 * (size_t)mw.Ncp + e) * Dp;
        float* xr = w.x + (size_t)m * Dp;
        float* x0r = w.x0 + (size_t)m * Dp;
        float* pr = w.p + (size_t)m * Dp;
        const float V = fmaf(0.5f, row_dot(xr, gP, Dp, lane), vc);                 // V(x_L), or V(x0) at the start
        // p0 of a new trajectory: Lc z from its product on Philox draws (K = z.z / 2 given), the tape row in pr with K from M^-1 p0
        auto momentum = [&](float Kz) {
            if (a.p_tape) return 0.5f * row_dot(pr, gN, Dp, lane);
            for (int j = lane; j < Dp; j += 32) pr[j] = gN[j];
            return Kz;
        };
        if (start) {
            float K0 = 0.f;
            if (a.p_tape && a.iter_begin == 0) {                                    // K of the iteration-0 tape row (samplers.py:415)
                const double* t0 = a.p_tape + (size_t)c * (a.Niter + 1) * D;
                float s = 0.f;
                for (int j = lane; j < D; j += 32) s = fmaf((float)t0[j], gM[j], s);
                K0 = 0.5f * warp_sum<float>(s);
            }
            const float Kn = momentum(w.K_new[m]);
            if (lane == 0) { mw.V0[m] = V; w.K_new[m] = Kn; if (a.p_tape && a.iter_begin == 0) w.K0[m] = K0; }
            continue;
        }
        const float K = 0.5f * row_dot(pr, gM, Dp, lane);                          // samplers.py:455
        int it = w.it[m];
        const float Ei = w.E_init[m];
        const float dE = (V + K) - Ei;
        const bool accepted = (dE < 0.f) || (w.lnu[m] < -dE);                       // samplers.py:462
        const bool keep = it >= a.warm_up_num;
        const bool last = it >= a.iter_end;
        if (lane == 0) {
            w.E_prev[m] = Ei;                                                       // samplers.py:460
            if (accepted) mw.V0[m] = V;
            if (accepted && a.counters) atomicAdd(a.counters + (keep ? 1 : 0), 1ull);
            if (a.phi_q && (a.chain_id0 + c) == 0 && it <= a.N_save_chain0) a.decision_chain[it - 1] = accepted ? 1 : 0;
        }
        float* dst = keep ? (float*)a.q_chain + ((size_t)c * Lrow + ((it - a.warm_up_num) / a.thin_rate) % Lrow) * D : nullptr;
        float* sq = last ? (float*)a.state_q + (size_t)c * D : nullptr;
        // accepted: start point <- proposal (samplers.py:463-469); rejected: proposal <- start point (samplers.py:470-472)
        const float* from = accepted ? xr : x0r;
        float* to = accepted ? x0r : xr;
        for (int j = lane; j < Dp; j += 32) {
            const float v = from[j];
            to[j] = v;
            if (j < D) {
                if (dst) dst[j] = v + mu[j];
                if (sq) sq[j] = v + mu[j];
            }
        }
        // the next pass's operand: x0 (the pass wrote x_L before its re-derivation)
        bigd_write_parts<NPART>(w.xp + (size_t)w.wr * NPART * w.Ncp * Dp, w.Ncp, Dp, m, lane, x0r);
        if (last) {
            if (lane == 0) { w.mode[m] = MD_IDLE; w.it[m] = it + 1; a.state_eprev[c] = (double)Ei; }
        } else {
            it += 1;
            int L = 1; float lnu = 0.f;
            const float Kz = bigd_draw(a, Dp, c, it, lane, a.p_tape ? pr : nullptr, &L, &lnu);   // samplers.py:431, 441, 461
            const float Kn = momentum(Kz);
            if (lane == 0) { w.K_new[m] = Kn; w.L[m] = L; w.lnu[m] = lnu; w.l[m] = 0; w.it[m] = it; w.mode[m] = MD_FIRST; }
        }
    }
}


// carve the workspace; returns the bytes needed (ws may be NULL to only size it)
size_t carve(BigdWs& w, unsigned char* ws, long Nchain, int D, int npart, int bn) {
    BigdCarve c(ws, Nchain, D, bn);
    const long Ncp = c.Ncp;
    const int Dp = c.Dp, NT = c.NT;
    w.Ncp = (int)Ncp; w.NT = NT; w.npart = npart; w.Dp = Dp;
    w.xp = (uint16_t*)c.take((size_t)2 * npart * Ncp * Dp * 2);
    w.bp = (uint16_t*)c.take((size_t)npart * Dp * Dp * 2);
    w.x = (float*)c.take((size_t)Ncp * Dp * 4);
    w.x0 = (float*)c.take((size_t)Ncp * Dp * 4);
    w.p = (float*)c.take((size_t)Ncp * Dp * 4);
    w.mu = (float*)c.take((size_t)Dp * 4);
    w.dt = (float*)c.take((size_t)Dp * 4);
    w.red = (float*)c.take((size_t)Ncp * NT * 2 * 2 * 4);
    w.mode = (int*)c.take(Ncp * 4); w.l = (int*)c.take(Ncp * 4); w.L = (int*)c.take(Ncp * 4); w.it = (int*)c.take(Ncp * 4); w.init = (int*)c.take(Ncp * 4);
    w.K_new = (float*)c.take(Ncp * 4); w.K0 = (float*)c.take(Ncp * 4); w.lnu = (float*)c.take(Ncp * 4); w.E_init = (float*)c.take(Ncp * 4);
    w.E_prev = (float*)c.take(Ncp * 4);
    w.tile_active = (int*)c.take((Ncp / BM) * 4);
    w.list = (int*)c.take(Ncp * 4);
    w.counters = (int*)c.take(64);
    w.perm = (int*)c.take(Ncp * 4);
    w.plan = (int*)c.take(Ncp * 4);
    return c.off;
}

constexpr const char* kName = "large-D kernel";

template <int NPART, int BN, int CL, int BK, int STAGES>
int run_bigd(const hmc_random_args& a, cudaStream_t stream) {
    const int D = a.target.D;
    const bool dense = a.target.Pt != nullptr;                   // (with Mit and Lct: hmc_random_bigd_supported)
    BigdWs w;
    MetricWs mw{};
    size_t need = carve(w, (unsigned char*)a.workspace, a.Nchain, D, NPART, BN);
    if (dense) need = carve_metric(mw, (unsigned char*)a.workspace, need, a.Nchain, D);
    if (int rc = bigd_check_workspace(a.workspace, a.workspace_bytes, need, kName, "hmc_random_workspace_bytes")) return rc;
    int dev = 0, sms = 0;
    HMC_CUDA_CHECK(cudaGetDevice(&dev));
    HMC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int Dp = w.Dp;
    CUtensorMap mapA[2], mapS[2], mapB, mapP, mapX;
    if (int rc = bigd_target_operands<NPART, BN, CL, BK>(a.target, w, sms, stream, &mapB)) return rc;
    for (int b = 0; b < 2; ++b) {
        uint16_t* xb = w.xp + (size_t)b * NPART * w.Ncp * Dp;
        if (int rc = make_map(&mapA[b], bigd_dt16<NPART>(), 2, xb, (uint64_t)NPART * w.Ncp, Dp, BK, BM)) return rc;      // operand loads
        if (int rc = make_map(&mapS[b], bigd_dt16<NPART>(), 2, xb, (uint64_t)NPART * w.Ncp, Dp, CW, 32)) return rc;      // epilogue stores
    }
    if (int rc = make_map(&mapP, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, w.p, (uint64_t)w.Ncp, Dp, CW, 32)) return rc;
    if (int rc = make_map(&mapX, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, w.x, (uint64_t)w.Ncp, Dp, CW, 32)) return rc;
    // dense metric: the three products' operands and GEMM (bf16x3, 128-column tiles, clusters of two row blocks)
    constexpr int MCL = 2;
    auto mkern = bigd_gemm_step<MetricWs, EPI_GRAD, 3, 128, MCL, 32, 2>;
    CUtensorMap mapMA[3], mapMB[3], mapMG[3];
    cudaLaunchConfig_t mcfg;
    cudaLaunchAttribute mattr;
    if (dense) {
        const void* mats[3] = {a.target.Pt, a.target.Mit, a.p_tape ? a.target.Mit : a.target.Lct};
        for (int sg = 0; sg < 3; ++sg) {
            uint16_t* xs = mw.xp + (size_t)sg * 3 * mw.Ncp * Dp;
            uint16_t* bs = mw.bp + (size_t)sg * 3 * Dp * Dp;
            bigd_split_matrix<3><<<sms * 8, 256, 0, stream>>>((const float*)mats[sg], D, a.target.D_pad, Dp, 1.f, bs);
            if (int rc = make_map(&mapMA[sg], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, xs, (uint64_t)3 * mw.Ncp, Dp, 32, BM)) return rc;
            if (int rc = make_map(&mapMB[sg], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, bs, (uint64_t)3 * Dp, Dp, 32, 128 / MCL)) return rc;
            if (int rc = make_map(&mapMG[sg], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, mw.g + (size_t)sg * mw.Ncp * Dp, (uint64_t)mw.Ncp, Dp, CW, 32))
                return rc;
        }
        if (int rc = bigd_launch_config(mcfg, mattr, mkern, MCL, (mw.Ncp / BM / MCL) * mw.NT, gemm_smem_bytes<3, 128, 32, 2>(), sms, stream,
                                        kName)) return rc;
    }
    // the list's per-trajectory products (`pass`: the list of that pass; start: every chain) up to the finish kernel, split in two
    // by the timing event `mid`
    auto metric_stage = [&](long pass, int start, cudaEvent_t mid) {
        bigd_gather<<<sms * 2, 256, 0, stream>>>(a, w, mw, (int)pass, start);
        for (int sg = 0; sg < 3; ++sg)
            if (cudaLaunchKernelEx(&mcfg, mkern, mapMA[sg], mapMB[sg], mapMG[sg], mapMG[sg], mapMG[sg], mw, mw.Ncp, Dp, (const float*)nullptr) !=
                cudaSuccess) return HMC_E_CUDA;
        if (mid) cudaEventRecord(mid, stream);
        bigd_finish<NPART><<<sms * 2, 256, 0, stream>>>(a, w, mw, (int)pass, start);
        return HMC_OK;
    };
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
    if (dense) if (int rc = metric_stage(0, 1, nullptr)) return bigd_loop_result(rc, kName);
    const int ntile_rows = w.Ncp / BM;
    HMC_CUDA_CHECK(cudaMemsetAsync(w.tile_active, 0xff, (size_t)ntile_rows * 4, stream));
    auto kern = bigd_gemm_step<BigdWs, EPI_LEAPFROG, NPART, BN, CL, BK, STAGES>;
    const int ntiles = (ntile_rows / CL) * w.NT;                 // work items of a cluster
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr;
    if (int rc = bigd_launch_config(cfg, attr, kern, CL, ntiles, gemm_smem_bytes<NPART, BN, BK, STAGES>(), sms, stream, kName)) return rc;
    const float* dtv = w.dt;
    const int Nch = a.Nchain;
    // pass n: operands from buffer n & 1, the epilogue (and the trajectory ends after it) write buffer (n + 1) & 1
    auto launch_gemm = [&](long pass) { w.wr = (int)((pass + 1) & 1);
                                        return cudaLaunchKernelEx(&cfg, kern, mapA[pass & 1], mapB, mapP, mapX, mapS[(pass + 1) & 1], w, Nch, Dp, dtv); };
    BigdRunning running;
    if (int rc = running.alloc()) return rc;
    const long max_pass = (long)(a.iter_end - a.iter_begin) * (a.L_high + 1) + 8;
    int rc = HMC_OK;
    // HMC_B200_BIGD_TIMING=1: CUDA-event times of the kernels of passes 4..11 on stderr (measurement aid); with a dense metric
    // the trajectory end is split into the product stage (gather + three GEMMs) and the finish kernel
    const bool timing = getenv("HMC_B200_BIGD_TIMING") != nullptr;
    const int nst = dense ? 4 : 3;
    cudaEvent_t ev[5];
    float tsum[4] = {0.f, 0.f, 0.f, 0.f};
    if (timing) for (int i = 0; i <= nst; ++i) cudaEventCreate(&ev[i]);
    for (long pass = 0; pass < max_pass; ++pass) {
        const bool timed = timing && pass >= 4 && pass < 12;
        if (timed) cudaEventRecord(ev[0], stream);
        if (launch_gemm(pass) != cudaSuccess) { rc = HMC_E_CUDA; break; }
        if (timed) cudaEventRecord(ev[1], stream);
        cudaMemsetAsync(w.counters + 2, 0, 4, stream);
        if (dense) {
            bigd_events<true><<<ntile_rows, BM, 0, stream>>>(a, w, (int)pass, mw.V0);
            if (timed) cudaEventRecord(ev[2], stream);
            if ((rc = metric_stage(pass, 0, timed ? ev[3] : nullptr)) != HMC_OK) break;
        } else {
            bigd_events<false><<<ntile_rows, BM, 0, stream>>>(a, w, (int)pass, nullptr);
            if (timed) cudaEventRecord(ev[2], stream);
            bigd_trajectory_end<NPART><<<sms * 2, 256, 0, stream>>>(a, w, (int)pass);
        }
        if (timed) {
            cudaEventRecord(ev[nst], stream);
            cudaEventSynchronize(ev[nst]);
            for (int i = 0; i < nst; ++i) { float ms = 0.f; cudaEventElapsedTime(&ms, ev[i], ev[i + 1]); tsum[i] += ms; }
            if (pass == 11 && !dense) fprintf(stderr, "[bigd timing] NPART=%d BN=%d BK=%d cluster=%d chains=%d D=%d: gemm_step %.3f ms, events %.3f ms, trajectory_end %.3f ms per pass (%d work items on %d CTAs)\n",
                                    NPART, BN, BK, CL, a.Nchain, D, tsum[0] / 8, tsum[1] / 8, tsum[2] / 8, ntiles, (int)cfg.gridDim.x);
            if (pass == 11 && dense) fprintf(stderr, "[bigd timing] NPART=%d BN=%d BK=%d cluster=%d chains=%d D=%d dense metric: gemm_step %.3f ms, events %.3f ms, products %.3f ms, finish %.3f ms per pass (%d work items on %d CTAs)\n",
                                             NPART, BN, BK, CL, a.Nchain, D, tsum[0] / 8, tsum[1] / 8, tsum[2] / 8, tsum[3] / 8, ntiles, (int)cfg.gridDim.x);
        }
        if ((pass & 7) == 7) {
            // chains that ended their last trajectory in this pass are still MD_PENDING for the events kernel's count: they are
            // counted as running and found idle at the next look
            const int n = running.read(w.counters, stream);
            if (n < 0) { rc = HMC_E_CUDA; break; }
            if (n == 0) break;
        }
    }
    if (timing) for (int i = 0; i <= nst; ++i) cudaEventDestroy(ev[i]);
    return bigd_loop_result(rc, kName);
}

}  // namespace

bool hmc_random_bigd_supported(const hmc_random_args& a, const char** why) {
    return bigd_covers(a.dtype, a.target, a.iter_begin, a.iter_end, why, true);
}

size_t hmc_random_bigd_workspace(const hmc_random_args& a) {
    BigdWs w;                                     // sized for the larger of the two variants
    MetricWs mw;
    const size_t n = carve(w, nullptr, a.Nchain, a.target.D, 3, 128);
    return a.target.Pt ? carve_metric(mw, nullptr, n, a.Nchain, a.target.D) : n;
}

int hmc_random_run_bigd(const hmc_random_args& a, cudaStream_t stream) {
    return bigd_run_variant(a.flags, [&](auto v) {
        using V = decltype(v);
        return run_bigd<V::NPART, V::BN, V::CL, V::BK, V::STAGES>(a, stream);
    });
}
