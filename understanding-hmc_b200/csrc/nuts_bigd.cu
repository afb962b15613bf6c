// Large-D NUTS path: HMC_sampler.gen_sample_NUTS (/root/reference/samplers.py:495-808) for float32, identity momentum metric and
// any 128 <= D <= 8192, with the gradient of all chains as the tcgen05 GEMM of the large-D path (bigd_gemm.cuh).
//
// Same semantics and draws as nuts_generic.cu / nuts_tc.cu: iterative doubling with a direction coin per doubling, uniform
// progressive sampling inside the new sub-trajectory, sub-tree U-turn checks at even points against the saved odd points (the
// closed forms of nuts_generic.cu), the biased old/new choice, termination when BOTH ends have turned (Q6), the |dE| > 1000
// guard, d_max (Q7), per-chain scalars in float64 (SURVEY H5).  Momenta hmc_normal4 keyed by (seed, global chain, iteration,
// slot), coins HMC_STREAM_NUTS, inner uniforms HMC_STREAM_NUTS_INNER -- or the injected tapes, consumed in order per chain.
//
// Each chain is a state machine that advances one leapfrog step per PASS (as in nuts_tc.cu):
//     STEP         the gradient is that of the new point: second half kick, energy, the reference's per-point logic
//     ITER_START   gradient at the start point of an iteration (fresh momentum): E_initial, first doubling
//     CHAIN_START  the same for a new chain (also records E_chain[., 0])
//     GRAD         gradient at the trajectory end a doubling switched to (a doubling that continues in the direction of the last
//                  one starts from the point whose gradient is at hand and needs no such pass)
// A pass is two kernels, enqueued back to back:
//   bigd_gemm_step<EPI_GRAD>  G[Ncp][Dp] = (q - mu) F^T for every row block with a chain that is not finished (the GEMM of the
//                  Random path, fp16x2 or bf16x3 split; its epilogue stores the fp32 gradient rows by TMA)
//   nuts_bigd_step one warp per chain, 128-bit accesses over the row: second half kick with G, energy (M = I:
//                  V = 0.5 (q - mu).g + v_const, K = 0.5 p.p), saves at odd points, check dots at even points, progressive
//                  sampling, live and boundary rows, end of a doubling, next coin, then the first half kick and drift of the next
//                  step; writes x, p and the split position (the next pass's A operand)
// Rows are chains in their own order (tree sizes are not known in advance, so there is no sort); a row block whose chains have
// all finished leaves the GEMM through tile_active.  The host looks at the number of running chains every 8 passes.  The set-up
// around the GEMM and the momentum-row / split-position helpers are shared with random_bigd.cu (bigd_gemm.cuh).
//
// State: the check-point stack and the live / boundary rows are the caller's scratch ([Nchain + 128][2 (d_max+1) + 7][D_pad],
// the layout of nuts_generic.cu, cursors of the injected streams in row R + 6).  Everything the GEMM touches is in the workspace,
// Dp = D rounded up to 32 wide and zero in the padded dimensions (no force, no momentum, dt = 0 there), as in random_bigd.cu.
// The position is kept shifted, x = q - mu; at every iteration end it is re-derived from the stored sample (x = (x + mu) - mu in
// float32), so a run split into iteration blocks (resumed from state_q) is bit-identical to a single launch.
//
// Unfused: G is written and read back (8 B per element and pass) and the step kernel reads / writes x, p and stack rows on top
// of the GEMM's operand traffic.
#include "bigd_gemm.cuh"
#include <cstdlib>
#include <cstdio>

namespace {

enum { HMC_STREAM_NUTS_INNER = 3 };
enum : int { NB_IDLE = 0, NB_CHAIN_START = 1, NB_ITER_START = 2, NB_STEP = 3, NB_GRAD = 4 };
constexpr int NB_WARPS = 16;                 // step kernel: 16 warps per block, 8 rows each = one 128-row block of the GEMM

struct NbChain {                             // per-chain state between passes (float64 scalars, SURVEY H5)
    double E_initial, E_prev, E_max_old, pi_old, E_max_new, pi_new, u_biased;
    long long n_dir, n_u;                    // cursors of the injected streams
    long long leap;                          // leapfrog steps of this launch
    int ph, it, depth, k, u_dir, doub, instab, dmax;
};

struct NbWs {                                // workspace carved by the host (all device pointers)
    uint16_t* xp;                            // [NPART][Ncp][Dp]  split position = A operand (the step kernel writes it after the GEMM has finished)
    uint16_t* bp;                            // [NPART][Dp][Dp]   split force matrix (x 2^s for the fp16 split), zero outside D x D
    float* x;                                // [Ncp][Dp] shifted position q - mu
    float* p;                                // [Ncp][Dp] momentum
    float* g;                                // [Ncp][Dp] gradient F (q - mu) of the last pass (the GEMM's output)
    float* mu;                               // [Dp] target mean, zero from D on
    float* dt;                               // [Dp] step sizes, zero from D on
    NbChain* ch;                             // [Ncp]
    int* mode;                               // [Ncp] MD_MID: the row takes part in the next GEMM, MD_IDLE: finished or padding
    int* tile_active;                        // [Ncp / 128]
    int* counters;                           // [2] running chains after the last step kernel; [8] matrix abs-max scratch
    unsigned long long* grads;               // [1] gradient rows evaluated (sum over passes of the running chains; timing aid)
    float binv;                              // 2^-s
    int Ncp, NT, Dp;
};

__device__ __forceinline__ double nb_unif(uint32_t w) { return ((double)(w >> 8) + 0.5) * 5.9604644775390625e-08; }

// momentum of (chain m, iteration) into the Dp-wide row pr (zero from D on); returns |p|^2 (warp-reduced).  Same draws as
// nuts_generic.cu: normal j of the row is component j & 3 of hmc_normal4(seed, chain, iteration, j >> 2).
__device__ float nb_draw(const hmc_nuts_args& a, int Dp, long m, int iter, int lane, float* pr) {
    const int D = a.target.D;
    const double* tape = a.p_tape ? a.p_tape + ((size_t)m * (a.Niter + 1) + iter) * D : nullptr;
    return warp_sum<float>(bigd_momentum(tape, a.seed, (uint64_t)(a.chain_id0 + m), iter, D, Dp, lane, pr, 0));
}

// chain start (samplers.py:548-555) or resume from state_q / state_eprev / the cursors: one warp per row
template <int NPART>
__global__ void __launch_bounds__(128) nuts_bigd_init(hmc_nuts_args a, NbWs w) {
    const int lane = threadIdx.x & 31, D = a.target.D, Dp = w.Dp, Dpad = a.target.D_pad;
    const long m = (long)blockIdx.x * 4 + (threadIdx.x >> 5);
    if (m >= w.Ncp) return;
    float* xr = w.x + (size_t)m * Dp;
    float* pr = w.p + (size_t)m * Dp;
    if (m >= a.Nchain) {                                                    // padding rows of the last row blocks
        for (int j = lane; j < Dp; j += 32) { xr[j] = 0.f; pr[j] = 0.f; }
        bigd_write_parts<NPART>(w.xp, w.Ncp, Dp, m, lane, xr);
        if (lane == 0) { w.mode[m] = MD_IDLE; w.ch[m].ph = NB_IDLE; }
        return;
    }
    const bool fresh = a.iter_begin == 0;
    const float* src = (fresh ? (const float*)a.q_start : (const float*)a.state_q) + (size_t)m * D;
    const long Lc = 1 + (a.Niter - a.warm_up_num) / a.thin_rate;
    for (int j = lane; j < Dp; j += 32) {
        const float v = j < D ? src[j] : 0.f;
        if (fresh && j < D) ((float*)a.q_chain)[(size_t)m * Lc * D + j] = v;           // samplers.py:548
        xr[j] = v - w.mu[j];
    }
    bigd_write_parts<NPART>(w.xp, w.Ncp, Dp, m, lane, xr);
    const int R = 2 * (a.d_max + 1);
    const long long* cur = reinterpret_cast<const long long*>((const float*)a.scratch + ((size_t)m * (R + 7) + R + 6) * Dpad);
    nb_draw(a, Dp, m, fresh ? 0 : a.iter_begin + 1, lane, pr);                      // samplers.py:549 / 565
    if (lane == 0) {
        NbChain c = {};
        c.ph = fresh ? NB_CHAIN_START : NB_ITER_START;
        c.it = a.iter_begin + 1;
        c.E_prev = fresh ? 0.0 : a.state_eprev[m];
        if (!fresh && a.dir_tape) { c.n_dir = cur[0]; c.n_u = cur[1]; }             // resume the injected streams
        w.ch[m] = c;
        w.mode[m] = MD_MID;
    }
}

// one pass of the state machine: one warp per chain, 16 warps = the 128 rows of one GEMM row block
template <int NPART>
__global__ void __launch_bounds__(32 * NB_WARPS) nuts_bigd_step(hmc_nuts_args a, NbWs w) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int D = a.target.D, Dp = w.Dp, Dpad = a.target.D_pad;
    const int R = 2 * (a.d_max + 1);
    const long Lc = 1 + (a.Niter - a.warm_up_num) / a.thin_rate;
    const double vconst = a.target.v_const;
    const bool ext4 = (D & 3) == 0;            // the caller's rows (stored samples, state_q) are D wide: 16-byte aligned only then
    int alive = 0;
    for (int r = 0; r < BM / NB_WARPS; ++r) {
        const long m = (long)blockIdx.x * BM + r * NB_WARPS + wid;
        if (m >= a.Nchain) break;
        NbChain c = w.ch[m];
        if (c.ph == NB_IDLE) continue;
        const uint64_t gid = (uint64_t)(a.chain_id0 + m);
        float* xr = w.x + (size_t)m * Dp;
        float* pr = w.p + (size_t)m * Dp;
        const float* gr = w.g + (size_t)m * Dp;
        const float* dt = w.dt;
        float* scr = (float*)a.scratch + (size_t)m * (R + 7) * Dpad;
        auto row = [&](int i) { return scr + (size_t)i * Dpad; };
        // copies between the workspace rows (Dp wide) and stack rows (D_pad wide; the workspace is zero beyond D); every lane
        // touches the same elements in every loop of this kernel, so no warp synchronisation is needed between them
        auto store_row = [&](int i, const float* v, float sgn) {
            float* d = row(i);
            for (int j = 4 * lane; j < Dpad; j += 128) {
                const float4 t = *reinterpret_cast<const float4*>(v + j);
                *reinterpret_cast<float4*>(d + j) = make_float4(sgn * t.x, sgn * t.y, sgn * t.z, sgn * t.w);
            }
        };
        auto load_row = [&](int i, float* v) {
            const float* s = row(i);
            for (int j = 4 * lane; j < Dpad; j += 128) *reinterpret_cast<float4*>(v + j) = *reinterpret_cast<const float4*>(s + j);
        };
        auto copy_rows = [&](int from, int to) {
            const float* s = row(from);
            float* d = row(to);
            for (int j = 4 * lane; j < Dpad; j += 128) *reinterpret_cast<float4*>(d + j) = *reinterpret_cast<const float4*>(s + j);
        };
        auto draw_dir = [&](int iter, int dep) -> int {
            if (a.dir_tape) return a.dir_tape[(size_t)m * a.tape_dir_stride + c.n_dir++];
            const Philox4 rr = philox4x32_10((uint32_t)gid, (uint32_t)iter, (uint32_t)dep, HMC_STREAM_NUTS | ((uint32_t)(gid >> 32) << 8),
                                             (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
            c.u_biased = nb_unif(rr.y);
            return (int)(rr.x >> 31);
        };
        auto draw_u_inner = [&](int iter, int dep, int kk) -> double {
            if (a.u_tape) return a.u_tape[(size_t)m * a.tape_u_stride + c.n_u++];
            // step kk of the sub-trajectory of depth dep uses word (kk & 3) of Philox counter ((1 << dep) + kk) >> 2
            const Philox4 rr = philox4x32_10((uint32_t)gid, (uint32_t)iter, ((1u << dep) + (uint32_t)kk) >> 2,
                                             HMC_STREAM_NUTS_INNER | ((uint32_t)(gid >> 32) << 8), (uint32_t)a.seed, (uint32_t)(a.seed >> 32));
            return nb_unif((kk & 3) == 0 ? rr.x : (kk & 3) == 1 ? rr.y : (kk & 3) == 2 ? rr.z : rr.w);
        };

        // ===== consume the gradient: second half kick (STEP), q.g and p.p, the save of an odd point =========================
        const bool stepping = c.ph == NB_STEP;
        const int pt = c.k + 1;                                         // number of the point the step reached
        const bool save = stepping && (pt & 1);                         // odd point (1 included): samplers.py:623-626, 654-658
        const int sslot = __popc((unsigned)(pt - 1) >> 1);
        float hv = 0.f, hk = 0.f;
        for (int j = 4 * lane; j < Dp; j += 128) {
            const float4 g4 = *reinterpret_cast<const float4*>(gr + j), x4 = *reinterpret_cast<const float4*>(xr + j);
            float4 p4 = *reinterpret_cast<const float4*>(pr + j);
            hv = fmaf(x4.x, g4.x, fmaf(x4.y, g4.y, fmaf(x4.z, g4.z, fmaf(x4.w, g4.w, hv))));
            if (stepping) {                                             // samplers.py:837
                const float4 d4 = *reinterpret_cast<const float4*>(dt + j);
                p4.x = fmaf(g4.x, -0.5f * d4.x, p4.x); p4.y = fmaf(g4.y, -0.5f * d4.y, p4.y);
                p4.z = fmaf(g4.z, -0.5f * d4.z, p4.z); p4.w = fmaf(g4.w, -0.5f * d4.w, p4.w);
                *reinterpret_cast<float4*>(pr + j) = p4;
            }
            hk = fmaf(p4.x, p4.x, fmaf(p4.y, p4.y, fmaf(p4.z, p4.z, fmaf(p4.w, p4.w, hk))));
            if (save && j < Dpad) {
                *reinterpret_cast<float4*>(row(sslot) + j) = x4;
                *reinterpret_cast<float4*>(row(a.d_max + 1 + sslot) + j) = p4;
            }
        }
        const double V = 0.5 * (double)warp_sum<float>(hv) + vconst;   // utils.py:213-218
        const double Kc = 0.5 * (double)warp_sum<float>(hk);

        // ===== the chain's state machine ================================================================================
        bool finish = false, new_doubling = false, traj_test = false, start_iter = false;
        if (c.ph == NB_CHAIN_START) {
            const double E0 = V + Kc;                                   // samplers.py:551-555
            if (lane == 0) { a.E_chain[(size_t)m * Lc] = E0; a.dE_chain[(size_t)m * Lc] = 0.0; }
            c.E_prev = E0;
            const float s = nb_draw(a, Dp, m, c.it, lane, pr);          // samplers.py:565: the momentum of the first iteration
            c.E_initial = V + 0.5 * (double)s;                          // samplers.py:569 (same position, same gradient)
            start_iter = true;
        } else if (c.ph == NB_ITER_START) {
            c.E_initial = V + Kc;                                       // samplers.py:569
            start_iter = true;
        } else if (c.ph == NB_STEP) {
            c.leap++;
            const double E_tmp = V + Kc;                                // samplers.py:618, 643
            bool reject = false;
            if (c.k == 0) {                                             // first point of the new sub-trajectory (samplers.py:611-626)
                store_row(R + 0, xr, 1.f);
                c.E_max_new = E_tmp;
                c.pi_new = 1.0;
            } else if (fabs(E_tmp - c.E_initial) > 1000.0) {            // samplers.py:647-651
                reject = true;
                c.instab++;
            } else {
                if (!(pt & 1)) {                                        // even point: sub-tree U-turn checks (samplers.py:699-736)
                    for (int jj = __ffs(pt) - 1; jj >= 1; --jj) {
                        const int l = pt - (1 << jj) + 1;
                        const int slot = __popc((unsigned)(l - 1) >> 1);
                        const float* qs = row(slot);
                        const float* ps = row(a.d_max + 1 + slot);
                        float s_cur = 0.f, s_chk = 0.f;                 // (q - q_check).p  and  (q - q_check).p_check
                        for (int j = 4 * lane; j < Dpad; j += 128) {
                            const float4 x4 = *reinterpret_cast<const float4*>(xr + j), p4 = *reinterpret_cast<const float4*>(pr + j);
                            const float4 qc = *reinterpret_cast<const float4*>(qs + j), pc = *reinterpret_cast<const float4*>(ps + j);
                            const float d0 = x4.x - qc.x, d1 = x4.y - qc.y, d2 = x4.z - qc.z, d3 = x4.w - qc.w;
                            s_cur = fmaf(d0, p4.x, fmaf(d1, p4.y, fmaf(d2, p4.z, fmaf(d3, p4.w, s_cur))));
                            s_chk = fmaf(d0, pc.x, fmaf(d1, pc.y, fmaf(d2, pc.z, fmaf(d3, pc.w, s_chk))));
                        }
                        // the same two signs for either direction (nuts_generic.cu)
                        if (warp_sum<float>(s_cur) < 0.f && warp_sum<float>(s_chk) < 0.f) { reject = true; break; }
                    }
                }
                if (!reject) {                                          // uniform progressive sampling (samplers.py:743-751)
                    const double E_prev_max = c.E_max_new;
                    c.E_max_new = fmax(E_prev_max, E_tmp);
                    const double ex = exp(fabs(E_tmp - E_prev_max));
                    const bool new_max = E_tmp > E_prev_max;
                    const double numer = new_max ? 1.0 : ex;
                    c.pi_new = numer + (new_max ? ex : 1.0) * c.pi_new;
                    if (draw_u_inner(c.it, c.depth, c.k) < numer / c.pi_new) store_row(R + 0, xr, 1.f);
                }
            }
            if (reject) finish = true;                                  // samplers.py:754-755: the sample stays live_old
            else if (c.k == (1 << c.depth) - 1) {
                // the new sub-trajectory is complete: extend the end (samplers.py:758-761), biased choice (:766-776, Q8)
                if (c.u_dir == 0) { store_row(R + 4, xr, 1.f); store_row(R + 5, pr, 1.f); }
                else { store_row(R + 2, xr, 1.f); store_row(R + 3, pr, 1.f); }
                const double rb = exp(-(c.E_max_new - c.E_max_old)) * c.pi_old / c.pi_new;
                const double E_max_old_prev = c.E_max_old;
                c.E_max_old = fmax(E_max_old_prev, c.E_max_new);
                c.pi_old = exp(-(c.E_max_new - c.E_max_old)) * c.pi_new + exp(-(E_max_old_prev - c.E_max_old)) * c.pi_old;
                const double A = fmin(1.0, rb);
                const double ub = a.u_tape ? a.u_tape[(size_t)m * a.tape_u_stride + c.n_u++] : c.u_biased;
                if (ub < A) copy_rows(R + 0, R + 1);                    // live_old <- live_new
                // whole-trajectory U-turn test (samplers.py:779-781): the other end comes from the stack rows
                const float* oq = row(c.u_dir == 0 ? R + 2 : R + 4);
                const float* op = row(c.u_dir == 0 ? R + 3 : R + 5);
                float s_r = 0.f, s_l = 0.f;
                for (int j = 4 * lane; j < Dpad; j += 128) {
                    const float4 x4 = *reinterpret_cast<const float4*>(xr + j), p4 = *reinterpret_cast<const float4*>(pr + j);
                    const float4 q4 = *reinterpret_cast<const float4*>(oq + j), o4 = *reinterpret_cast<const float4*>(op + j);
                    const float xv[4] = {x4.x, x4.y, x4.z, x4.w}, pv[4] = {p4.x, p4.y, p4.z, p4.w};
                    const float oqv[4] = {q4.x, q4.y, q4.z, q4.w}, opv[4] = {o4.x, o4.y, o4.z, o4.w};
#pragma unroll
                    for (int e = 0; e < 4; ++e) {                       // dq = right_q - left_q; s_r = dq.right_p; s_l = -dq.left_p
                        const float dq = (c.u_dir == 0) ? xv[e] - oqv[e] : oqv[e] - xv[e];
                        s_r = fmaf(dq, (c.u_dir == 0) ? pv[e] : opv[e], s_r);
                        s_l = fmaf(-dq, (c.u_dir == 0) ? opv[e] : pv[e], s_l);
                    }
                }
                const bool right_term = warp_sum<float>(s_r) < 0.f, left_term = warp_sum<float>(s_l) < 0.f;
                traj_test = true;
                c.depth += 1;                                           // samplers.py:784
                if (left_term && right_term) finish = true;             // samplers.py:595 (Q6: both ends)
                else new_doubling = true;
            } else {
                c.k += 1;                                               // next point of the sub-trajectory
            }
        }
        if (start_iter) {
            // samplers.py:571-594: stored energies, live point, both boundary points, running maxima
            if (c.it >= a.warm_up_num && lane == 0) {
                const long idx = (c.it - a.warm_up_num) / a.thin_rate;
                a.E_chain[(size_t)m * Lc + idx] = c.E_initial;
                a.dE_chain[(size_t)m * Lc + idx] = c.E_initial - c.E_prev;
            }
            store_row(R + 1, xr, 1.f);
            store_row(R + 2, xr, 1.f);
            store_row(R + 3, pr, -1.f);
            store_row(R + 4, xr, 1.f);
            store_row(R + 5, pr, 1.f);
            c.E_max_old = c.E_initial; c.pi_old = 1.0;
            c.depth = 0;
            new_doubling = true;
        }
        int next_ph = c.ph;
        bool advance = false, new_x = false;
        if (new_doubling && !finish) {
            if (c.depth > a.d_max - 1) {                                // samplers.py:596-598 (Q7)
                c.dmax++;
                if (a.status && lane == 0) a.status[m] |= 1;
                finish = true;
            } else {
                c.doub++;
                const int prev_dir = c.u_dir;
                c.u_dir = draw_dir(c.it, c.depth);                      // samplers.py:608
                c.k = 0;
                next_ph = NB_STEP;
                if (start_iter) {
                    // both ends are the current point: the left end carries -p (samplers.py:577-594, 611-614)
                    if (c.u_dir == 1)
                        for (int j = 4 * lane; j < Dp; j += 128) {
                            const float4 t = *reinterpret_cast<const float4*>(pr + j);
                            *reinterpret_cast<float4*>(pr + j) = make_float4(-t.x, -t.y, -t.z, -t.w);
                        }
                    advance = true;
                } else if (c.u_dir == prev_dir) {
                    advance = true;                                     // this end is the current point and G is its gradient
                } else {
                    load_row(c.u_dir == 0 ? R + 4 : R + 2, xr);         // the other end (samplers.py:611-614): its gradient first
                    load_row(c.u_dir == 0 ? R + 5 : R + 3, pr);
                    new_x = true;
                    next_ph = NB_GRAD;
                }
            }
        } else if (c.ph == NB_GRAD) {
            advance = true; next_ph = NB_STEP;
        } else if (c.ph == NB_STEP && !finish && !traj_test) {
            advance = true;
        }
        if (finish) {
            // samplers.py:787-791: E_previous; the stored sample is live_old, and the next iteration starts from it as stored
            c.E_prev = c.E_initial;
            const bool keep = c.it >= a.warm_up_num;
            const bool last = c.it >= a.iter_end;
            float* dst = keep ? (float*)a.q_chain + ((size_t)m * Lc + (c.it - a.warm_up_num) / a.thin_rate) * D : nullptr;
            float* sq = last ? (float*)a.state_q + (size_t)m * D : nullptr;
            const float* lo = row(R + 1);
            for (int j = 4 * lane; j < Dpad; j += 128) {
                const float4 v = *reinterpret_cast<const float4*>(lo + j), mu4 = *reinterpret_cast<const float4*>(w.mu + j);
                const float4 q = make_float4(v.x + mu4.x, v.y + mu4.y, v.z + mu4.z, v.w + mu4.w);
                *reinterpret_cast<float4*>(xr + j) = make_float4(q.x - mu4.x, q.y - mu4.y, q.z - mu4.z, q.w - mu4.w);
                if (ext4) {
                    if (dst) *reinterpret_cast<float4*>(dst + j) = q;
                    if (sq) *reinterpret_cast<float4*>(sq + j) = q;
                }
            }
            if (!ext4) {
                __syncwarp();
                for (int j = lane; j < D; j += 32) {
                    const float q = lo[j] + w.mu[j];
                    if (dst) dst[j] = q;
                    if (sq) sq[j] = q;
                }
            }
            if (last) {
                // chain done for this launch: resume state, per-chain records, counters
                if (lane == 0) {
                    a.state_eprev[m] = c.E_prev;
                    long long* cur = reinterpret_cast<long long*>(row(R + 6));
                    cur[0] = c.n_dir; cur[1] = c.n_u;
                    if (a.n_leapfrog) a.n_leapfrog[m] += (int64_t)c.leap;
                    atomicAdd(a.counters + 0, (unsigned long long)c.leap);
                    atomicAdd(a.counters + 1, (unsigned long long)c.doub);
                    atomicAdd(a.counters + 2, (unsigned long long)c.instab);
                    atomicAdd(a.counters + 3, (unsigned long long)c.dmax);
                }
                next_ph = NB_IDLE;
            } else {
                c.it += 1;
                nb_draw(a, Dp, m, c.it, lane, pr);                      // samplers.py:565
                new_x = true;
                next_ph = NB_ITER_START;
            }
        }
        if (advance) {
            // first half kick + drift of the next leapfrog step (samplers.py:835-836)
            for (int j = 4 * lane; j < Dp; j += 128) {
                const float4 g4 = *reinterpret_cast<const float4*>(gr + j), d4 = *reinterpret_cast<const float4*>(dt + j);
                float4 x4 = *reinterpret_cast<const float4*>(xr + j), p4 = *reinterpret_cast<const float4*>(pr + j);
                p4.x = fmaf(g4.x, -0.5f * d4.x, p4.x); p4.y = fmaf(g4.y, -0.5f * d4.y, p4.y);
                p4.z = fmaf(g4.z, -0.5f * d4.z, p4.z); p4.w = fmaf(g4.w, -0.5f * d4.w, p4.w);
                x4.x = fmaf(p4.x, d4.x, x4.x); x4.y = fmaf(p4.y, d4.y, x4.y); x4.z = fmaf(p4.z, d4.z, x4.z); x4.w = fmaf(p4.w, d4.w, x4.w);
                *reinterpret_cast<float4*>(pr + j) = p4;
                *reinterpret_cast<float4*>(xr + j) = x4;
            }
            new_x = true;
        }
        if (new_x) bigd_write_parts<NPART>(w.xp, w.Ncp, Dp, m, lane, xr);
        c.ph = next_ph;
        if (lane == 0) { w.ch[m] = c; w.mode[m] = next_ph == NB_IDLE ? MD_IDLE : MD_MID; }
        alive += next_ph != NB_IDLE;
    }
    // the rows of this block are one row block of the GEMM
    __shared__ int nrun[NB_WARPS];
    if (lane == 0) nrun[wid] = alive;
    __syncthreads();
    if (threadIdx.x == 0) {
        int n = 0;
        for (int i = 0; i < NB_WARPS; ++i) n += nrun[i];
        w.tile_active[blockIdx.x] = n > 0;
        if (n) { atomicAdd(&w.counters[2], n); atomicAdd(w.grads, (unsigned long long)n); }
    }
}

size_t carve(NbWs& w, unsigned char* ws, long Nchain, int D, int npart, int bn) {
    BigdCarve c(ws, Nchain, D, bn);
    const long Ncp = c.Ncp;
    const int Dp = c.Dp;
    w.Ncp = (int)Ncp; w.NT = c.NT; w.Dp = Dp;
    w.xp = (uint16_t*)c.take((size_t)npart * Ncp * Dp * 2);
    w.bp = (uint16_t*)c.take((size_t)npart * Dp * Dp * 2);
    w.x = (float*)c.take((size_t)Ncp * Dp * 4);
    w.p = (float*)c.take((size_t)Ncp * Dp * 4);
    w.g = (float*)c.take((size_t)Ncp * Dp * 4);
    w.mu = (float*)c.take((size_t)Dp * 4);
    w.dt = (float*)c.take((size_t)Dp * 4);
    w.ch = (NbChain*)c.take((size_t)Ncp * sizeof(NbChain));
    w.mode = (int*)c.take(Ncp * 4);
    w.tile_active = (int*)c.take((Ncp / BM) * 4);
    w.counters = (int*)c.take(64);
    w.grads = (unsigned long long*)c.take(8);
    return c.off;
}

constexpr const char* kName = "large-D NUTS kernel";

template <int NPART, int BN, int CL, int BK, int STAGES>
int run_nuts_bigd(const hmc_nuts_args& a, cudaStream_t stream) {
    const int D = a.target.D;
    NbWs w;
    const size_t need = carve(w, (unsigned char*)a.workspace, a.Nchain, D, NPART, BN);
    if (int rc = bigd_check_workspace(a.workspace, a.workspace_bytes, need, kName, "hmc_nuts_workspace_bytes")) return rc;
    int dev = 0, sms = 0;
    HMC_CUDA_CHECK(cudaGetDevice(&dev));
    HMC_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const int Dp = w.Dp;
    HMC_CUDA_CHECK(cudaMemsetAsync(w.grads, 0, 8, stream));
    CUtensorMap mapA, mapB, mapG;
    if (int rc = bigd_target_operands<NPART, BN, CL, BK>(a.target, w, sms, stream, &mapB)) return rc;
    if (int rc = make_map(&mapA, bigd_dt16<NPART>(), 2, w.xp, (uint64_t)NPART * w.Ncp, Dp, BK, BM)) return rc;          // operand loads
    if (int rc = make_map(&mapG, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, w.g, (uint64_t)w.Ncp, Dp, CW, 32)) return rc;   // gradient stores
    nuts_bigd_init<NPART><<<(w.Ncp + 3) / 4, 128, 0, stream>>>(a, w);
    const int ntile_rows = w.Ncp / BM;
    HMC_CUDA_CHECK(cudaMemsetAsync(w.tile_active, 0xff, (size_t)ntile_rows * 4, stream));
    auto kern = bigd_gemm_step<NbWs, EPI_GRAD, NPART, BN, CL, BK, STAGES>;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute attr;
    if (int rc = bigd_launch_config(cfg, attr, kern, CL, (ntile_rows / CL) * w.NT, gemm_smem_bytes<NPART, BN, BK, STAGES>(), sms, stream,
                                    kName)) return rc;
    const int Nch = a.Nchain;
    auto launch_gemm = [&]() { return cudaLaunchKernelEx(&cfg, kern, mapA, mapB, mapG, mapG, mapG, w, Nch, Dp, (const float*)w.dt); };
    BigdRunning running;
    if (int rc = running.alloc()) return rc;
    // a chain needs at most 1 + d_max gradient-only passes and 2^d_max - 1 steps per iteration, plus its chain start
    const long max_pass = (long)(a.iter_end - a.iter_begin) * ((1L << a.d_max) + a.d_max + 2) + 8;
    int rc = HMC_OK;
    // HMC_B200_BIGD_TIMING=1: CUDA-event times of the GEMM and the step kernel of passes 4..11, and at the end the number of passes
    // and of gradient rows evaluated, on stderr (measurement aid)
    const bool timing = getenv("HMC_B200_BIGD_TIMING") != nullptr;
    cudaEvent_t ev[3];
    float tsum[2] = {0.f, 0.f};
    if (timing) for (int i = 0; i < 3; ++i) cudaEventCreate(&ev[i]);
    long pass = 0;
    for (; pass < max_pass; ++pass) {
        const bool timed = timing && pass >= 4 && pass < 12;
        if (timed) cudaEventRecord(ev[0], stream);
        if (launch_gemm() != cudaSuccess) { rc = HMC_E_CUDA; break; }
        if (timed) cudaEventRecord(ev[1], stream);
        cudaMemsetAsync(w.counters + 2, 0, 4, stream);
        nuts_bigd_step<NPART><<<ntile_rows, 32 * NB_WARPS, 0, stream>>>(a, w);
        if (timed) {
            cudaEventRecord(ev[2], stream);
            cudaEventSynchronize(ev[2]);
            for (int i = 0; i < 2; ++i) { float ms = 0.f; cudaEventElapsedTime(&ms, ev[i], ev[i + 1]); tsum[i] += ms; }
            if (pass == 11) fprintf(stderr, "[nuts bigd timing] NPART=%d BN=%d cluster=%d chains=%d D=%d: gemm %.3f ms, step %.3f ms per pass (passes 4..11)\n",
                                    NPART, BN, CL, a.Nchain, D, tsum[0] / 8, tsum[1] / 8);
        }
        if ((pass & 7) == 7) {
            const int n = running.read(w.counters, stream);
            if (n < 0) { rc = HMC_E_CUDA; break; }
            if (n == 0) { ++pass; break; }
        }
    }
    if (rc == HMC_OK && pass >= max_pass) {                       // the bound holds every chain's passes: this look finds none running
        const int n = running.read(w.counters, stream);
        if (n < 0) rc = HMC_E_CUDA;
        else if (n != 0) {
            hmc_set_error("large-D NUTS kernel: %d chains still running after %ld passes", n, max_pass);
            return HMC_E_CUDA;
        }
    }
    if (timing) {
        unsigned long long ng = 0;
        cudaMemcpyAsync(&ng, w.grads, 8, cudaMemcpyDeviceToHost, stream);
        cudaStreamSynchronize(stream);
        fprintf(stderr, "[nuts bigd passes] passes=%ld gradient_rows=%llu chains=%d\n", pass, ng, a.Nchain);
        for (int i = 0; i < 3; ++i) cudaEventDestroy(ev[i]);
    }
    return bigd_loop_result(rc, kName);
}

}  // namespace

bool hmc_nuts_bigd_supported(const hmc_nuts_args& a, const char** why) {
    return bigd_covers(a.dtype, a.target, a.iter_begin, a.iter_end, why);
}

size_t hmc_nuts_bigd_workspace(const hmc_nuts_args& a) {
    NbWs w;                                       // sized for the larger of the two splits
    return carve(w, nullptr, a.Nchain, a.target.D, 3, 128);
}

// bf16x3 unless the caller asks for fp16x2 (tree decisions are sign tests and near-ties; DESIGN 4.0 / 4.7)
int hmc_nuts_run_bigd(const hmc_nuts_args& a, cudaStream_t stream) {
    return bigd_run_variant(a.flags, [&](auto v) {
        using V = decltype(v);
        return run_nuts_bigd<V::NPART, V::BN, V::CL, V::BK, V::STAGES>(a, stream);
    });
}
