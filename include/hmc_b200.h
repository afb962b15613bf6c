/*
 * hmc_b200.h -- C-ABI of the B200-native HMC hot path (libhmc_b200.so).
 *
 * The reference (jaekor91/understanding-HMC) is pure Python and has no FFI layer; the boundary it exposes is
 * the class API of samplers.py / utils.py.  Each entry point below replaces the body of one reference
 * method (cited per function); the Python mirror of that API (understanding-hmc_b200/samplers.py, utils.py)
 * binds these symbols with ctypes.  See INTEGRATION.md for the reference-side binding.
 *
 * Conventions: extern "C", int status return (0 = ok, see HMC_E_*), no exceptions cross the boundary, every
 * buffer is caller-allocated DEVICE memory (e.g. torch tensors' data_ptr()) unless marked "host", the library
 * keeps no memory between calls, work is enqueued on the caller's cudaStream_t (passed as void*) and is
 * asynchronous with respect to the host.  Thread-compatible: one stream per device per thread.
 *
 * Data layout in HBM (DESIGN.md "Data layout"), the reference's own (samplers.py:33, 359-360), chain-major:
 *   q_chain   [Nchain][L_chain][D]   sample stream in the compute dtype; one stored sample = one contiguous row
 *   E_chain   [Nchain][L_chain]      float64 (per-chain scalars are always float64)
 *   dE_chain  [Nchain][L_chain]      float64
 * with L_chain = 1 + (Niter - warm_up_num) / thin_rate (samplers.py:31).  Chains shard over GPUs as contiguous
 * slabs; a chain's whole time series is contiguous, which keeps the lagged re-reads of the variogram in L2.
 */
#ifndef HMC_B200_H
#define HMC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HMC_B200_VERSION 100

enum {
    HMC_OK = 0,
    HMC_E_BADARG = 1,      /* argument check failed (the reference's ctor/shape asserts: samplers.py:331-348, 396, 510) */
    HMC_E_UNSUPPORTED = 2, /* configuration outside what the CUDA kernels cover (there is NO CPU fallback) */
    HMC_E_CUDA = 3,        /* a CUDA runtime call failed; see hmc_last_error_string() */
    HMC_E_DMAX = 4         /* NUTS: some chain needed depth > d_max (samplers.py:596-598 `assert False`) */
};

enum { HMC_F32 = 0, HMC_F64 = 1 };

/* which kernel implements the run */
enum {
    HMC_KERNEL_AUTO = 0,    /* tensor-core kernel if it covers the run, else the large-D GEMM path (when a workspace is given and
                               D % 256 == 0 or D > 1024; with a dense momentum metric for D > 1024 only), else the FFMA2 kernel, else
                               the generic one.  NUTS: the tensor-core kernel,
                               else the large-D path when a workspace is given, it covers the run and D > 256, else the generic one
                               (with hmc_nuts_args.store_ring > 0: the large-D path from D = 128, nothing else) */
    HMC_KERNEL_GENERIC = 1, /* one warp per chain, any D <= 1024 (NUTS: D <= 256), float or double (parity workhorse) */
    HMC_KERNEL_FAST = 2,    /* FP32 FFMA2 register-tile kernel, 20 < D <= 128, identity momentum metric */
    HMC_KERNEL_TC = 3,      /* tcgen05 tensor-core kernel (bf16x3 / fp16x2 split, fp32 accumulate in TMEM), D <= 100 and a multiple of 4
                               (smaller targets run zero padded in the 100-wide tile; AUTO picks it from D = 52), identity metric */
    HMC_KERNEL_BIGD = 4     /* large D, any 128 <= D <= 8192, float32, identity metric: one tcgen05 GEMM over all chains per leapfrog
                               step, operands by TMA, the leapfrog update fused into the epilogue; works on D rounded up to 32 (the
                               padded dimensions stay zero); needs hmc_random_args.workspace.  The Random sampler also takes a dense
                               momentum metric (target.Pt, Mit and Lct) for 1024 < D <= 8192: the steps multiply by F = M^-1 P as
                               always, and V, K and the momentum draw p = Lc z are batched tensor-core products (bf16x3) of the chains
                               that end or start a trajectory in a pass.  Up to D = 1024 the generic kernel runs a dense metric, and
                               this path refuses it there.  NUTS too (hmc_nuts_args.workspace, identity metric only): the same GEMM
                               writes the gradient rows and a step kernel advances every chain's tree by one point */
};

/* hmc_random_args.flags, hmc_nuts_args.flags */
enum {
    HMC_FLAG_UNIFORM_DT = 1, /* every entry of target.dt is equal (lets the fused kernels fold dt into constants) */
    HMC_FLAG_TC_FP16X2 = 2   /* tensor-core kernels (NUTS: the large-D path only; with a dense metric on the large-D path it selects the
                                split of the gradient passes only -- V, K and Lc z always use bf16x3): the caller vouches that |q - mu| stays below ~1.6e4 and that the target's
                                scale is not far below 1 (no component of interest under 2^-14), which lets the gradient
                                product use the two-part fp16 split (3 tensor passes, FP32-grade) instead of the three-part
                                bf16 split (6 passes); a trajectory that leaves the fp16 range ends in a rejection */
};

/*
 * MVN target + integrator constants, all DEVICE pointers in the compute dtype (float or double).
 * Replaces the driver closures V / dVdq (case1-script.py:39-49) and HMC_sampler.dt / inv_cov_p
 * (samplers.py:333, 352-356).  D_pad = D rounded up to a multiple of 4 (row pitch of the matrices).
 *   Ft  [D][D_pad]  transpose of the force matrix F = M^-1 P      (leap_frog, samplers.py:835-837)
 *   Pt  [D][D_pad]  transpose of the precision matrix P, or NULL when M = I (then F == P)
 *   Mit [D][D_pad]  transpose of M^-1 = inv(cov_p), or NULL when M = I       (K, samplers.py:811-817)
 *   Lct [D][D_pad]  transpose of a factor Lc with Lc Lc^T = cov_p (p = Lc z), or NULL when M = I
 *                   (p_sample, samplers.py:825-829; only used when momenta come from Philox).  Mit must be inv(Lc Lc^T): the
 *                   large-D path relies on it for K(p0) = p0^T M^-1 p0 / 2 = z^T z / 2 of a Philox draw (no product)
 *   mu  [D_pad]     target mean q0
 *   dt  [D_pad]     per-dimension time step (a scalar dt is broadcast by the host; samplers.py:333)
 *   v_const         0.5 (D ln 2pi + ln det cov0), the constant of -logpdf (utils.py:213-218)
 */
typedef struct hmc_target {
    int32_t D;
    int32_t D_pad;
    const void* Ft;
    const void* Pt;
    const void* Mit;
    const void* Lct;
    const void* mu;
    const void* dt;
    double v_const;
} hmc_target;

/*
 * HMC_sampler.leap_frog (samplers.py:831-839) for B independent (p, q) pairs, rows of [B][D] arrays in `dtype`:
 *   p' = p - dt F (q - mu) / 2,  q' = q + dt p',  p'' = p' - dt F (q' - mu) / 2      (F = M^-1 P; q moves by p, not M^-1 p: quirk Q9)
 * `nsteps` >= 1 repetitions.  The public primitive of the path (the samplers fuse it into their trajectory kernels, one gradient
 * per step); D <= 1024 (hmc_leap_frog_bigd: float32 up to D = 8192).
 */
int hmc_leap_frog(int32_t dtype, const hmc_target* target, int64_t B, const void* p_old, const void* q_old, void* p_new, void* q_new,
                  int32_t nsteps, void* cuda_stream);

/*
 * hmc_leap_frog for float32 and any 128 <= D <= 8192, on the tcgen05 GEMM of the large-D path (csrc/bigd_primitives.cu): any
 * metric (only target.Ft, mu and dt enter), B rows of [B][D] arrays.  The nsteps steps run as nsteps + 1 gradient products: the
 * closing half kick of a step and the opening half kick of the next are merged into one full kick, so with nsteps > 1 the result
 * differs from nsteps separate calls in the last bits.  flags: HMC_FLAG_TC_FP16X2 selects the two-part fp16 split (default: the
 * three-part bf16 split), with the same range condition as for the samplers.  `workspace`: device scratch of at least
 * hmc_leap_frog_workspace_bytes(target, B, flags) bytes, 1024-byte aligned; a missing or short one is HMC_E_BADARG.  float64 or D
 * outside [128, 8192] is HMC_E_UNSUPPORTED.  The size is non-zero exactly for 128 <= D <= 8192 and 1 <= B <= 2^30 (it depends on
 * target->D and B only and covers both splits); 0 otherwise.
 */
int64_t hmc_leap_frog_workspace_bytes(const hmc_target* target, int64_t B, int32_t flags);
int hmc_leap_frog_bigd(int32_t dtype, const hmc_target* target, int64_t B, const void* p_old, const void* q_old, void* p_new,
                       void* q_new, int32_t nsteps, int32_t flags, void* workspace, int64_t workspace_bytes, void* cuda_stream);

/*
 * Random-trajectory-length sampler: replaces HMC_sampler.gen_sample_random (samplers.py:387-491) together
 * with K / E / p_sample / leap_frog (samplers.py:811-839) for chains [0, Nchain) of this device, global
 * chain ids chain_id0 + m (the Philox streams are keyed by GLOBAL chain id, so results do not depend on how
 * chains are sharded over GPUs).  Iterations (iter_begin, iter_end] are run; iter_begin = 0 starts from
 * q_start and also performs the chain initialisation of samplers.py:413-420, iter_begin > 0 resumes from
 * state_q / state_eprev written by the previous call ("one launch per iteration block").
 */
typedef struct hmc_random_args {
    int32_t dtype;          /* HMC_F32 | HMC_F64 */
    int32_t kernel;         /* HMC_KERNEL_* */
    int32_t Nchain;         /* chains on this device */
    int32_t flags;          /* HMC_FLAG_* */
    int64_t chain_id0;      /* global id of local chain 0 */
    int32_t Niter;          /* total iterations of the run (samplers.py:26) */
    int32_t iter_begin;     /* iterations already done */
    int32_t iter_end;       /* run up to and including this iteration (<= Niter) */
    int32_t warm_up_num;    /* samplers.py:28 */
    int32_t thin_rate;      /* samplers.py:27 */
    int32_t L_low;          /* trajectory length drawn from {L_low .. L_high-1} (samplers.py:441, upper bound exclusive) */
    int32_t L_high;
    int32_t N_save_chain0;  /* chain-0 trajectory capture for make_movie (samplers.py:397-400, 442-452) */
    uint64_t seed;          /* Philox key */
    hmc_target target;
    const void* q_start;    /* [Nchain][D] compute dtype (used when iter_begin == 0) */
    /* injected draws (the reference's own), all float64/int32, or NULL to use Philox: */
    const double* p_tape;   /* [Nchain][Niter+1][D]  momenta in consumption order (samplers.py:415, 431) */
    const int32_t* L_tape;  /* [Nchain][Niter]       (samplers.py:441) */
    const double* u_tape;   /* [Nchain][Niter]       (samplers.py:461) */
    /* outputs */
    void* q_chain;          /* [Nchain][L_chain][D] compute dtype */
    double* E_chain;        /* [Nchain][L_chain] */
    double* dE_chain;       /* [Nchain][L_chain] */
    void* state_q;          /* [Nchain][D] compute dtype: chain position after iter_end (in: position after iter_begin) */
    void* state_g;          /* scratch of at least max(Nchain*D, Nchain + 64) elements of the compute dtype (work queue head, per-chain
                               progress words; int32 word [16 + Nchain] is raised by the tensor-core kernel when HMC_FLAG_TC_FP16X2
                               was set and a start point has |q - mu| >= 16384: repeat the run without the flag); may be NULL
                               for the generic kernel */
    double* state_eprev;    /* [Nchain] E_previous (samplers.py:420, 460) */
    unsigned long long* counters; /* [4]: accepted during warm-up, accepted after, sum L, sum L^2 (atomically added) */
    /* chain-0 trace (only written by the device that owns global chain 0), or NULL: */
    double* phi_q;          /* [N_save_chain0][L_high][2]  rows 0..L of iteration i at [i-1] (samplers.py:444-452) */
    int32_t* phi_len;       /* [N_save_chain0]  L+1 */
    int32_t* decision_chain;/* [N_save_chain0+1] (samplers.py:399, 464) */
    int32_t store_ring;     /* 0: q_chain / E_chain / dE_chain hold all L_chain stored samples per chain (the reference's layout).
                               R > 0: they hold R rows per chain and stored sample j goes to row j % R -- a ring of the last R
                               stored samples for runs whose full stream does not fit (streaming / benchmark use) */
    int32_t reserved0;
    void* workspace;        /* scratch of hmc_random_workspace_bytes(args) bytes for HMC_KERNEL_BIGD (1024-byte aligned); NULL otherwise */
    int64_t workspace_bytes;
} hmc_random_args;

int hmc_random_run(const hmc_random_args* args, void* cuda_stream);
/* bytes of hmc_random_args.workspace the large-D path needs for this configuration: non-zero exactly for the runs it covers
   (float32; identity metric and 128 <= D <= 8192, or a dense metric -- Pt, Mit and Lct all given -- and 1024 < D <= 8192), whatever
   kernel is asked for; 0 otherwise.  Depends on Nchain, D and whether the metric is dense.  A dense metric adds the products'
   operands and results: 9 Ncp Dp x 2 B of split rows, 9 Dp^2 x 2 B of split matrices, 3 Ncp Dp x 4 B of products (Ncp = Nchain
   rounded up to 512, Dp = D rounded up to 32): about 33 GB on top of the identity size's ~26 GB at 131,072 chains and D = 8192. */
int64_t hmc_random_workspace_bytes(const hmc_random_args* args);

/*
 * NUTS sampler: replaces HMC_sampler.gen_sample_NUTS (samplers.py:495-808) and the index helpers
 * find_next / retrieve_save_index / check_points / release_fast (utils.py:222-304, 367-385; closed forms).
 * Draw order per chain: one momentum per iteration; one direction coin per doubling (samplers.py:608); one
 * uniform per surviving inner step (samplers.py:748) and one per completed doubling (samplers.py:773).
 * Kernels: the generic one (D <= 256, float or double, any metric), the tensor-core one (D = 100, float32, identity metric,
 * d_max <= 12), the large-D path (any 128 <= D <= 8192, float32, identity metric; needs `workspace`).
 * store_ring: as hmc_random_args.store_ring (0: L_chain rows per chain; R > 0: q_chain / E_chain / dE_chain hold R rows per
 * chain and stored index j goes to row j % R), served by the large-D path only.  With store_ring > 0, AUTO takes the large-D path
 * whenever `workspace` is given and the path covers the run (any 128 <= D <= 8192, not only D > 256); an explicit generic or tc
 * kernel, or an AUTO run the path does not cover, is HMC_E_UNSUPPORTED.  store_ring < 0 is HMC_E_BADARG.
 */
typedef struct hmc_nuts_args {
    int32_t dtype;
    int32_t kernel;
    int32_t Nchain;
    int32_t d_max;          /* samplers.py:306, 348 */
    int64_t chain_id0;
    int32_t Niter;
    int32_t iter_begin;
    int32_t iter_end;
    int32_t warm_up_num;
    int32_t thin_rate;
    int32_t on_dmax;        /* 0 = "assert", 1 = "stop".  In both modes a chain that needs depth > d_max keeps its live point, sets
                               bit 0 of status[] and counts in counters[3]; the call is asynchronous, so the CALLER turns
                               counters[3] > 0 into the reference's failure (samplers.py:596-598) when on_dmax == 0 -- the Python
                               mirror raises AssertionError; HMC_E_DMAX is the code reserved for wrappers that synchronise */
    uint64_t seed;
    hmc_target target;
    const void* q_start;
    const double* p_tape;   /* [Nchain][Niter+1][D] or NULL */
    const int32_t* dir_tape;/* [Nchain][tape_dir_stride]  direction coins in consumption order, or NULL */
    const double* u_tape;   /* [Nchain][tape_u_stride]    uniforms in consumption order, or NULL */
    int32_t tape_dir_stride;
    int32_t tape_u_stride;
    void* q_chain;
    double* E_chain;
    double* dE_chain;
    void* state_q;
    double* state_eprev;
    void* scratch;          /* [Nchain + 128][2*(d_max+1)+7][D_pad] compute dtype, zeroed before the first launch of a run: check-point
                               stack (q,p), live and boundary points, cursors (row blocks by chain; the tensor-core kernel uses them by
                               resident slot, hence the 128 extra) */
    unsigned long long* counters; /* [4]: leapfrog steps, doublings, energy-instability rejections, d_max hits */
    int32_t* status;        /* [Nchain] bit0: d_max exceeded; may be NULL */
    int64_t* n_leapfrog;    /* [Nchain] leapfrog steps per chain (accumulated); may be NULL */
    int32_t flags;          /* HMC_FLAG_TC_FP16X2 selects the two-part fp16 split on the large-D path (default: bf16x3) */
    int32_t store_ring;     /* 0: the reference layout (L_chain rows per chain); R > 0: a ring of the last R stored samples per chain
                               (large-D path only, see above) */
    void* workspace;        /* scratch of hmc_nuts_workspace_bytes(args) bytes for HMC_KERNEL_BIGD (1024-byte aligned); NULL otherwise */
    int64_t workspace_bytes;
} hmc_nuts_args;

int hmc_nuts_run(const hmc_nuts_args* args, void* cuda_stream);
/* bytes of hmc_nuts_args.workspace the large-D path needs for this configuration: non-zero exactly for the runs it covers
   (float32, identity metric, 128 <= D <= 8192), whatever kernel is asked for; 0 otherwise.  Depends on Nchain and D only. */
int64_t hmc_nuts_workspace_bytes(const hmc_nuts_args* args);

/*
 * Diagnostics: replace utils.convergence_stats / utils.variogram (utils.py:77-179) as two HBM-bound
 * reductions over the chain-major sample stream.  `q` points at the first USED sample of local chain 0
 * (the Python mirror drops stored index 0 as samplers.py:61 does), `stride_chain` = elements between
 * consecutive chains (L_chain * D), `n` = samples per half chain after the odd-length drop (utils.py:96-102);
 * split chain 2m is samples [0,n), 2m+1 is [n,2n) of chain m.
 *
 *   hmc_diag_moments : per split chain mean and ddof=1 standard deviation (utils.py:107-118), reduced to
 *                      per-device partial sums  out[0][D] = sum_j std_j, out[1][D] = sum_j (mean_j - c),
 *                      out[2][D] = sum_j (mean_j - c)^2  (float64), and the shift out[3][D] = c = the first sample of
 *                      this device's first chain: the between-chain sum of squares then does not cancel when the chains
 *                      sit far from zero.  Devices are combined on the host from their (count, sums, shift) records
 *                      (one all-gather; pairwise variance update).
 *   hmc_diag_variogram : out[t - lag0][D] = sum over split chains and i of (x[i+t]-x[i])^2 for
 *                      t in [lag0, lag0+nlags), nlags <= 32  (utils.py:161-179, numerator only; float64).
 * Both zero `out` first (on the stream) and then accumulate with float64 atomics.
 */
int hmc_diag_moments(int32_t dtype, const void* q, int64_t Nchain, int64_t n, int32_t D, int64_t stride_chain,
                     double* out4xD, void* cuda_stream);
int hmc_diag_variogram(int32_t dtype, const void* q, int64_t Nchain, int64_t n, int32_t D, int64_t stride_chain,
                       int32_t lag0, int32_t nlags, double* out_nlags_x_D, void* cuda_stream);
/* Short series (n <= 32): both reductions above in ONE pass over the samples (every value is read once and kept in
 * registers); out_lags[t - 1][D] for t in [1, nlags], nlags <= 31.  Same outputs as hmc_diag_moments followed by
 * hmc_diag_variogram(lag0 = 1).  float32 streams with an even D take packed (two dimensions per thread, FADD2 / FFMA2)
 * kernels; any D is accepted (dimensions are processed in tiles). */
int hmc_diag_short_series(int32_t dtype, const void* q, int64_t Nchain, int64_t n, int32_t D, int64_t stride_chain,
                          int32_t nlags, double* out4xD, double* out_lags, void* cuda_stream);

/* Every lag at once (float32 streams, 32 < n <= 512, D % 4 == 0, 16-byte aligned rows; anything else returns
 * HMC_E_UNSUPPORTED and the caller stays with hmc_diag_variogram): out[t - 1][D] for t in [1, nlags], nlags <= n - 1, the same
 * numerators as hmc_diag_variogram, from ONE pass over the samples -- a 1024-point FFT per (chain, dimension) carrying both
 * split chains as real and imaginary part, power spectra summed over chains in float64, the cosine transform and the edge
 * sums of squares finished by a small float64 kernel (csrc/diag_fft.cu; utils.py:141-152 calls variogram once per lag).
 * `workspace`: device scratch of hmc_diag_variogram_all_workspace_bytes(n, D) bytes, zeroed by the call. */
int64_t hmc_diag_variogram_all_workspace_bytes(int64_t n, int32_t D);
int hmc_diag_variogram_all(int32_t dtype, const void* q, int64_t Nchain, int64_t n, int32_t D, int64_t stride_chain,
                           int32_t nlags, double* out_nlags_x_D, void* workspace, int64_t workspace_bytes, void* cuda_stream);

/*
 * Streamed diagnostics (csrc/diag_stream.cu): the partial sums of hmc_diag_moments and hmc_diag_variogram for the lags 1..T, folded
 * in block by block from a ring q_ring [Nchain][R][D] (compute dtype; stored index j of chain c in row j % R, as
 * hmc_random_args.store_ring = R writes it), so that R_q and n_eff_q of a run need only the last R stored samples per chain on the
 * device.  The split is the one above: with n = (L_chain - 1) / 2, split chain 2m is stored indices [1, n] of chain m and 2m+1 is
 * [n+1, 2n] (index 0 and, for an odd L_chain - 1, the last index are not used).
 *
 *   hmc_diag_stream_update : hands over stored indices [j0, j1) of every local chain; every index must be final (its thin window
 *                            closed) and rows [j0 - T, j1) must still be in the ring, so R >= T + (j1 - j0).  Calls of one run cover
 *                            [0, L_chain) in order; the call with j0 = 0 zeroes the accumulated sums.  Each index is added to its
 *                            split chain's float64 shifted sum and sum of squares (state per chain and dimension); at index n or 2n the
 *                            split chain's mean and ddof = 1 std are folded into the moment rows.  Every pair (i - t, i) with i in
 *                            [j0, j1), 1 <= t <= T and both in one split chain is added to lag t: per chain over at most 64 new indices
 *                            in the stream's precision (as the windowed kernel does over a whole split chain), then in float64.
 *   hmc_diag_stream_finish : out4xD [4][D] = the rows hmc_diag_moments writes (sums of std_j, mean_j - c, (mean_j - c)^2, and c = the
 *                            first used sample of local chain 0), out_lags [T][D] = the numerators hmc_diag_variogram writes for lags
 *                            1..T.  Copies on the stream; the workspace is left as it was.
 * `workspace`: device scratch of hmc_diag_stream_workspace_bytes(Nchain, D, T) = 8 D (4 + T + 3 Nchain) bytes, kept by the caller
 * for the whole run (the library keeps nothing between calls).  The size is non-zero exactly for Nchain >= 1, 1 <= D <= 8192 and
 * 1 <= T <= 2^20.  HMC_E_BADARG: R < T + (j1 - j0), T < 1 or T > n - 1, j0 / j1 outside 0 <= j0 <= j1 <= L_chain, D outside
 * [1, 8192], a NULL ring, a missing or short workspace.
 */
int64_t hmc_diag_stream_workspace_bytes(int64_t Nchain, int32_t D, int32_t T);
int hmc_diag_stream_update(int32_t dtype, const void* q_ring, int64_t Nchain, int32_t D, int32_t R, int64_t L_chain, int32_t T,
                           int64_t j0, int64_t j1, void* workspace, int64_t workspace_bytes, void* cuda_stream);
int hmc_diag_stream_finish(const void* workspace, int64_t workspace_bytes, int32_t D, int32_t T, double* out4xD, double* out_lags,
                           void* cuda_stream);

/*
 * Start points on the device: replaces utils.start_pts (utils.py:204-209, np.random.multivariate_normal(q0, cov0, size)).
 * out[m][:] = q0 + Lc z_m with z_m ~ N(0, I) from Philox keyed by (seed, chain_id0 + m), so the points do not depend on
 * how chains are sharded.  q0 [D], Lc [D][D] (row-major lower-triangular factor, Lc Lc^T = cov0) or NULL, sd [D]
 * (used when Lc is NULL: diagonal cov0, sd = sqrt(diag)) are float64 DEVICE arrays; out [Nchain][D] in `dtype`.
 */
int hmc_start_pts(int32_t dtype, uint64_t seed, int64_t chain_id0, int64_t Nchain, int32_t D, const double* q0,
                  const double* Lc, const double* sd, void* out, void* cuda_stream);

/*
 * q_m = q0 + Lc z_m on the tensor cores (csrc/bigd_primitives.cu), float32 out, 128 <= D <= 8192: the same Philox normals as
 * hmc_start_pts (seed, global chain id, HMC_STREAM_START, full-precision Box-Muller), so for the same (seed, chain_id0) the two
 * entry points draw the same z.  Lc: row-major lower-triangular float64 [D][D] (the lower triangle is read), rounded to float32
 * and split into three bf16 parts, fp32 accumulation; or NULL with sd [D] (diagonal cov0: elementwise, no GEMM, the same rows as
 * hmc_start_pts).  `workspace` (used with Lc only): device scratch of at least hmc_start_pts_workspace_bytes(Nchain, D) bytes,
 * 1024-byte aligned; a missing or short one is HMC_E_BADARG.  float64 or D outside [128, 8192] is HMC_E_UNSUPPORTED.  The size
 * is non-zero exactly for 128 <= D <= 8192 and 1 <= Nchain <= 2^30, 0 otherwise.
 */
int64_t hmc_start_pts_workspace_bytes(int64_t Nchain, int32_t D);
int hmc_start_pts_bigd(int32_t dtype, uint64_t seed, int64_t chain_id0, int64_t Nchain, int32_t D, const double* q0,
                       const double* Lc, const double* sd, void* out, void* workspace, int64_t workspace_bytes, void* cuda_stream);

/*
 * Sample summaries: the inputs of sampler.plot_samples (samplers.py:84-113, 160-186, 209-250) as HBM-bound reductions over
 * the device-resident outputs, so that the host never materialises q_chain (26 GB at 65,536 chains).
 *   hmc_summary_moments : out[0][D] = sum, out[1][D] = sum of squares over chains [0, Nchain) x samples [0, nsamp) of the
 *                         rows at q + chain * stride_chain + sample * pitch (float64 partial sums per device).
 *   hmc_summary_hist    : np.histogram of v = x - shift on the given bin edges (edges [nbins + 1] float64 device, ascending;
 *                         last bin closed on the right); counts [nbins + 2]: the bins, then #below, #above.  The series is
 *                         x[chain * stride_chain + sample * stride_sample] (a column of q_chain, or E_chain / dE_chain).
 *   hmc_summary_select  : one pass of a radix select over the order-preserving integer keys of the series (32-bit keys for
 *                         float32, 64-bit for float64): out[2048] += histogram of digit (key >> digit_shift) & (2^digit_bits - 1)
 *                         over the elements with key >> prefix_shift == prefix (prefix_shift = 64: all elements).  The host walks
 *                         the digits from the top to the k-th smallest value (np.percentile's order statistics).
 * Counts are per device; sum them over ranks (they are plain sums) for a sharded run.
 */
int hmc_summary_moments(int32_t dtype, const void* q, int64_t Nchain, int64_t nsamp, int32_t D, int64_t pitch,
                        int64_t stride_chain, double* out2xD, void* cuda_stream);
int hmc_summary_hist(int32_t dtype, const void* x, int64_t Nchain, int64_t nsamp, int64_t stride_sample,
                     int64_t stride_chain, double shift, const double* edges, int32_t nbins,
                     unsigned long long* out_counts, void* cuda_stream);
int hmc_summary_select(int32_t dtype, const void* x, int64_t Nchain, int64_t nsamp, int64_t stride_sample,
                       int64_t stride_chain, uint64_t prefix, int32_t prefix_shift, int32_t digit_shift,
                       int32_t digit_bits, unsigned long long* out_hist2048, void* cuda_stream);

/* Debug/test aid: the draws the kernels make for (seed, global chain id, iteration): 4*ceil(D/4) normals
 * (float32 Box-Muller widened to float64), the trajectory length and the acceptance uniform.  Lets the
 * oracle be fed exactly the device's own Philox draws.  out_p [Nchain][Niter+1][D], out_L/out_u [Nchain][Niter]. */
int hmc_philox_draws(uint64_t seed, int64_t chain_id0, int32_t Nchain, int32_t Niter, int32_t D,
                     int32_t L_low, int32_t L_high, double* out_p, int32_t* out_L, double* out_u,
                     void* cuda_stream);

/* FP32 FFMA roofline probe (SURVEY 8d: "measure an FFMA microbenchmark on the box"): runs a dependent-chain
 * free FFMA2 loop on every SM and returns achieved FLOP/s in *out_flops (host pointer). */
int hmc_ffma_peak(double* out_flops_host, int32_t use_ffma2, void* cuda_stream);

int hmc_version(void);
const char* hmc_last_error_string(void);

#ifdef __cplusplus
}
#endif
#endif /* HMC_B200_H */
