/*
 * kissmcmc_cuda.h -- C-ABI of libkissmcmc_cuda.so, the B200 (sm_100a) implementation of
 * KissMCMC.jl's emcee stretch-move hot path.
 *
 * The reference (KissMCMC.jl v0.2.2) has no FFI: its boundary is three exported Julia
 * functions (src/KissMCMC.jl:8) and the call pdf(theta) to a user closure
 * (src/samplers.jl:257, :209, :334-336).  This header is the interface a
 * `KissMCMC.CUDABackend` Julia module binds with `ccall` (see INTEGRATION.md) and that the
 * Python host mirror (kissmcmc.jl_b200/) binds with ctypes.  Each entry point cites the
 * reference code it replaces.
 *
 * Conventions
 *   - every function returns int32 status, 0 = ok; kmc_last_error() returns a thread-local
 *     message for the last non-zero status.  No exceptions, no callbacks into the host.
 *   - plain pointers and sizes only.  The CALLER owns every host buffer and must keep it
 *     alive for the duration of the call (Julia: GC.@preserve).
 *   - opaque handles own all device memory.  A sampler handle is used by one host thread at a
 *     time.
 *   - walker arrays cross the ABI as dense FP64 `d x nw` column-major (Julia
 *     `reduce(hcat, theta0s)`), which is C row-major [nw][d].  Chains come back as
 *     `d x ns x nw` column-major = C [nw][ns][d] -- the (ntheta, nsamples, nchains) layout of
 *     the reference's int_acorr (src/analysis.jl:143); log-densities as `ns x nw` = C [nw][ns].
 *   - walker indices are 0-based across the ABI (the Julia wrapper subtracts 1).
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails.
 */
#ifndef KISSMCMC_CUDA_H
#define KISSMCMC_CUDA_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KMC_OK 0
#define KMC_ERR_INVALID 1     /* bad argument (the reference's @assert, src/samplers.jl:200-205) */
#define KMC_ERR_CUDA 2        /* CUDA runtime error or no device */
#define KMC_ERR_UNSUPPORTED 3 /* density / dimension combination with no kernel */
#define KMC_ERR_STATE 4       /* call not valid in the handle's current state */

#define KMC_MODE_PHILOX 0 /* free-running, counter-based Philox4x32-10 draws */
#define KMC_MODE_REPLAY 1 /* partner / z / u uploaded by the caller */

/* How the shards of one ensemble see each other's rows (kmc_emcee_opts.exchange, sharded samplers only). */
#define KMC_EXCHANGE_REPLICA 0 /* every shard holds the FULL ensemble's positions; the caller exchanges the updated
                                  half between half-steps (all-gather), or the legacy pull mode (kmc_emcee_set_peers) */
#define KMC_EXCHANGE_PUSH 1    /* every shard holds ONLY its rows plus a receive ring; the owners of the passive half
                                  push the partner rows every peer will ask for (kmc_emcee_window_*, kmc_multi_*) */

/* kmc_emcee_create_multi modes */
#define KMC_MULTI_SHARDED 0     /* ONE ensemble sharded by walker index over the devices (push exchange) */
#define KMC_MULTI_INDEPENDENT 1 /* one independent ensemble per device, no communication */

typedef struct kmc_density_s *kmc_density_t;
typedef struct kmc_sampler_s *kmc_sampler_t;
typedef struct kmc_multi_s *kmc_multi_t;

typedef struct kmc_emcee_opts {
    int64_t niter_walker;   /* niter / nwalkers    (src/samplers.jl:203) */
    int64_t nburnin_walker; /* nburnin / nwalkers  (src/samplers.jl:204) */
    int64_t nthin;          /* store every nthin-th iteration (:268) */
    double a_scale;         /* stretch scale a > 1 (:200) */
    uint64_t seed;          /* Philox key */
    int32_t mode;           /* KMC_MODE_* */
    int32_t device;         /* CUDA device ordinal */
    int64_t walker_id_base; /* added to local walker indices in the Philox counter, so shards of
                               one ensemble (or independent ensembles) draw distinct streams */
    int32_t launch_mode;    /* 0 = persistent kernel, grid barrier between half-steps (default);
                               1 = one launch per half-step */
    int32_t exchange;       /* KMC_EXCHANGE_* (sharded samplers; 0 otherwise) */
    /* Sharded ensemble (one ensemble over several GPUs, SURVEY.md section 8e): this sampler holds
     * the FULL ensemble's positions but updates only positions [shard_begin, shard_begin +
     * shard_count) of each half; the caller makes the updated slices of the other shards visible
     * between half-steps (all-gather).  shard_count = 0: the whole half (single GPU).  Draws are
     * keyed by the global walker index, so a sharded run reproduces the single-GPU run exactly. */
    int64_t shard_begin;
    int64_t shard_count;
    /* KMC_EXCHANGE_PUSH tuning; 0 = the library's choice.  push_chunk: active walkers per push (the unit of the
     * "rows have landed" flags; <= 1024; default min(1024, 256 * ranks)), push_cap: rows per receive-ring slot (<= 384;
     * rows past it are read from the owner directly; default mean + 8 sigma of the hit count), push_lag: chunks by
     * which the updates trail the pushes in the ordered task hand-out (default 5/16 of the chunks); -1 selects the
     * adaptive hand-out (an update is taken when its rows are seen landed, else a push). */
    int32_t push_chunk;
    int32_t push_cap;
    int32_t push_lag;
    int32_t reserved;
} kmc_emcee_opts;

/* Library / device ------------------------------------------------------------------- */
int32_t kmc_version(void);
const char *kmc_last_error(void);
int32_t kmc_device_count(int32_t *count);
/* Device buffers of destroyed samplers are cached for reuse; this releases them to the driver. */
int32_t kmc_trim(void);

/* Log-density plugin registry: replaces the user closure `pdf` (src/samplers.jl:257,:209).
 *   "exponential"  README.md:15             params: none; any d <= 4096 (fused kernels for d in {1..6, 8, 10, 12, 16})
 *   "rosenbrock"   test/runtests.jl:68      params: [a, b, T] (reference: 1, 100, 20), d = 2
 *   "gaussian"     test/runtests.jl:53,61   params: [mu(d), A(d*d row-major), lognorm],
 *                                           logp = lognorm - 0.5*|A (x-mu)|^2; any d <= 4096 (fused FP64 kernels for
 *                                           d in {1..6, 8, 10, 12, 16}; batched FP64 otherwise, the matrix in shared
 *                                           memory up to d = 128 and in L2 beyond)
 *   "lognormal"    test/runtests.jl:56      params: [mu, sigma, log(sigma)+0.5*log(2pi)], d = 1
 *   "logistic"     BASELINE.json config 4   params: [prior_sigma]; data: float32 X[N][d] then y[N]; any d <= 512
 *   "gaussian_mixture"  sum_k w_k MvNormal(mu_k, Sigma_k)   params: K components of q = d + d(d+1)/2 + 1 doubles,
 *                                           each [mu_k(d), upper triangle of A_k = chol(Sigma_k^-1)^T row by row (row i
 *                                           holds j = i..d-1, diagonal > 0), c_k = log(w_k/sum w) + lognorm_k];
 *                                           logp = logsumexp_k(c_k - 0.5*|A_k (x-mu_k)|^2); d in {1..6, 8, 10, 12, 16},
 *                                           1 <= K <= Kmax(d) = floor(272/q): 90, 45, 27, 18, 12, 9, 6, 4, 2, 1 for
 *                                           d = 1, 2, 3, 4, 5, 6, 8, 10, 12, 16 (KMC_ERR_UNSUPPORTED beyond; nparams not a
 *                                           multiple of q, a non-finite value or a diagonal entry <= 0: KMC_ERR_INVALID)
 * `data` may be NULL.  params/data are copied; the caller may free them on return. */
int32_t kmc_density_create(const char *name, int32_t d, const double *params, int64_t nparams,
                           const void *data, int64_t data_bytes, int32_t device,
                           kmc_density_t *out);
int32_t kmc_density_destroy(kmc_density_t h);
/* Options: "tensor_cores" = 0/1.  Every plugin is exact FP64 by default.  1 opts in to the tcgen05 kernels, which are
 * APPROXIMATE with a stated tolerance: the dense Gaussian with 16 < d <= 128 (|logp - logp_fp64| <= 1e-5 (1 + |y|^2))
 * and logistic regression with d <= 64 and bf16-representable data, whose error grows with the size of the logits:
 * per point |logp - logp_fp64| <= u [(0.5 + 1.05 m) sum_n sum_k |theta_k x_nk| + 8.5 sum_n |theta . x_n|] + 5 u N,
 * u = 2^-24, m = ceil(d/16) (at most 13.2 u sum_n sum_k |theta_k x_nk| + 5 u N), and the sum of two points' bounds on
 * their difference.  At d = 32, N = 10^6 and theta* ~ N(0, 1/d) (mean |logit| 0.7) that is ~1.3 per point (measured:
 * a common offset of ~3e-2 that cancels in every accept test, 2e-3 on differences); with the data drawn from 16 theta*
 * (mean |logit| 11), ~13.  Returns KMC_ERR_UNSUPPORTED if the density has no tensor-core path.
 * "fused_variant" = 2/1: which fused persistent kernel the tensor-core dense Gaussian uses in
 * launch_mode 0 -- 2 (default): matrix pieces resident in TMEM; 1: matrix pieces in shared memory
 * (bit-identical to the three-kernel pipeline of launch_mode 1).
 * Info keys: "tensor_cores" (1 if the tcgen05 path will be used), "tensor_cores_available", "batched",
 * "fused_variant". */
int32_t kmc_density_set_option(kmc_density_t h, const char *key, double value);
int32_t kmc_density_get_info(kmc_density_t h, const char *key, double *value);
/* Batched log-density of nw points (host in, host out).  Used for the initial p0s
 * (src/samplers.jl:209-210) and by make_theta0s (:334-338). */
int32_t kmc_density_eval(kmc_density_t h, const double *thetas, int64_t nw, double *logp_out);

/* Sampler: _emcee, src/samplers.jl:232-293 ------------------------------------------- */
/* Uploads theta0s (never mutated, :198), checks the reference's asserts (:200-205: a_scale > 1,
 * even nwalkers, nwalkers >= d + 2), evaluates the initial log-densities (:209) and allocates
 * the thinned chain store (ns = (niter_walker - nburnin_walker) / nthin samples per walker). */
int32_t kmc_emcee_create(kmc_density_t density, const double *theta0s, int64_t nwalkers,
                         int32_t d, const kmc_emcee_opts *opts, kmc_sampler_t *out);
int32_t kmc_emcee_destroy(kmc_sampler_t s);
/* Launch on a caller-owned CUDA stream (a cudaStream_t passed as void*); NULL = the
 * sampler's own stream. */
int32_t kmc_emcee_set_stream(kmc_sampler_t s, void *cuda_stream);
/* Replay mode: draws for `niters` outer iterations starting at the sampler's current
 * iteration, each array of length niters*nwalkers indexed ((t*2 + batch)*(nwalkers/2) + i),
 * i = position of the active walker in its half (:247-252,:260).  partner = global 0-based
 * index of the passive walker, z = stretch factor, u = accept uniform. */
int32_t kmc_emcee_set_replay(kmc_sampler_t s, const int64_t *partner, const double *z,
                             const double *u, int64_t niters);
/* Advance `niters` outer iterations (niters < 0: all that remain).  Asynchronous on the
 * sampler's stream. */
int32_t kmc_emcee_run(kmc_sampler_t s, int64_t niters);
/* Advance `nhalfsteps` half-ensemble sweeps (:246-273); two per outer iteration.  A sharded
 * run alternates kmc_emcee_run_half(s, 1) with the exchange of the just-updated half. */
int32_t kmc_emcee_run_half(kmc_sampler_t s, int64_t nhalfsteps);
int32_t kmc_emcee_sync(kmc_sampler_t s);
/* Peer mode (sharded ensemble, one process per GPU on one NVLink/NVSwitch node): instead of an
 * all-gather after every half-step, each rank's persistent kernel gathers partner rows directly
 * from the owner GPU's memory and the ranks meet at a flag barrier in peer memory per half-step.
 * kmc_emcee_ipc_export writes two 64-byte CUDA IPC handles (positions, flags); the caller
 * exchanges them (e.g. torch.distributed.all_gather) and passes all ranks' handles, rank-major,
 * to kmc_emcee_set_peers.  Then every rank calls kmc_emcee_run(s, -1) concurrently, ONCE: the ranks only synchronise
 * between the half-steps of one launch, so a job split over several launches returns KMC_ERR_STATE.  Superseded by the
 * push exchange below, which has no such restriction and is faster. */
int32_t kmc_emcee_ipc_export(kmc_sampler_t s, void *handle_x, void *handle_flags);
int32_t kmc_emcee_set_peers(kmc_sampler_t s, const void *handles_x, const void *handles_flags, int32_t nranks,
                            int32_t rank);
/* Push mode (KMC_EXCHANGE_PUSH; csrc/kmc_push.cuh), one process per GPU: the sampler's positions, receive ring and
 * chunk flags live in ONE device allocation (the "window").  kmc_emcee_window_export writes its 64-byte CUDA IPC
 * handle; the caller exchanges the handles and passes all ranks' handles, rank-major, to kmc_emcee_window_attach.
 * Then every rank calls kmc_emcee_run concurrently: no collective, no cross-GPU barrier -- the owners of the passive
 * half push packed partner rows over NVLink and every consumer starts as soon as its chunk's rows have landed.
 * Replaces, across GPUs, the shared-memory read of the passive half at src/samplers.jl:255 (sweep :246-273). */
int32_t kmc_emcee_window_export(kmc_sampler_t s, void *handle);
int32_t kmc_emcee_window_attach(kmc_sampler_t s, const void *handles, int32_t nranks, int32_t rank);
/* Device pointers of the ensemble state (x: [nw][d] FP64, logp: [nw] FP64, naccept: [nw] u32),
 * valid until kmc_emcee_destroy; for stream-ordered exchanges by the caller. */
int32_t kmc_emcee_device_ptrs(kmc_sampler_t s, void **x, void **logp, void **naccept);
/* Device time of the kernels launched by the last kmc_emcee_run (CUDA events on the launch
 * stream) and how many kernels that was.  Synchronises. */
int32_t kmc_emcee_last_run_ms(kmc_sampler_t s, double *ms, int64_t *launches);
/* Accept-counter statistics of the progress display (:276-278): mean, std (n-1) and number
 * of walkers more than 2 std from the mean, reduced on the device.  Synchronises. */
int32_t kmc_emcee_progress(kmc_sampler_t s, int64_t *iters_done, double *naccept_mean,
                           double *naccept_std, int64_t *outliers);
int32_t kmc_emcee_nsamples(kmc_sampler_t s, int64_t *ns);
/* Walkers this sampler stores chains for: nwalkers, or 2*shard_count when sharded. */
int32_t kmc_emcee_nlocal(kmc_sampler_t s, int64_t *nl);
/* Results (:291-292).  thetas [nl][ns][d], logp [nl][ns], accept_ratio [nl]; any may be NULL.
 * nl = nwalkers, or 2*shard_count for a sharded sampler (its slice of half 0, then of half 1). */
int32_t kmc_emcee_copy_results(kmc_sampler_t s, double *thetas, double *logp,
                               double *accept_ratio);
/* Posterior moments of the samples stored so far (all walkers squashed, src/samplers.jl:372-428),
 * reduced on the device: mean [d], unbiased variance [d], number of samples.  Avoids copying
 * chains of 10^9+ samples to the host.  Samples stored so far: those of the iterations run, the
 * whole chain once the run is complete; an emcee iteration with one half-step left adds none.
 * KMC_ERR_STATE while none is stored (before the first run, during burn-in). */
int32_t kmc_emcee_chain_moments(kmc_sampler_t s, double *mean, double *var, int64_t *count);
/* Covariance of the same rows as kmc_emcee_chain_moments (emcee or Metropolis handle), the samples stored so far:
 * mean [d], unbiased covariance cov [d][d] (ddof = 1, row-major, symmetric), number of samples; shifted by the first
 * stored sample.  A fixed grid and a fixed-order final sum: the result's bits depend only on the stored chain.
 * d <= 128, else KMC_ERR_UNSUPPORTED; KMC_ERR_STATE while no sample is stored.  The pilot-run estimate a correlated
 * Metropolis proposal is tuned from. */
int32_t kmc_emcee_chain_covariance(kmc_sampler_t s, double *mean, double *cov, int64_t *count);
/* Current ensemble: theta [nw][d], logp [nw], naccept [nw]; any may be NULL. */
int32_t kmc_emcee_copy_state(kmc_sampler_t s, double *theta, double *logp, int64_t *naccept);


/* The callers either side of the sampler, on the device ------------------------------ */
/* g-distribution helpers (src/samplers.jl:223-230).  g_pdf (:224; test-only in the reference, test/emcee.jl:2-14) and
 * cdf_g_inv (:227) are evaluated on the host with the reference's operation order; kmc_sample_g (:230) draws n values
 * of z on the device through the sampler's own draw path (Philox uniform -> cdf_g_inv). */
int32_t kmc_g_pdf(const double *z, int64_t n, double a_scale, double *out);
int32_t kmc_cdf_g_inv(const double *u, int64_t n, double a_scale, double *out);
int32_t kmc_sample_g(double a_scale, uint64_t seed, int64_t n, int32_t device, double *out);
/* Device-side squash_walkers (src/samplers.jl:372-428) of the sampler's stored chains: optional drop of the walkers
 * with accept_ratio <= median - drop_fact*std (:379-393; median and std (n-1) from exact integer statistics of the
 * accept counters), walker-major concatenation of the kept walkers (:398-399) or, with order != 0, the time-major order
 * of the stable sortperm at :415-426.  thetas [nkept*ns][d] and logp [nkept*ns] may be NULL (then only the counts and
 * statistics are returned: call once to size the buffers).  accept_mean = mean(accept_ratio[kept]) (:427). */
int32_t kmc_emcee_squash(kmc_sampler_t s, int32_t drop_low_accept_ratio, double drop_fact, int32_t order,
                         double *thetas, double *logp, int64_t *nkept, double *accept_mean, double *accept_median,
                         double *accept_std);
/* Device-side make_theta0s (src/samplers.jl:311-349): Gaussian ball theta0 .+ randn(d) .* ball_radius (:328-332) with
 * counter-based Philox / Box-Muller normals, rejection of points whose plugin log-density is not > -Inf (:338), the
 * reference's loop semantics (cumulative radius halving :326, silent skip of a walker that exhausts every try).  All
 * pending walkers are tried at once.  out [nwalkers][d] receives the nfound (<= nwalkers) points in walker order.
 * kmc_ball_randn returns the normals the device uses for walkers [walker0, walker0 + n), halving step k, try j
 * (1-based like the reference loops) -- what a replay of the reference loop needs to reproduce the result. */
int32_t kmc_make_theta0s(kmc_density_t density, const double *theta0, const double *ball_radius, int64_t nwalkers,
                         int32_t ball_radius_halfing_steps, int32_t ntries, uint64_t seed, double *out,
                         int64_t *nfound);
int32_t kmc_ball_randn(uint64_t seed, int64_t walker0, int64_t nwalkers, int32_t k, int32_t j, int32_t d,
                       int32_t device, double *out);

/* Metropolis: batched independent random-walk chains, the reference's `metropolis` (src/samplers.jl:9-128) ---------
 * One kmc_sampler_t holds nchains independent chains (theta0s [nchains][d], deep-copied; p0 = pdf(theta0) evaluated on
 * the device, no error if it is -Inf).  The user closure sample_ppdf becomes a symmetric Gaussian random walk,
 * theta1 = theta0 .+ sigma .* n with n ~ N(0, I) (mul, then add): sigma [nsigma] with nsigma = 1 (scalar) or d, finite
 * and > 0.  Accept iff p1 - p0 > log(u) (:103; strict, FP64, NaN rejects).  The kmc_emcee_opts are reused as is:
 * niter_walker = niter and nburnin_walker = nburnin PER CHAIN, nthin, seed, mode, device, walker_id_base = id of chain 0
 * (ids must stay below 2^32); a_scale is not read; launch_mode, exchange, shard_* and push_* must be 0.
 * ns = (niter - nburnin) / nthin samples per chain, accept_ratio = naccept / (niter - nburnin), accepts counted after
 * burn-in.  Draws of step t = ni + nburnin - 1 (0-based) of chain id c are a pure function of (seed, c, t): Philox4x32-10
 * with counter (c, t lo, t hi, 0x4D48 << 16 | pair) -> Box-Muller normals 2 pair, 2 pair + 1 from words r0, r1; the
 * accept uniform ((r2 & 0xFFFF) << 32 | r3) * 2^-48 of pair 0.  So chain c is the same chain whatever the batch size.
 * These take a Metropolis handle and mean the same as for emcee: kmc_emcee_run (niters = steps), _sync, _destroy,
 * _set_stream, _nsamples, _nlocal (= nchains), _device_ptrs, _copy_results, _copy_state, _chain_moments, _squash,
 * _progress, _last_run_ms.  kmc_emcee_set_replay, _run_half, _ipc_export, _set_peers and _window_* return
 * KMC_ERR_STATE on it. */
int32_t kmc_metropolis_create(kmc_density_t density, const double *theta0s, int64_t nchains, int32_t d,
                              const double *sigma, int64_t nsigma, const kmc_emcee_opts *opts, kmc_sampler_t *out);
/* The same with a correlated Gaussian random walk (the reference's closure drawing from MvNormal): chol [d][d] is
 * the lower-triangular Cholesky factor L of the proposal covariance, row-major (Julia's column-major
 * cholesky(Sigma).U has this layout).  With z the step's normals (the same draws as above): for i = 0 .. d-1,
 * s = 0.0; s = s + L[i][j] * z[j] for j = 0 .. i ascending (mul, then add, never fused); theta1[i] = theta0[i] + s.
 * L = diag(sigma) gives the chains of kmc_metropolis_create bit for bit.  KMC_ERR_INVALID as kmc_metropolis_create,
 * and if an entry is not finite, a diagonal entry is <= 0 or an entry above the diagonal is non-zero.  The handle is
 * a Metropolis handle like any other; kmc_metropolis_set_replay takes the normals z. */
int32_t kmc_metropolis_create_chol(kmc_density_t density, const double *theta0s, int64_t nchains, int32_t d,
                                   const double *chol, const kmc_emcee_opts *opts, kmc_sampler_t *out);
/* Replay mode: normals [niters][nchains][d] and accept uniforms [niters][nchains] for the steps from the sampler's
 * current step on (sample_ppdf and the rand() of :103).  KMC_ERR_STATE on an emcee handle. */
int32_t kmc_metropolis_set_replay(kmc_sampler_t s, const double *normals, const double *u, int64_t niters);
/* The normals [niters][nchains][d] and uniforms [niters][nchains] the device draws for chain ids
 * [chain0, chain0 + nchains) at steps [t0, t0 + niters). */
int32_t kmc_metropolis_draws(uint64_t seed, int64_t chain0, int64_t nchains, int64_t t0, int64_t niters, int32_t d,
                             int32_t device, double *normals, double *u);

/* Library-owned multi-GPU (single process, SURVEY.md section 8b: opts {devices[], sharded / independent}) -------- */
/* One emcee run over `ndev` devices of this process.  devices[] lists CUDA ordinals (an ordinal may repeat: its
 * sub-samplers then share that GPU, which is how the sharded path is tested on one GPU).  densities[] holds one plugin
 * handle per entry of devices[] (fused plugins keep no device memory, so the same handle may be repeated).
 *   KMC_MULTI_SHARDED      theta0s is ONE ensemble [nwalkers][d]; entry r updates positions [r*S, (r+1)*S) of each half,
 *                          S = nwalkers/2/ndev, with the push exchange over peer memory (cudaDeviceEnablePeerAccess);
 *                          results are the reference 3 arrays for the WHOLE ensemble in global walker order,
 *                          bit-identical to the single-GPU run.  Parallel region replaced: src/samplers.jl:246-273.
 *   KMC_MULTI_INDEPENDENT  theta0s is [ndev][nwalkers][d]: ndev ensembles, ensemble r with walker ids r*nwalkers..,
 *                          no communication; results are concatenated ensemble-major ([ndev*nwalkers] walkers).
 * opts->device / shard_* / exchange / walker_id_base are filled in by the library. */
int32_t kmc_emcee_create_multi(const kmc_density_t *densities, const double *theta0s, int64_t nwalkers, int32_t d,
                               const kmc_emcee_opts *opts, const int32_t *devices, int32_t ndev, int32_t mode,
                               kmc_multi_t *out);
int32_t kmc_multi_destroy(kmc_multi_t m);
/* Advance every device `niters` outer iterations (< 0: all that remain); asynchronous. */
int32_t kmc_multi_run(kmc_multi_t m, int64_t niters);
int32_t kmc_multi_sync(kmc_multi_t m);
/* Device time of the last kmc_multi_run: the maximum over the devices' kernels.  Synchronises. */
int32_t kmc_multi_last_run_ms(kmc_multi_t m, double *ms);
/* Samples per walker and walkers in the result arrays (nwalkers, or ndev*nwalkers for independent ensembles). */
int32_t kmc_multi_shape(kmc_multi_t m, int64_t *ns, int64_t *nwalkers_out);
/* thetas [nw_out][ns][d], logp [nw_out][ns], accept_ratio [nw_out]; any may be NULL. */
int32_t kmc_multi_copy_results(kmc_multi_t m, double *thetas, double *logp, double *accept_ratio);

#ifdef __cplusplus
}
#endif
#endif /* KISSMCMC_CUDA_H */
