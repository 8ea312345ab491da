/*
 * kmo_metropolis.c -- CPU ORACLE for the batched random-walk Metropolis sampler.  TEST INFRASTRUCTURE ONLY.
 *
 * Builds on the emcee oracle (oracle/kmc_oracle.c, included unchanged): the same log-density plugins (kmo_logpdf)
 * and the same arithmetic contract -- IEEE binary64, round-to-nearest, no fused multiply-add (-ffp-contract=off).
 * The product (libkissmcmc_cuda.so) never links, loads or calls this file.
 *
 * What it restates: the reference's `metropolis` / `_metropolis`, src/samplers.jl:9-128 (accept test :103).  The
 * reference source is not vendored in this checkout, so the loop below is a RESTATEMENT written to the conventions
 * of `_emcee` that kmc_oracle.c pins; like emcee, its parity with Julia is UNPINNED (Julia's RNG stream, its randn
 * and Base.log cannot run here).  The draws are inputs, so any draw source can be replayed through it:
 *
 *   p0 = pdf(theta0)                                     no error if p0 == -Inf
 *   naccept = 0
 *   for ni in (1-nburnin):(niter-nburnin)                step t = ni + nburnin - 1 (0-based)
 *       theta1 = theta0 .+ sigma .* n_t                  mul, then add
 *       p1 = pdf(theta1)
 *       if p1 - p0 > log(u_t)                            strict >, FP64; NaN rejects
 *           theta0 = theta1; p0 = p1; naccept += 1
 *       if ni > 0 && rem(ni, nthin) == 0: store (theta0, p0) as sample ni/nthin
 *       if ni == 0: naccept = 0
 *   accept_ratio = naccept / (niter - nburnin)
 *
 * kmo_metropolis_chol is the same loop with the correlated proposal of kmc_metropolis_create_chol (L lower-triangular,
 * [d][d] row-major):
 *       for i in 0..d-1: s = 0.0; for j in 0..i: s = s + L[i][j] * n_t[j];  theta1[i] = theta0[i] + s
 */
#include "../oracle/kmc_oracle.c"

/*
 *  x        [nchains][d] in/out: theta0 of every chain, the final state on return
 *  lp       [nchains] out: the final log-density
 *  sigma    [nsigma], nsigma = 1 or d (chol == NULL); chol [d][d] lower-triangular, row-major (sigma == NULL)
 *  normals  [niter][nchains][d], u [niter][nchains]: the draws of step t of chain c at [t][c]
 *  chain_x  [nchains][ns][d], chain_lp [nchains][ns] (may be NULL), ns = (niter - nburnin) / nthin
 *  naccept, accept_ratio [nchains] out
 *  min_margin: min over finite decisions of |(p1 - p0) - log(u)| (how far any decision was from a tie)
 */
static int kmo_metropolis_loop(const kmo_density *dn, double *x, double *lp, int64_t nchains, int64_t niter,
                               int64_t nburnin, int64_t nthin, const double *sigma, int64_t nsigma, const double *chol,
                               const double *normals, const double *u, double *chain_x, double *chain_lp,
                               int64_t *naccept, double *accept_ratio, double *min_margin, int32_t nthreads) {
    const int d = dn->d;
    if (nchains < 1 || nthin < 1 || niter < 0 || nburnin < 0 || d < 1 || d > 4096 ||
        (!chol && nsigma != 1 && nsigma != d))
        return 1;
    const int64_t ns = niter > nburnin ? (niter - nburnin) / nthin : 0;
    double margin = INFINITY;
#ifdef _OPENMP
    if (nthreads < 1) nthreads = omp_get_max_threads();
#else
    nthreads = 1;
#endif
#pragma omp parallel for schedule(dynamic, 16) num_threads(nthreads) reduction(min : margin) if (nthreads > 1)
    for (int64_t c = 0; c < nchains; ++c) {
        double *th = x + c * d;
        double y[d];
        double p0 = kmo_logpdf(dn, th);
        int64_t na = 0;
        int64_t t = 0;
        for (int64_t ni = 1 - nburnin; ni <= niter - nburnin; ++ni, ++t) {
            const double *n = normals + (t * nchains + c) * d;
            if (chol) {
                for (int i = 0; i < d; ++i) {
                    double s = 0.0;
                    for (int j = 0; j <= i; ++j) s = s + chol[(int64_t)i * d + j] * n[j];
                    y[i] = th[i] + s;
                }
            } else {
                for (int k = 0; k < d; ++k) y[k] = th[k] + sigma[nsigma == 1 ? 0 : k] * n[k];
            }
            const double p1 = kmo_logpdf(dn, y);
            const double lhs = p1 - p0, lu = log(u[t * nchains + c]);
            if (lhs > lu) {
                for (int k = 0; k < d; ++k) th[k] = y[k];
                p0 = p1;
                na += 1;
            }
            if (isfinite(lhs) && isfinite(lu)) {
                const double mg = fabs(lhs - lu);
                if (mg < margin) margin = mg;
            }
            if (ni > 0 && ni % nthin == 0 && chain_x) {
                const int64_t sidx = ni / nthin - 1;
                for (int k = 0; k < d; ++k) chain_x[(c * ns + sidx) * d + k] = th[k];
                chain_lp[c * ns + sidx] = p0;
            }
            if (ni == 0) na = 0;
        }
        lp[c] = p0;
        naccept[c] = na;
        accept_ratio[c] = (double)na / (double)(niter - nburnin);
    }
    if (min_margin) *min_margin = margin;
    return 0;
}

int kmo_metropolis(const kmo_density *dn, double *x, double *lp, int64_t nchains, int64_t niter, int64_t nburnin,
                   int64_t nthin, const double *sigma, int64_t nsigma, const double *normals, const double *u,
                   double *chain_x, double *chain_lp, int64_t *naccept, double *accept_ratio, double *min_margin,
                   int32_t nthreads) {
    return kmo_metropolis_loop(dn, x, lp, nchains, niter, nburnin, nthin, sigma, nsigma, NULL, normals, u, chain_x,
                               chain_lp, naccept, accept_ratio, min_margin, nthreads);
}

int kmo_metropolis_chol(const kmo_density *dn, double *x, double *lp, int64_t nchains, int64_t niter, int64_t nburnin,
                        int64_t nthin, const double *chol, const double *normals, const double *u, double *chain_x,
                        double *chain_lp, int64_t *naccept, double *accept_ratio, double *min_margin, int32_t nthreads) {
    if (!chol) return 1;
    return kmo_metropolis_loop(dn, x, lp, nchains, niter, nburnin, nthin, NULL, 0, chol, normals, u, chain_x, chain_lp,
                               naccept, accept_ratio, min_margin, nthreads);
}
