/*
 * kmo_mixture.c -- CPU ORACLE for the "gaussian_mixture" log-density plugin.  TEST INFRASTRUCTURE ONLY.
 *
 * Builds on the emcee oracle (oracle/kmc_oracle.c, included unchanged): its density record, Philox draws and plugins.
 * The product (libkissmcmc_cuda.so) never links, loads or calls this file.  Compile with -ffp-contract=off: IEEE
 * binary64, round-to-nearest, no fused multiply-add, glibc exp and log.
 *
 * The mixture (kind 5): K = nparams / q components of q = d + d(d+1)/2 + 1 params
 *   [mu_k(d), upper triangle of A_k = chol(Sigma_k^-1)^T row by row (row i holds j = i..d-1), c_k = log(w_k/sum w) +
 *   lognorm_k], and, in this order,
 *     y_i = 0.0; y_i = y_i + A_k[i][j]*(x_j - mu_k[j]) for j = i..d-1 ascending;  ss = 0.0; ss = ss + y_i*y_i;
 *     l_k = c_k - 0.5*ss;  m = max_k l_k with NaN propagated ((l > m || l != l) ? l : m), returned if NaN or -Inf;
 *     s = 0.0; s = s + exp(l_k - m) for k ascending;  return m + log(s).
 *
 * kmo_mix_emcee and kmo_mix_metropolis are the loops of kmo_emcee (oracle/kmc_oracle.c) and kmo_metropolis_loop
 * (metropolis_oracle/kmo_metropolis.c) restated line for line over kmo_mix_logpdf, which is the mixture for kind 5 and
 * kmo_logpdf for every other kind (tests/test_mixture_host.py checks that both loops give the bits of the originals
 * on the other plugins).
 */
#include "../oracle/kmc_oracle.c"

#define KMO_GAUSSIAN_MIXTURE 5

/* l_k of one component pk = [mu_k(d), upper triangle of A_k row by row, c_k] */
static double mix_component(const double *pk, int d, const double *x) {
    const double *a = pk + d;
    double ss = 0.0;
    for (int i = 0; i < d; ++i) {
        double y = 0.0;
        for (int j = i; j < d; ++j) y = y + *a++ * (x[j] - pk[j]);
        ss = ss + y * y;
    }
    return *a - 0.5 * ss;
}

double kmo_mix_logpdf(const kmo_density *dn, const double *x) {
    if (dn->kind != KMO_GAUSSIAN_MIXTURE) return kmo_logpdf(dn, x);
    const int d = dn->d, q = d + d * (d + 1) / 2 + 1;
    const int64_t K = dn->nparams / q;
    const double *p = dn->params;
    double m = -INFINITY;
    for (int64_t k = 0; k < K; ++k) {
        const double l = mix_component(p + k * q, d, x);
        m = (l > m || l != l) ? l : m;
    }
    if (m != m || m == -INFINITY) return m;
    double s = 0.0;
    for (int64_t k = 0; k < K; ++k) s = s + exp(mix_component(p + k * q, d, x) - m);
    return m + log(s);
}

void kmo_mix_eval(const kmo_density *dn, const double *thetas, int64_t nw, double *out, int32_t nthreads) {
#ifdef _OPENMP
    if (nthreads < 1) nthreads = omp_get_max_threads();
#endif
#pragma omp parallel for schedule(static) num_threads(nthreads) if (nthreads > 1)
    for (int64_t w = 0; w < nw; ++w) out[w] = kmo_mix_logpdf(dn, thetas + w * dn->d);
}

/* kmo_emcee (src/samplers.jl:232-293) over kmo_mix_logpdf; arguments as there */
int kmo_mix_emcee(const kmo_density *dn, double *x, double *lp, int64_t nw, int64_t niter_walker,
                  int64_t nburnin_walker, int64_t nthin, double a_scale, int32_t mode, uint64_t seed,
                  const int64_t *rp_partner, const double *rp_z, const double *rp_u, double *chain_x,
                  double *chain_lp, int64_t *naccept, double *accept_ratio, int64_t *tr_partner, double *tr_z,
                  double *tr_u, uint8_t *tr_accept, double *min_margin, int32_t nthreads) {
    const int d = dn->d;
    if (nw < 2 || (nw & 1) || !(a_scale > 1.0) || nthin < 1 || d < 1 || d > 4096) return 1;
    const int64_t nhalf = nw / 2;
    const int64_t ns = (niter_walker - nburnin_walker) / nthin;
    const double sa = sqrt(a_scale), sia = sqrt(1.0 / a_scale);
    const double span = sa - sia;
    const double nm1 = (double)(d - 1);
    double margin = INFINITY;
#ifdef _OPENMP
    if (nthreads < 1) nthreads = omp_get_max_threads();
#else
    nthreads = 1;
#endif
    for (int64_t w = 0; w < nw; ++w) naccept[w] = 0;
    int64_t t = 0;
    for (int64_t n = 1 - nburnin_walker; n <= niter_walker - nburnin_walker; ++n, ++t) {
        for (int batch = 0; batch < 2; ++batch) {
            const int64_t a0 = batch == 0 ? 0 : nhalf;
            const int64_t p0 = batch == 0 ? nhalf : 0;
            const int store = (n > 0 && n % nthin == 0);
            const int64_t sidx = store ? n / nthin - 1 : 0;
#pragma omp parallel for schedule(static) num_threads(nthreads) reduction(min : margin) if (nthreads > 1)
            for (int64_t i = 0; i < nhalf; ++i) {
                const int64_t k = a0 + i;
                const int64_t slot = (t * 2 + batch) * nhalf + i;
                int64_t j;
                double z, u;
                if (mode == KMO_MODE_REPLAY) {
                    j = rp_partner[slot];
                    z = rp_z[slot];
                    u = rp_u[slot];
                } else {
                    int64_t pl;
                    double uz;
                    kmo_draw(seed, (uint64_t)k, (uint64_t)t, (uint32_t)batch, (uint64_t)nhalf, &pl, &uz, &u);
                    j = p0 + pl;
                    double s = uz * span + sia;
                    z = s * s;
                }
                double y[d];
                const double *xk = x + k * d, *xj = x + j * d;
                for (int c = 0; c < d; ++c) y[c] = xj[c] + z * (xk[c] - xj[c]);
                const double p1 = kmo_mix_logpdf(dn, y);
                const double lhs = (nm1 * log(z) + p1) - lp[k];
                const double lu = log(u);
                const int acc = lhs >= lu;
                if (acc) {
                    for (int c = 0; c < d; ++c) x[k * d + c] = y[c];
                    lp[k] = p1;
                    naccept[k] += 1;
                }
                if (isfinite(lhs) && isfinite(lu)) {
                    double mg = fabs(lhs - lu);
                    if (mg < margin) margin = mg;
                }
                if (tr_partner) tr_partner[slot] = j;
                if (tr_z) tr_z[slot] = z;
                if (tr_u) tr_u[slot] = u;
                if (tr_accept) tr_accept[slot] = (uint8_t)acc;
                if (store && chain_x) {
                    for (int c = 0; c < d; ++c) chain_x[(k * ns + sidx) * d + c] = x[k * d + c];
                    chain_lp[k * ns + sidx] = lp[k];
                }
            }
        }
        if (n == 0)
            for (int64_t w = 0; w < nw; ++w) naccept[w] = 0;
    }
    for (int64_t w = 0; w < nw; ++w) accept_ratio[w] = (double)naccept[w] / (double)(niter_walker - nburnin_walker);
    if (min_margin) *min_margin = margin;
    return 0;
}

/* kmo_metropolis_loop (metropolis_oracle/kmo_metropolis.c) over kmo_mix_logpdf: sigma [nsigma] (chol == NULL) or the
 * lower-triangular chol [d][d] row-major (sigma == NULL); other arguments as there */
int kmo_mix_metropolis(const kmo_density *dn, double *x, double *lp, int64_t nchains, int64_t niter, int64_t nburnin,
                       int64_t nthin, const double *sigma, int64_t nsigma, const double *chol, const double *normals,
                       const double *u, double *chain_x, double *chain_lp, int64_t *naccept, double *accept_ratio,
                       double *min_margin, int32_t nthreads) {
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
        double p0 = kmo_mix_logpdf(dn, th);
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
            const double p1 = kmo_mix_logpdf(dn, y);
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
