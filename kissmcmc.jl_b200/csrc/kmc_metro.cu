// kmc_metro.cu -- C-ABI of the batched Metropolis sampler (the reference's `metropolis`, src/samplers.jl:9-128):
// handle creation, replay upload, the draws entry point and the run dispatch.  A Metropolis run is a kmc_sampler_t,
// so the result, state, statistics and squash entry points of kmc_api.cu / kmc_aux.cu serve it unchanged.
#include <cmath>
#include <cstring>

#include "kmc_internal.cuh"
#include "kmc_metropolis.cuh"

using namespace kmc_host;

namespace kmc_host {

namespace {

// The Metropolis run paths: each enqueues steps [t0, t1) of p, recording ev0 where its timed window starts, and reports
// its kernel launches.

// Fused plugins: the whole range in one launch, state in registers.
int32_t mh_run_fused(kmc_sampler_s *s, kmc::MhParams &p, long long t0, long long t1, long long &launches) {
    const bool replay = s->opts.mode == KMC_MODE_REPLAY;
    CU_TRY(cudaEventRecord(s->ev0, s->stream));
    p.t0 = t0;
    p.t1 = t1;
    void *args[] = {&p, s->dn->params.data(), s->chol ? s->chol_packed.data() : s->sigma.data()};
    const unsigned grid = (unsigned)((s->nw + kmc::kMhThreads - 1) / kmc::kMhThreads);
    const void *k = s->chol ? s->dn->ops.mh_chol[replay ? 1 : 0] : s->dn->ops.mh[replay ? 1 : 0];
    CU_TRY(cudaLaunchKernel(k, dim3(grid), dim3(kmc::kMhThreads), args, 0, s->stream));
    launches = 1;
    return KMC_OK;
}

// Batched plugins: propose -> batched log-density -> accept, per step.
int32_t mh_run_batched(kmc_sampler_s *s, kmc::MhParams &p, long long t0, long long t1, long long &launches) {
    const bool replay = s->opts.mode == KMC_MODE_REPLAY;
    const int d = s->d;
    CU_TRY(cudaEventRecord(s->ev0, s->stream));
    const long long npair = (d + 1) / 2;
    const unsigned gp = (unsigned)((s->nw * npair + 255) / 256), ga = (unsigned)((s->nw * 32 + 255) / 256);
    const dim3 gt((unsigned)((s->nw + kmc::kMhTri - 1) / kmc::kMhTri), (unsigned)((d + kmc::kMhTri - 1) / kmc::kMhTri));
    auto normals = replay ? kmc::mh_normals_kernel<true> : kmc::mh_normals_kernel<false>;
    auto propose = replay ? kmc::mh_propose_kernel<true> : kmc::mh_propose_kernel<false>;
    for (long long t = t0; t < t1; ++t) {
        p.t0 = t;
        p.t1 = t + 1;
        const auto clk = kmc::ThinClock<>::at(t, s->opts.nburnin_walker, s->opts.nthin);
        const int store = clk.store() ? 1 : 0;
        if (s->chol) {  // Z, U; then Y = X + L Z
            normals<<<gp, 256, 0, s->stream>>>(p, t, d, s->d_z, s->bb.u);
            kmc::mh_chol_kernel<<<gt, dim3(kmc::kMhTri, 8), 0, s->stream>>>(s->x, s->d_chol, s->d_z, s->nw, d, s->bb.Y);
        } else {
            propose<<<gp, 256, 0, s->stream>>>(p, s->d_sigma, t, d, s->bb.Y, s->bb.u);
        }
        CU_TRY(eval_on_device(*s->dn, s->bb.Y, s->nw, s->bb.p1, s->bsc, s->stream));
        kmc::mh_accept_kernel<<<ga, 256, 0, s->stream>>>(p, s->bb.Y, s->bb.p1, s->bb.u, d, clk.n, store, clk.sidx);
    }
    CU_TRY(cudaGetLastError());
    launches = (t1 - t0) * ((s->chol ? 3 : 2) + eval_launches(*s->dn));
    return KMC_OK;
}

}  // namespace

int32_t metro_run(kmc_sampler_s *s, long long nsteps) {
    return run_range(s, s->tdone, s->opts.niter_walker, nsteps, 1,
                     [s](long long t0, long long t1, long long &launches) -> int32_t {
        kmc::MhParams p{};
        p.x = s->x;
        p.lp = s->lp;
        p.nacc = s->nacc;
        p.chain_x = s->chain_x;
        p.chain_lp = s->chain_lp;
        p.rp_n = s->rp_n;
        p.rp_u = s->rp_u;
        p.rp_t0 = s->rp_t0;
        p.nchains = s->nw;
        p.nburnin = s->opts.nburnin_walker;
        p.nthin = s->opts.nthin;
        p.keys = kmc::philox_keys(s->opts.seed);
        p.id_base = (unsigned)s->opts.walker_id_base;
        return s->dn->ops.batch ? mh_run_batched(s, p, t0, t1, launches) : mh_run_fused(s, p, t0, t1, launches);
    });
}

}  // namespace kmc_host

// kmc_metropolis_create (chol == NULL: y = x + sigma .* z) and kmc_metropolis_create_chol (sigma == NULL: y = x + L z).
static int32_t metro_create(kmc_density_t density, const double *theta0s, int64_t nchains, int32_t d, const double *sigma,
                            int64_t nsigma, const double *chol, const kmc_emcee_opts *opts, kmc_sampler_t *out) {
    if (!out) return fail(KMC_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (!density || !theta0s || !(sigma || chol) || !opts) return fail(KMC_ERR_INVALID, "NULL argument");
    if (d != density->d) return fail(KMC_ERR_INVALID, "d=%d does not match the density (d=%d)", d, density->d);
    if (nchains < 1) return fail(KMC_ERR_INVALID, "nchains must be >= 1");
    if (opts->walker_id_base < 0 || opts->walker_id_base + nchains > (1LL << 32))
        return fail(KMC_ERR_INVALID, "chain ids [%lld, %lld) do not fit the 32-bit Philox counter word",
                    (long long)opts->walker_id_base, (long long)(opts->walker_id_base + nchains));
    if (opts->nthin < 1) return fail(KMC_ERR_INVALID, "nthin must be >= 1");
    if (opts->niter_walker < 0 || opts->nburnin_walker < 0) return fail(KMC_ERR_INVALID, "niter and nburnin must be >= 0");
    if (opts->mode != KMC_MODE_PHILOX && opts->mode != KMC_MODE_REPLAY)
        return fail(KMC_ERR_INVALID, "unknown mode %d", opts->mode);
    if (opts->launch_mode || opts->exchange || opts->shard_begin || opts->shard_count || opts->push_chunk ||
        opts->push_cap || opts->push_lag)
        return fail(KMC_ERR_INVALID, "launch_mode, exchange, shard_* and push_* must be 0 for Metropolis");
    if (chol) {  // d x d row-major, lower-triangular with a positive diagonal: a full covariance fails here
        for (int i = 0; i < d; ++i)
            for (int j = 0; j < d; ++j) {
                const double v = chol[(size_t)i * d + j];
                if (!std::isfinite(v)) return fail(KMC_ERR_INVALID, "chol[%d][%d] = %g is not finite", i, j, v);
                if (j > i && v != 0.0)
                    return fail(KMC_ERR_INVALID, "chol[%d][%d] = %g: the factor must be lower-triangular (row-major)", i, j, v);
                if (j == i && !(v > 0.0))
                    return fail(KMC_ERR_INVALID, "chol[%d][%d] = %g: the diagonal must be > 0", i, j, v);
            }
    } else {
        if (nsigma != 1 && nsigma != d)
            return fail(KMC_ERR_INVALID, "sigma has %lld entries: give 1 or d=%d", (long long)nsigma, d);
        for (int64_t k = 0; k < nsigma; ++k)
            if (!(std::isfinite(sigma[k]) && sigma[k] > 0.0))
                return fail(KMC_ERR_INVALID, "sigma[%lld] = %g: proposal scales must be finite and > 0", (long long)k, sigma[k]);
    }
    if (!density->ops.batch && !density->ops.mh[0])
        return fail(KMC_ERR_UNSUPPORTED, "no Metropolis kernel for this plugin and d=%d", d);
    if (density->ops.batch && opts->device != density->device)
        return fail(KMC_ERR_INVALID, "the density's parameters / data live on device %d, the sampler was asked for device %d",
                    density->device, opts->device);

    CU_TRY(cudaSetDevice(opts->device));
    SamplerPtr s(new kmc_sampler_s, kmc_emcee_destroy);
    s->metro = true;
    s->dn = density;
    s->opts = *opts;
    s->nw = s->nl = s->nstate = s->scnt = nchains;  // squash reads the counters as one block of scnt
    s->d = d;
    const long long nspan = opts->niter_walker - opts->nburnin_walker;
    s->ns = nspan > 0 ? nspan / opts->nthin : 0;  // ns = (niter - nburnin) / nthin
    s->sigma.assign(d, 0.0);
    if (chol) {
        s->chol = true;
        s->chol_packed.resize((size_t)d * (d + 1) / 2);
        for (int i = 0; i < d; ++i)
            for (int j = 0; j <= i; ++j) s->chol_packed[(size_t)i * (i + 1) / 2 + j] = chol[(size_t)i * d + j];
    } else {
        for (int k = 0; k < d; ++k) s->sigma[k] = sigma[nsigma == 1 ? 0 : k];
    }
    if (const int32_t rc = sampler_init(s.get(), theta0s); rc != KMC_OK) return rc;
    if (density->ops.batch) {  // the proposal in device memory
        CU_TRY(dev_alloc(&s->d_sigma, sizeof(double) * d, opts->device));
        CU_TRY(cudaMemcpyAsync(s->d_sigma, s->sigma.data(), sizeof(double) * d, cudaMemcpyHostToDevice, s->stream));
        if (chol) {
            CU_TRY(dev_alloc(&s->d_chol, sizeof(double) * d * d, opts->device));
            CU_TRY(dev_alloc(&s->d_z, sizeof(double) * nchains * d, opts->device));
            CU_TRY(cudaMemcpyAsync(s->d_chol, chol, sizeof(double) * d * d, cudaMemcpyHostToDevice, s->stream));
        }
    }
    CU_TRY(cudaStreamSynchronize(s->stream));
    *out = s.release();
    return KMC_OK;
}

extern "C" {

int32_t kmc_metropolis_create(kmc_density_t density, const double *theta0s, int64_t nchains, int32_t d,
                              const double *sigma, int64_t nsigma, const kmc_emcee_opts *opts, kmc_sampler_t *out) {
    return metro_create(density, theta0s, nchains, d, sigma, nsigma, nullptr, opts, out);
}

int32_t kmc_metropolis_create_chol(kmc_density_t density, const double *theta0s, int64_t nchains, int32_t d,
                                   const double *chol, const kmc_emcee_opts *opts, kmc_sampler_t *out) {
    return metro_create(density, theta0s, nchains, d, nullptr, 0, chol, opts, out);
}

int32_t kmc_metropolis_set_replay(kmc_sampler_t s, const double *normals, const double *u, int64_t niters) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    if (!s->metro) return fail(KMC_ERR_STATE, "not a Metropolis handle: use kmc_emcee_set_replay");
    if (s->opts.mode != KMC_MODE_REPLAY) return fail(KMC_ERR_STATE, "sampler is not in replay mode");
    if (niters < 0 || (niters > 0 && (!normals || !u))) return fail(KMC_ERR_INVALID, "bad argument");
    CU_TRY(cudaSetDevice(s->opts.device));
    CU_TRY(cudaStreamSynchronize(s->stream));
    dev_free(s->rp_n);
    dev_free(s->rp_u);
    s->rp_n = s->rp_u = nullptr;
    s->rp_niters = 0;
    const long long n = niters * s->nw;
    if (n > 0) {
        CU_TRY(dev_alloc(&s->rp_n, sizeof(double) * n * s->d, s->opts.device));
        CU_TRY(dev_alloc(&s->rp_u, sizeof(double) * n, s->opts.device));
        CU_TRY(cudaMemcpy(s->rp_n, normals, sizeof(double) * n * s->d, cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(s->rp_u, u, sizeof(double) * n, cudaMemcpyHostToDevice));
    }
    s->rp_t0 = s->tdone;
    s->rp_niters = niters;
    return KMC_OK;
}

int32_t kmc_metropolis_draws(uint64_t seed, int64_t chain0, int64_t nchains, int64_t t0, int64_t niters, int32_t d,
                             int32_t device, double *normals, double *u) {
    if (chain0 < 0 || nchains < 0 || chain0 + nchains > (1LL << 32) || t0 < 0 || niters < 0 || d < 1)
        return fail(KMC_ERR_INVALID, "bad argument");
    const long long n = nchains * niters;
    if (n == 0) return KMC_OK;
    if (!normals || !u) return fail(KMC_ERR_INVALID, "NULL output");
    CU_TRY(cudaSetDevice(device));
    DevBuf<double> dn, du;
    CU_TRY(dev_alloc(dn, sizeof(double) * n * d, device));
    CU_TRY(dev_alloc(du, sizeof(double) * n, device));
    const long long ne = n * ((d + 1) / 2);
    kmc::mh_draws_kernel<<<(unsigned)((ne + 255) / 256), 256>>>(kmc::philox_keys(seed), (unsigned)chain0, nchains, t0,
                                                                 niters, d, dn.get(), du.get());
    CU_TRY(cudaMemcpy(normals, dn.get(), sizeof(double) * n * d, cudaMemcpyDeviceToHost));
    CU_TRY(cudaMemcpy(u, du.get(), sizeof(double) * n, cudaMemcpyDeviceToHost));
    return KMC_OK;
}

int32_t kmc_emcee_chain_covariance(kmc_sampler_t s, double *mean, double *cov, int64_t *count) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    const long long nrows = stored_samples(s) * s->nl;  // the rows kmc_emcee_chain_moments reduces
    const int d = s->d;
    if (count) *count = nrows;
    if (d > kmc::kCovMaxD) return fail(KMC_ERR_UNSUPPORTED, "chain covariance supports d <= %d, got d=%d", kmc::kCovMaxD, d);
    if (nrows < 1) return fail(KMC_ERR_STATE, "no samples stored");
    CU_TRY(cudaSetDevice(s->opts.device));
    const int P = (d + 1) * (d + 2) / 2;  // upper triangle over the d components and the constant column
    DevBuf<double> part;
    CU_TRY(dev_alloc(part, sizeof(double) * ((size_t)kmc::kCovGrid + 1) * P, s->opts.device));
    double *sums = part.get() + (size_t)kmc::kCovGrid * P;
    std::vector<double> h(P), shift(d);
    kmc::mh_cov_partial_kernel<<<kmc::kCovGrid, kmc::kCovThreads, 0, s->stream>>>(s->chain_x, nrows, d, part.get());
    kmc::mh_cov_final_kernel<<<(P + 255) / 256, 256, 0, s->stream>>>(part.get(), P, kmc::kCovGrid, sums);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(h.data(), sums, sizeof(double) * P, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaMemcpyAsync(shift.data(), s->chain_x, sizeof(double) * d, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    const int dc = d + 1;
    auto at = [&](int a, int b) { return h[(size_t)a * dc - (size_t)a * (a - 1) / 2 + (b - a)]; };  // a <= b
    const double n = (double)nrows;
    for (int a = 0; a < d; ++a) {
        const double sa = at(a, d);
        if (mean) mean[a] = shift[a] + sa / n;
        if (cov)
            for (int b = a; b < d; ++b) {
                const double v = nrows > 1 ? (at(a, b) - sa * at(b, d) / n) / (n - 1.0) : 0.0;
                cov[(size_t)a * d + b] = cov[(size_t)b * d + a] = v;
            }
    }
    return KMC_OK;
}

}  // extern "C"
