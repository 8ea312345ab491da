// kmc_aux.cu -- C-ABI entry points around the sampler: library-owned multi-GPU (kmc_emcee_create_multi / kmc_multi_*),
// the g-distribution helpers, and the device-side squash_walkers / make_theta0s.
#include <math_constants.h>

#include <algorithm>
#include <cmath>
#include <cstring>

#include "kmc_internal.cuh"

using namespace kmc_host;

struct kmc_multi_s {
    int mode = KMC_MULTI_SHARDED;
    long long nw = 0;  // walkers per ensemble
    int d = 0;
    std::vector<kmc_sampler_s *> subs;
};

extern "C" {

int32_t kmc_multi_destroy(kmc_multi_t m) {
    if (!m) return KMC_OK;
    for (auto *s : m->subs)  // nobody tears its window down while a peer's kernel may still write into it
        if (s) {
            cudaSetDevice(s->opts.device);
            cudaStreamSynchronize(s->stream);
        }
    for (auto *s : m->subs) kmc_emcee_destroy(s);
    delete m;
    return KMC_OK;
}

int32_t kmc_emcee_create_multi(const kmc_density_t *densities, const double *theta0s, int64_t nwalkers, int32_t d,
                               const kmc_emcee_opts *opts, const int32_t *devices, int32_t ndev, int32_t mode,
                               kmc_multi_t *out) {
    if (!out) return fail(KMC_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (!densities || !theta0s || !opts || !devices) return fail(KMC_ERR_INVALID, "NULL argument");
    if (ndev < 1 || ndev > kmc::kPushMaxRanks) return fail(KMC_ERR_INVALID, "ndev must be in [1, 8]");
    if (mode != KMC_MULTI_SHARDED && mode != KMC_MULTI_INDEPENDENT) return fail(KMC_ERR_INVALID, "unknown mode %d", mode);
    for (int r = 0; r < ndev; ++r)
        if (!densities[r]) return fail(KMC_ERR_INVALID, "densities[%d] is NULL", r);
    if (mode == KMC_MULTI_SHARDED && (nwalkers < 2 || (nwalkers & 1) || (nwalkers / 2) % ndev))
        return fail(KMC_ERR_INVALID, "nwalkers/2 must be a multiple of the number of devices");
    // the handle under construction, deleted by kmc_multi_destroy (which sets no error) on every exit but the last
    std::unique_ptr<kmc_multi_s, int32_t (*)(kmc_multi_t)> m(new kmc_multi_s, kmc_multi_destroy);
    m->mode = mode;
    m->nw = nwalkers;
    m->d = d;
    m->subs.assign(ndev, nullptr);
    const long long S = nwalkers / 2 / ndev;
    for (int r = 0; r < ndev; ++r) {
        kmc_emcee_opts o = *opts;
        o.device = devices[r];
        if (mode == KMC_MULTI_SHARDED) {
            o.exchange = KMC_EXCHANGE_PUSH;
            o.shard_begin = r * S;
            o.shard_count = S;
            o.launch_mode = 0;
        } else {  // independent ensembles: disjoint walker ids => disjoint Philox streams
            o.exchange = KMC_EXCHANGE_REPLICA;
            o.shard_begin = o.shard_count = 0;
            o.walker_id_base = opts->walker_id_base + (int64_t)r * nwalkers;
        }
        const double *th = mode == KMC_MULTI_SHARDED ? theta0s : theta0s + (size_t)r * nwalkers * d;
        const int32_t rc = kmc_emcee_create(densities[r], th, nwalkers, d, &o, &m->subs[r]);
        if (rc != KMC_OK) return rc;
    }
    if (mode == KMC_MULTI_SHARDED) {
        for (int a = 0; a < ndev; ++a) {
            kmc_sampler_s *sa = m->subs[a];
            int share = 0;
            for (int b = 0; b < ndev; ++b) share += devices[b] == devices[a] ? 1 : 0;
            sa->share = share;  // sub-samplers of one GPU must all be co-resident: split the CTA slots
            sa->grid = std::max(1u, sa->grid / (unsigned)share);
            sa->lag = push_default_lag(sa->nchunks, opts->push_lag);
            CU_TRY(cudaSetDevice(devices[a]));
            for (int b = 0; b < ndev; ++b) {
                if (devices[b] != devices[a]) {
                    int can = 0;
                    cudaDeviceCanAccessPeer(&can, devices[a], devices[b]);
                    if (!can) return fail(KMC_ERR_CUDA, "device %d cannot access device %d's memory", devices[a], devices[b]);
                    const cudaError_t e = cudaDeviceEnablePeerAccess(devices[b], 0);
                    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled)
                        return fail(KMC_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d) failed: %s", devices[a], devices[b],
                                    cudaGetErrorString(e));
                    cudaGetLastError();
                }
                push_set_peer(sa, b, m->subs[b]->window);
            }
            sa->attached = true;
        }
    }
    *out = m.release();
    return KMC_OK;
}

int32_t kmc_multi_run(kmc_multi_t m, int64_t niters) {
    if (!m) return fail(KMC_ERR_INVALID, "NULL handle");
    for (auto *s : m->subs) {  // asynchronous launches: the devices' kernels synchronise among themselves
        const int32_t rc = kmc_emcee_run(s, niters);
        if (rc != KMC_OK) return rc;
    }
    return KMC_OK;
}

int32_t kmc_multi_sync(kmc_multi_t m) {
    if (!m) return fail(KMC_ERR_INVALID, "NULL handle");
    for (auto *s : m->subs) {
        const int32_t rc = kmc_emcee_sync(s);
        if (rc != KMC_OK) return rc;
    }
    return KMC_OK;
}

int32_t kmc_multi_last_run_ms(kmc_multi_t m, double *ms) {
    if (!m || !ms) return fail(KMC_ERR_INVALID, "NULL argument");
    *ms = 0.0;
    for (auto *s : m->subs) {
        double v = 0.0;
        const int32_t rc = kmc_emcee_last_run_ms(s, &v, nullptr);
        if (rc != KMC_OK) return rc;
        *ms = std::max(*ms, v);
    }
    return KMC_OK;
}

int32_t kmc_multi_shape(kmc_multi_t m, int64_t *ns, int64_t *nwalkers_out) {
    if (!m) return fail(KMC_ERR_INVALID, "NULL handle");
    if (ns) *ns = m->subs[0]->ns;
    if (nwalkers_out) *nwalkers_out = m->mode == KMC_MULTI_SHARDED ? m->nw : m->nw * (long long)m->subs.size();
    return KMC_OK;
}

int32_t kmc_multi_copy_results(kmc_multi_t m, double *thetas, double *logp, double *accept_ratio) {
    if (!m) return fail(KMC_ERR_INVALID, "NULL handle");
    const long long ns = m->subs[0]->ns, nw = m->nw;
    const int d = m->d, ndev = (int)m->subs.size();
    if (m->mode == KMC_MULTI_INDEPENDENT) {
        for (int r = 0; r < ndev; ++r) {
            const int32_t rc = kmc_emcee_copy_results(m->subs[r], thetas ? thetas + (size_t)r * nw * ns * d : nullptr,
                                                      logp ? logp + (size_t)r * nw * ns : nullptr,
                                                      accept_ratio ? accept_ratio + (size_t)r * nw : nullptr);
            if (rc != KMC_OK) return rc;
        }
        return KMC_OK;
    }
    // sharded: sub r returns its slice of half 0 then of half 1 ([2S] walkers); global order = all slices of half 0, then of half 1
    const long long S = nw / 2 / ndev;
    std::vector<double> th, lp, ar;
    if (thetas) th.resize((size_t)2 * S * ns * d);
    if (logp) lp.resize((size_t)2 * S * ns);
    if (accept_ratio) ar.resize((size_t)2 * S);
    for (int r = 0; r < ndev; ++r) {
        const int32_t rc = kmc_emcee_copy_results(m->subs[r], thetas ? th.data() : nullptr, logp ? lp.data() : nullptr,
                                                  accept_ratio ? ar.data() : nullptr);
        if (rc != KMC_OK) return rc;
        for (int b = 0; b < 2; ++b) {
            const size_t dst = (size_t)b * (nw / 2) + (size_t)r * S, src = (size_t)b * S;
            if (thetas) memcpy(thetas + dst * ns * d, th.data() + src * ns * d, sizeof(double) * S * ns * d);
            if (logp) memcpy(logp + dst * ns, lp.data() + src * ns, sizeof(double) * S * ns);
            if (accept_ratio) memcpy(accept_ratio + dst, ar.data() + src, sizeof(double) * S);
        }
    }
    return KMC_OK;
}

}  // extern "C"

// ====================================================================================================================
// g-distribution helpers (src/samplers.jl:223-230).  g_pdf is test-only in the reference (test/emcee.jl:2-14) but part
// of its source; cdf_g_inv / sample_g are what the sampler's z draw is made of (:252 -> :230 -> :227).
namespace {

// z = cdf_g_inv(u, a) for n device-generated uniforms: the SAME draw path as a walker-step (kmc::draw, z transform of
// step_draws), walker id = sample index, iteration 0, batch 0.
__global__ void sample_g_kernel(kmc::PhiloxKeys keys, double sia, double span, long long n, double *out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned pl;
    double uz, ua;
    kmc::draw(keys, (unsigned)i, (unsigned)(i >> 32), 0u, 0u, 2u, 0u, pl, uz, ua);
    const double s = kmc::dadd(kmc::dmul(uz, span), sia);  // :227
    out[i] = kmc::dmul(s, s);
}

}  // namespace

extern "C" {

int32_t kmc_g_pdf(const double *z, int64_t n, double a_scale, double *out) {
    if ((n > 0 && (!z || !out)) || n < 0) return fail(KMC_ERR_INVALID, "bad argument");
    if (!(a_scale > 1.0)) return fail(KMC_ERR_INVALID, "a_scale must be > 1");
    const double a = a_scale;
    for (int64_t i = 0; i < n; ++i)  // :224  1/sqrt(z) * 1/(2*(sqrt(a)-sqrt(1/a))) on [1/a, a], else 0
        out[i] = (1.0 / a <= z[i] && z[i] <= a) ? 1.0 / std::sqrt(z[i]) * 1.0 / (2.0 * (std::sqrt(a) - std::sqrt(1.0 / a))) : 0.0;
    return KMC_OK;
}

int32_t kmc_cdf_g_inv(const double *u, int64_t n, double a_scale, double *out) {
    if ((n > 0 && (!u || !out)) || n < 0) return fail(KMC_ERR_INVALID, "bad argument");
    if (!(a_scale > 1.0)) return fail(KMC_ERR_INVALID, "a_scale must be > 1");
    const double sa = std::sqrt(a_scale), sia = std::sqrt(1.0 / a_scale);
    for (int64_t i = 0; i < n; ++i) {  // :227
        const double s = u[i] * (sa - sia) + sia;
        out[i] = s * s;
    }
    return KMC_OK;
}

int32_t kmc_sample_g(double a_scale, uint64_t seed, int64_t n, int32_t device, double *out) {
    if (n < 0 || (n > 0 && !out)) return fail(KMC_ERR_INVALID, "bad argument");
    if (!(a_scale > 1.0)) return fail(KMC_ERR_INVALID, "a_scale must be > 1");
    if (n == 0) return KMC_OK;
    CU_TRY(cudaSetDevice(device));
    DevBuf<double> dz;
    CU_TRY(dev_alloc(dz, sizeof(double) * n, device));
    const double sia = std::sqrt(1.0 / a_scale), span = std::sqrt(a_scale) - sia;
    sample_g_kernel<<<(unsigned)((n + 255) / 256), 256>>>(kmc::philox_keys(seed), sia, span, n, dz.get());
    CU_TRY(cudaMemcpy(out, dz.get(), sizeof(double) * n, cudaMemcpyDeviceToHost));
    return KMC_OK;
}

}  // extern "C"

// ====================================================================================================================
// Device-side squash_walkers (src/samplers.jl:372-428): the low-accept-ratio drop (:379-393), the walker-major
// concatenation (:398-399) and the time ordering (:415-426) without copying the per-walker chains to the host first.
namespace {

// counter i of this sampler's walkers: its slice of half 0 (the first na), then of half 1
__device__ __forceinline__ unsigned counter_at(const unsigned *__restrict__ a, const unsigned *__restrict__ b, long long na,
                                               long long i) {
    return i < na ? a[i] : b[i - na];
}

// histogram of (v >> shift) & 0xFFFF over the counters whose upper bits (v >> (shift + 16)) equal `prefix`
__global__ void nacc_hist_kernel(const unsigned *__restrict__ a, const unsigned *__restrict__ b, long long na, long long n,
                                 int shift, unsigned prefix, unsigned *__restrict__ hist) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const unsigned v = counter_at(a, b, na, i);
        if (shift == 16 || (v >> 16) == prefix) atomicAdd(hist + ((v >> shift) & 0xFFFFu), 1u);
    }
}

// exact sum and sum of squares (128-bit: lo/hi with carry) of the counters
__global__ void nacc_sums_kernel(const unsigned *__restrict__ a, const unsigned *__restrict__ b, long long na, long long n,
                                 unsigned long long *__restrict__ out /* sum, sq_lo, sq_hi */) {
    unsigned long long s = 0, lo = 0, hi = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const unsigned long long v = counter_at(a, b, na, i);
        s += v;
        const unsigned long long sq = v * v, nl = lo + sq;
        hi += nl < lo ? 1ull : 0ull;
        lo = nl;
    }
    atomicAdd(out, s);
    const unsigned long long old = atomicAdd(out + 1, lo);
    if (old + lo < old) ++hi;
    if (hi) atomicAdd(out + 2, hi);
}

// ---- ordered compaction: the kept threads' items in thread order, by blocks of kKeepBlock threads.  Each block
// counts its kept threads (compact_count), the host scans the counts into block offsets (compact_offsets), and a
// second launch of the same grid writes each kept item to its slot (compact_slot).
constexpr int kKeepBlock = 1024;

__device__ __forceinline__ void compact_count(bool keep, unsigned *__restrict__ blk_cnt) {
    const int c = __syncthreads_count(keep);
    if (threadIdx.x == 0) blk_cnt[blockIdx.x] = (unsigned)c;
}

// the slot of a kept thread: its block's offset, the kept threads of the lower warps and the kept lanes below it
__device__ __forceinline__ unsigned compact_slot(bool keep, const unsigned *__restrict__ blk_off) {
    __shared__ unsigned wc[kKeepBlock / 32];
    const unsigned bl = __ballot_sync(0xffffffffu, keep), lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    if (lane == 0) wc[wp] = __popc(bl);
    __syncthreads();
    unsigned off = blk_off[blockIdx.x];
    for (unsigned k = 0; k < wp; ++k) off += wc[k];
    return off + __popc(bl & ((1u << lane) - 1u));
}

// d_blk[0, nblk) holds the blocks' counts: their exclusive scan goes to d_blk[nblk, 2 nblk), their sum to `total`
int32_t compact_offsets(unsigned *d_blk, long long nblk, cudaStream_t st, long long &total) {
    std::vector<unsigned> blk(2 * nblk);
    CU_TRY(cudaMemcpyAsync(blk.data(), d_blk, sizeof(unsigned) * nblk, cudaMemcpyDeviceToHost, st));
    CU_TRY(cudaStreamSynchronize(st));
    total = 0;
    for (long long b = 0; b < nblk; ++b) {
        blk[nblk + b] = (unsigned)total;
        total += blk[b];
    }
    CU_TRY(cudaMemcpyAsync(d_blk + nblk, blk.data() + nblk, sizeof(unsigned) * nblk, cudaMemcpyHostToDevice, st));
    return KMC_OK;
}

// walker w is kept unless drop is on and its accept ratio is <= thr (:384-391); v = its counter (0 past the end)
__device__ __forceinline__ bool walker_kept(const unsigned *__restrict__ a, const unsigned *__restrict__ b, long long na,
                                            long long n, long long w, double den, double thr, int drop, unsigned &v) {
    v = w < n ? counter_at(a, b, na, w) : 0u;
    return w < n && (!drop || !((double)v / den <= thr));
}

// per-block kept counts and the exact sum of the kept counters
__global__ void __launch_bounds__(kKeepBlock) keep_count_kernel(const unsigned *__restrict__ a, const unsigned *__restrict__ b,
                                                                long long na, long long n, double den, double thr, int drop,
                                                                unsigned *__restrict__ blk_cnt, unsigned long long *__restrict__ kept_sum) {
    unsigned v;
    const bool keep = walker_kept(a, b, na, n, (long long)blockIdx.x * kKeepBlock + threadIdx.x, den, thr, drop, v);
    unsigned long long sv = keep ? v : 0u;
    for (int o = 16; o > 0; o >>= 1) sv += __shfl_xor_sync(0xffffffffu, sv, o);
    if ((threadIdx.x & 31) == 0 && sv) atomicAdd(kept_sum, sv);
    compact_count(keep, blk_cnt);
}

// kept walker indices in walker order
__global__ void __launch_bounds__(kKeepBlock) keep_index_kernel(const unsigned *__restrict__ a, const unsigned *__restrict__ b,
                                                                long long na, long long n, double den, double thr, int drop,
                                                                const unsigned *__restrict__ blk_off, unsigned *__restrict__ idx) {
    const long long w = (long long)blockIdx.x * kKeepBlock + threadIdx.x;
    unsigned v;
    const bool keep = walker_kept(a, b, na, n, w, den, thr, drop, v);
    const unsigned slot = compact_slot(keep, blk_off);
    if (keep) idx[slot] = (unsigned)w;
}

// time-major gather (order=true, :415-426: the stable sortperm of (1:ns, 1:ns, ...) = sample-major, walkers in kept
// order) of samples [s0, s0+sc): out[((s-s0)*nk + k)*d + c] = in[(s*nl + idx[k])*d + c]
__global__ void squash_time_major_kernel(const double *__restrict__ in, double *__restrict__ out, long long nl, long long nk,
                                         const unsigned *__restrict__ idx, long long s0, long long sc, int d) {
    const long long total = sc * nk * d;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (long long)gridDim.x * blockDim.x) {
        const long long row = e / d;
        const int c = (int)(e - row * d);
        const long long s = row / nk, k = row - s * nk;
        out[e] = in[((s0 + s) * nl + idx[k]) * d + c];
    }
}

// the k-th smallest (0-based) of the n counters: two 16-bit histogram passes
cudaError_t select_kth(const unsigned *a, const unsigned *b, long long na, long long n, long long k, unsigned *d_hist,
                       std::vector<unsigned> &h_hist, cudaStream_t st, unsigned *out) {
    const unsigned grid = (unsigned)std::min<long long>((n + 255) / 256, 1184);
    unsigned prefix = 0;
    for (int pass = 0; pass < 2; ++pass) {
        cudaError_t e = cudaMemsetAsync(d_hist, 0, sizeof(unsigned) * 65536, st);
        if (e != cudaSuccess) return e;
        nacc_hist_kernel<<<grid, 256, 0, st>>>(a, b, na, n, pass == 0 ? 16 : 0, prefix, d_hist);
        e = cudaMemcpyAsync(h_hist.data(), d_hist, sizeof(unsigned) * 65536, cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) return e;
        e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) return e;
        long long acc = 0;
        unsigned bin = 0;
        for (; bin < 65536; ++bin) {
            if (acc + h_hist[bin] > k) break;
            acc += h_hist[bin];
        }
        k -= acc;
        if (pass == 0) prefix = bin;
        else *out = (prefix << 16) | bin;
    }
    return cudaSuccess;
}

}  // namespace

extern "C" {

int32_t kmc_emcee_squash(kmc_sampler_t s, int32_t drop_low_accept_ratio, double drop_fact, int32_t order, double *thetas,
                         double *logp, int64_t *nkept, double *accept_mean, double *accept_median, double *accept_std) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    CU_TRY(cudaSetDevice(s->opts.device));
    CU_TRY(cudaStreamSynchronize(s->stream));
    cudaStream_t st = s->stream;
    const long long nl = s->nl, ns = s->ns, S = s->scnt;
    const int d = s->d;
    // this sampler's counters: its slice of half 0, then of half 1 (the order of its chain rows)
    const unsigned *na = s->nacc + s->loff, *nb = s->nacc + s->hoff + s->loff;
    const double den = (double)(s->opts.niter_walker - s->opts.nburnin_walker);  // :291
    const long long nblk = (nl + kKeepBlock - 1) / kKeepBlock;

    DevBuf<unsigned> d_hist, d_blk, d_idx;
    DevBuf<unsigned long long> d_sums;
    DevBuf<double> stage;
    CU_TRY(dev_alloc(d_hist, sizeof(unsigned) * 65536, s->opts.device));
    CU_TRY(dev_alloc(d_blk, sizeof(unsigned) * 2 * nblk, s->opts.device));
    CU_TRY(dev_alloc(d_idx, sizeof(unsigned) * nl, s->opts.device));
    CU_TRY(dev_alloc(d_sums, sizeof(unsigned long long) * 4, s->opts.device));

    // ---- :385  median and std (n-1) of the accept ratios, from exact integer statistics of the counters
    double med = 0.0, sd = 0.0, thr = 0.0;
    {
        std::vector<unsigned> h_hist(65536);
        unsigned c1 = 0, c2 = 0;
        CU_TRY(select_kth(na, nb, S, nl, (nl - 1) / 2, d_hist.get(), h_hist, st, &c1));
        CU_TRY(select_kth(na, nb, S, nl, nl / 2, d_hist.get(), h_hist, st, &c2));
        med = ((double)c1 / den + (double)c2 / den) / 2.0;  // median of an even count = mean of the two middle values
        if (c1 == c2) med = (double)c1 / den;
        unsigned long long hs[3] = {0, 0, 0};
        CU_TRY(cudaMemsetAsync(d_sums.get(), 0, sizeof(unsigned long long) * 4, st));
        nacc_sums_kernel<<<(unsigned)std::min<long long>((nl + 255) / 256, 1184), 256, 0, st>>>(na, nb, S, nl,
                                                                                                d_sums.get());
        CU_TRY(cudaMemcpyAsync(hs, d_sums.get(), sizeof hs, cudaMemcpyDeviceToHost, st));
        CU_TRY(cudaStreamSynchronize(st));
        const unsigned __int128 sum = hs[0], sq = ((unsigned __int128)hs[2] << 64) | hs[1];
        const unsigned __int128 num = (unsigned __int128)nl * sq - sum * sum;  // n * sum(c^2) - (sum c)^2 >= 0, exact
        const long double var = nl > 1 ? (long double)num / ((long double)nl * (long double)(nl - 1)) : 0.0L;
        sd = (double)(std::sqrt(var) / (long double)den);
        thr = med - drop_fact * sd;
    }
    if (accept_median) *accept_median = med;
    if (accept_std) *accept_std = sd;

    // ---- :380-396  walkers to keep, in walker order
    const int drop = drop_low_accept_ratio ? 1 : 0;
    CU_TRY(cudaMemsetAsync(d_sums.get(), 0, sizeof(unsigned long long) * 4, st));
    keep_count_kernel<<<(unsigned)nblk, kKeepBlock, 0, st>>>(na, nb, S, nl, den, thr, drop, d_blk.get(), d_sums.get());
    unsigned long long kept_sum = 0;
    CU_TRY(cudaMemcpyAsync(&kept_sum, d_sums.get(), sizeof kept_sum, cudaMemcpyDeviceToHost, st));
    long long nk = 0;
    if (const int32_t rc = compact_offsets(d_blk.get(), nblk, st, nk); rc != KMC_OK) return rc;
    keep_index_kernel<<<(unsigned)nblk, kKeepBlock, 0, st>>>(na, nb, S, nl, den, thr, drop, d_blk.get() + nblk,
                                                             d_idx.get());
    if (nkept) *nkept = nk;
    if (accept_mean) *accept_mean = nk > 0 ? (double)kept_sum / den / (double)nk : 0.0;  // :427 mean(accept_ratio[keep])

    // ---- :398-399 / :415-426  the kept chains, walker-major or time-major, staged through <= 64 MiB
    if (ns > 0 && nk > 0 && (thetas || logp)) {
        if (!order) return chain_gather(s, d_idx.get(), nk, thetas, logp);
        long long sc = std::max<long long>(1, (64LL << 20) / ((long long)sizeof(double) * d * nk));
        sc = std::min(sc, ns);
        CU_TRY(dev_alloc(stage, sizeof(double) * sc * nk * d, s->opts.device));
        for (long long s0 = 0; s0 < ns; s0 += sc) {
            const long long cur = std::min(sc, ns - s0);
            for (int what = 0; what < 2; ++what) {
                double *host = what == 0 ? thetas : logp;
                if (!host) continue;
                const int dd = what == 0 ? d : 1;
                const double *src = what == 0 ? s->chain_x : s->chain_lp;
                const unsigned grid = (unsigned)std::min<long long>((cur * nk * dd + 255) / 256, 148 * 16);
                squash_time_major_kernel<<<grid, 256, 0, st>>>(src, stage.get(), nl, nk, d_idx.get(), s0, cur, dd);
                CU_TRY(cudaMemcpyAsync(host + s0 * nk * dd, stage.get(), sizeof(double) * cur * nk * dd,
                                       cudaMemcpyDeviceToHost, st));
            }
        }
    }
    CU_TRY(cudaStreamSynchronize(st));  // the blocks go back to the cache idle (the sizing call ends with keep_index)
    CU_TRY(cudaGetLastError());
    return KMC_OK;
}

}  // extern "C"

// ====================================================================================================================
// Device-side make_theta0s (src/samplers.jl:311-349): the Gaussian ball around theta0 (:328-332), the rejection of
// points of zero density (:338) through the log-density plugin, and the reference's loop semantics including its quirks
// (cumulative, never-reset radius halving at :326; a walker that exhausts every try is silently skipped, :343-346).
// The normals are counter-based: a pure function of (seed, walker, halving step k, try j, component) -- Philox4x32-10,
// counter (walker, component pair, k<<16 | j, stream tag 0x4D54<<16), two 32-bit uniforms -> Box-Muller -- so any walker's
// try can be (re)generated anywhere.  All walkers still pending are tried at once (normally ONE round of three kernels
// for the whole ensemble); the host only drives the rare sequential path of a walker that needs a smaller ball.
namespace {

__device__ __forceinline__ void ball_normals(const kmc::PhiloxKeys &ks, unsigned walker, unsigned pair, unsigned kj,
                                             double &z0, double &z1) {
    kmc::philox_normals(ks, walker, pair, kj, 0x4D540000u, z0, z1);
}

// out[i][c] = the standard normals of walker widx[i] (or w0 + i), try (k, j)
__global__ void ball_randn_kernel(kmc::PhiloxKeys ks, const unsigned *__restrict__ widx, long long w0, long long n, int k,
                                  int j, int d, double *__restrict__ out) {
    const int npair = (d + 1) / 2;
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * npair) return;
    const long long i = e / npair;
    const int pr = (int)(e - i * npair);
    const unsigned w = widx ? widx[i] : (unsigned)(w0 + i);
    double z0, z1;
    ball_normals(ks, w, (unsigned)pr, ((unsigned)k << 16) | (unsigned)j, z0, z1);
    out[i * d + 2 * pr] = z0;
    if (2 * pr + 1 < d) out[i * d + 2 * pr + 1] = z1;
}

// candidates of the pending walkers: tmp = theta0 .+ randn(npara) .* ball_radius  (:328-332; mul, then add, no FMA)
__global__ void ball_candidates_kernel(kmc::PhiloxKeys ks, const unsigned *__restrict__ widx, long long n, int k, int j,
                                       int d, const double *__restrict__ th0, const double *__restrict__ br,
                                       double *__restrict__ cand) {
    const int npair = (d + 1) / 2;
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * npair) return;
    const long long i = e / npair;
    const int pr = (int)(e - i * npair);
    double z0, z1;
    ball_normals(ks, widx[i], (unsigned)pr, ((unsigned)k << 16) | (unsigned)j, z0, z1);
    const int c = 2 * pr;
    cand[i * d + c] = kmc::dadd(th0[c], kmc::dmul(z0, br[c]));
    if (c + 1 < d) cand[i * d + c + 1] = kmc::dadd(th0[c + 1], kmc::dmul(z1, br[c + 1]));
}

// :338  accepted iff logp > -Inf (NaN is not): copy the row, else the walker stays pending
__global__ void ball_accept_kernel(const double *__restrict__ cand, const double *__restrict__ lp,
                                   const unsigned *__restrict__ widx, long long n, int d, double *__restrict__ out,
                                   unsigned char *__restrict__ found, unsigned *__restrict__ pend_next,
                                   unsigned *__restrict__ npend_next) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned w = widx[i];
    if (lp[i] > -CUDART_INF) {
        for (int c = 0; c < d; ++c) out[(size_t)w * d + c] = cand[i * d + c];
        found[w] = 1;
    } else {
        pend_next[atomicAdd(npend_next, 1u)] = w;
    }
}

__global__ void iota_kernel(unsigned *__restrict__ a, long long n, unsigned first) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = first + (unsigned)i;
}

__global__ void min_u32_kernel(const unsigned *__restrict__ a, long long n, unsigned *__restrict__ out) {
    unsigned m = 0xFFFFFFFFu;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        m = min(m, a[i]);
    for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMin(out, m);
}

__global__ void found_clear_kernel(unsigned char *__restrict__ found, long long first, long long n) {
    const long long i = first + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) found[i] = 0;
}

// per-block counts / ordered rows of the found walkers (the ordered compaction of the squash keep list)
__global__ void __launch_bounds__(kKeepBlock) found_count_kernel(const unsigned char *__restrict__ found, long long n,
                                                                 unsigned *__restrict__ blk_cnt) {
    const long long w = (long long)blockIdx.x * kKeepBlock + threadIdx.x;
    compact_count(w < n && found[w], blk_cnt);
}
__global__ void __launch_bounds__(kKeepBlock) found_gather_kernel(const unsigned char *__restrict__ found, long long n, int d,
                                                                  const unsigned *__restrict__ blk_off,
                                                                  const double *__restrict__ rows, double *__restrict__ out) {
    const long long w = (long long)blockIdx.x * kKeepBlock + threadIdx.x;
    const bool keep = w < n && found[w];
    const size_t o = (size_t)compact_slot(keep, blk_off) * d;
    if (keep)
        for (int c = 0; c < d; ++c) out[o + c] = rows[(size_t)w * d + c];
}

}  // namespace

extern "C" {

int32_t kmc_ball_randn(uint64_t seed, int64_t walker0, int64_t nwalkers, int32_t k, int32_t j, int32_t d, int32_t device,
                       double *out) {
    if (nwalkers < 0 || d < 1 || k < 1 || j < 1 || k > 0xFFFF || j > 0xFFFF || (nwalkers > 0 && !out))
        return fail(KMC_ERR_INVALID, "bad argument");
    if (nwalkers == 0) return KMC_OK;
    CU_TRY(cudaSetDevice(device));
    DevBuf<double> dz;
    CU_TRY(dev_alloc(dz, sizeof(double) * nwalkers * d, device));
    const long long ne = nwalkers * ((d + 1) / 2);
    ball_randn_kernel<<<(unsigned)((ne + 255) / 256), 256>>>(kmc::philox_keys(seed), nullptr, walker0, nwalkers, k, j, d,
                                                             dz.get());
    CU_TRY(cudaMemcpy(out, dz.get(), sizeof(double) * nwalkers * d, cudaMemcpyDeviceToHost));
    return KMC_OK;
}

int32_t kmc_make_theta0s(kmc_density_t density, const double *theta0, const double *ball_radius, int64_t nwalkers,
                         int32_t ball_radius_halfing_steps, int32_t ntries, uint64_t seed, double *out, int64_t *nfound) {
    if (!density || !theta0 || !ball_radius || !nfound || nwalkers < 0 || (nwalkers > 0 && !out))
        return fail(KMC_ERR_INVALID, "bad argument");
    if (ntries < 1 || ntries > 0xFFFF || ball_radius_halfing_steps < 1 || ball_radius_halfing_steps > 0xFFFF)
        return fail(KMC_ERR_INVALID, "ntries and ball_radius_halfing_steps must be in [1, 65535]");
    if (nwalkers >= (1LL << 32)) return fail(KMC_ERR_INVALID, "too many walkers");
    *nfound = 0;
    if (nwalkers == 0) return KMC_OK;
    const int d = density->d, dev = density->device;
    const long long nw = nwalkers;
    CU_TRY(cudaSetDevice(dev));
    const kmc::PhiloxKeys ks = kmc::philox_keys(seed);
    std::vector<double> br(ball_radius, ball_radius + d);

    DevBuf<double> d_th0, d_br, d_cand, d_lp, d_rows, d_out;
    DevBuf<unsigned> d_pend[2], d_cnt, d_blk;
    DevBuf<unsigned char> d_found;
    BatchScratch sc;
    const long long nblk = (nw + kKeepBlock - 1) / kKeepBlock;
    CU_TRY(dev_alloc(d_th0, sizeof(double) * d, dev));
    CU_TRY(dev_alloc(d_br, sizeof(double) * d, dev));
    CU_TRY(dev_alloc(d_cand, sizeof(double) * nw * d, dev));
    CU_TRY(dev_alloc(d_lp, sizeof(double) * nw, dev));
    CU_TRY(dev_alloc(d_rows, sizeof(double) * nw * d, dev));
    CU_TRY(dev_alloc(d_pend[0], sizeof(unsigned) * nw, dev));
    CU_TRY(dev_alloc(d_pend[1], sizeof(unsigned) * nw, dev));
    CU_TRY(dev_alloc(d_cnt, sizeof(unsigned) * 2, dev));
    CU_TRY(dev_alloc(d_blk, sizeof(unsigned) * 2 * nblk, dev));
    CU_TRY(dev_alloc(d_found, (size_t)nw, dev));
    CU_TRY(cudaMemcpy(d_th0.get(), theta0, sizeof(double) * d, cudaMemcpyHostToDevice));
    CU_TRY(cudaMemset(d_found.get(), 0, (size_t)nw));

    // one batched try (k, j) of the walkers in d_pend[cur][0..np): candidates -> plugin -> accept / stay pending
    auto try_round = [&](int cur, long long np, int k, int j, unsigned *np_next) -> cudaError_t {
        cudaError_t e = cudaMemset(d_cnt.get(), 0, sizeof(unsigned));
        if (e != cudaSuccess) return e;
        const long long ne = np * ((d + 1) / 2);
        ball_candidates_kernel<<<(unsigned)((ne + 255) / 256), 256>>>(ks, d_pend[cur].get(), np, k, j, d, d_th0.get(),
                                                                      d_br.get(), d_cand.get());
        e = eval_on_device(*density, d_cand.get(), np, d_lp.get(), sc, nullptr);  // :334-336 through the plugin
        if (e != cudaSuccess) return e;
        ball_accept_kernel<<<(unsigned)((np + 255) / 256), 256>>>(d_cand.get(), d_lp.get(), d_pend[cur].get(), np, d,
                                                                  d_rows.get(), d_found.get(), d_pend[cur ^ 1].get(),
                                                                  d_cnt.get());
        return cudaMemcpy(np_next, d_cnt.get(), sizeof(unsigned), cudaMemcpyDeviceToHost);
    };

    long long i0 = 0;
    while (i0 < nw) {  // :323 walkers i0.. with the CURRENT ball radius
        CU_TRY(cudaMemcpy(d_br.get(), br.data(), sizeof(double) * d, cudaMemcpyHostToDevice));
        long long np = nw - i0;
        int cur = 0;
        iota_kernel<<<(unsigned)((np + 255) / 256), 256>>>(d_pend[0].get(), np, (unsigned)i0);
        for (int j = 1; j <= ntries && np > 0; ++j) {  // k = 1: radius factor 1/2^0 = 1  (:326-327)
            unsigned nxt = 0;
            CU_TRY(try_round(cur, np, 1, j, &nxt));
            np = nxt;
            cur ^= 1;
        }
        if (np == 0) break;
        // the first walker whose k = 1 tries all failed: the reference now shrinks the ball for it AND, because the
        // radius is never reset (:326), for every later walker -- which must therefore be redone
        unsigned f = 0xFFFFFFFFu;
        CU_TRY(cudaMemset(d_cnt.get() + 1, 0xFF, sizeof(unsigned)));
        min_u32_kernel<<<(unsigned)std::min<long long>((np + 255) / 256, 1184), 256>>>(d_pend[cur].get(), np,
                                                                                        d_cnt.get() + 1);
        CU_TRY(cudaMemcpy(&f, d_cnt.get() + 1, sizeof(unsigned), cudaMemcpyDeviceToHost));
        if ((long long)f + 1 < nw)
            found_clear_kernel<<<(unsigned)((nw - f - 1 + 255) / 256), 256>>>(d_found.get(), (long long)f + 1, nw);
        bool got = false;
        for (int k = 2; k <= ball_radius_halfing_steps && !got; ++k) {  // :324
            for (int c = 0; c < d; ++c) br[c] = br[c] * (1.0 / std::pow(2.0, k - 1));  // :326 cumulative
            CU_TRY(cudaMemcpy(d_br.get(), br.data(), sizeof(double) * d, cudaMemcpyHostToDevice));
            for (int j = 1; j <= ntries && !got; ++j) {
                unsigned nxt = 0;
                CU_TRY(cudaMemcpy(d_pend[0].get(), &f, sizeof(unsigned), cudaMemcpyHostToDevice));
                CU_TRY(try_round(0, 1, k, j, &nxt));
                got = nxt == 0;
            }
        }
        i0 = (long long)f + 1;
    }

    // :348  the found walkers, in walker order (fewer than nwalkers if some walker exhausted every try)
    found_count_kernel<<<(unsigned)nblk, kKeepBlock>>>(d_found.get(), nw, d_blk.get());
    long long nf = 0;
    if (const int32_t rc = compact_offsets(d_blk.get(), nblk, nullptr, nf); rc != KMC_OK) return rc;
    if (nf > 0) {
        CU_TRY(dev_alloc(d_out, sizeof(double) * nf * d, dev));
        found_gather_kernel<<<(unsigned)nblk, kKeepBlock>>>(d_found.get(), nw, d, d_blk.get() + nblk, d_rows.get(),
                                                            d_out.get());
        CU_TRY(cudaMemcpy(out, d_out.get(), sizeof(double) * nf * d, cudaMemcpyDeviceToHost));
    }
    CU_TRY(cudaStreamSynchronize(nullptr));  // the blocks go back to the cache idle (nf = 0: the offsets' upload)
    CU_TRY(cudaGetLastError());
    *nfound = nf;
    return KMC_OK;
}

}  // extern "C"
