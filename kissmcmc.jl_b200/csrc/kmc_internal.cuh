// kmc_internal.cuh -- host-side declarations shared by the translation units of libkissmcmc_cuda.so
// (kmc_api.cu: handles, dispatch, run; kmc_aux.cu: multi-GPU, squash, make_theta0s, g-distribution helpers).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "../../include/kissmcmc_cuda.h"
#include "kmc_batched.cuh"
#include "kmc_ops.cuh"
#include "kmc_push.cuh"

namespace kmc_host {

// status + thread-local message (kmc_last_error)
int32_t fail(int32_t code, const char *fmt, ...);
const std::string &last_error();

// per-device cache of freed device blocks (kmc_trim releases them)
cudaError_t dev_alloc_raw(void **out, size_t bytes, int device);
template <typename T>
cudaError_t dev_alloc(T **out, size_t bytes, int device) {
    return dev_alloc_raw(reinterpret_cast<void **>(out), bytes, device);
}
void dev_free(void *p);
void cache_trim();

// A device block owned by its scope: it goes back to the cache when the owner is destroyed, so every user must have
// synchronised the block's stream by then.
struct DevFree {
    void operator()(void *p) const { dev_free(p); }
};
template <typename T>
using DevBuf = std::unique_ptr<T, DevFree>;

template <typename T>
cudaError_t dev_alloc(DevBuf<T> &b, size_t bytes, int device) {
    T *p = nullptr;
    const cudaError_t e = dev_alloc(&p, bytes, device);
    b.reset(p);
    return e;
}

// Grows b, which holds `have` bytes, to at least `need` bytes; the contents are not kept.
template <typename T>
cudaError_t reserve(DevBuf<T> &b, size_t &have, size_t need, int device) {
    if (need <= have) return cudaSuccess;
    b.reset();
    have = 0;
    const cudaError_t e = dev_alloc(b, need, device);
    if (e != cudaSuccess) return e;
    have = need;
    return cudaSuccess;
}

struct BatchScratch {
    DevBuf<double> part;  // logistic: partial sums [chunks][npts]
    size_t bytes = 0;
    DevBuf<__nv_bfloat16> pieces;  // tcgen05 path: theta split into 3 bf16 pieces [3][wpad][d]
    size_t pieces_bytes = 0;
};


}  // namespace kmc_host

#define CU_TRY(expr)                                                                            \
    do {                                                                                        \
        cudaError_t e_ = (expr);                                                                \
        if (e_ != cudaSuccess)                                                                  \
            return kmc_host::fail(KMC_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_),   \
                        __FILE__, __LINE__);                                                    \
    } while (0)


struct kmc_density_s {
    int kind = -1;
    int d = 0;
    int device = 0;
    std::vector<double> params;  // also the by-value kernel argument (padded to >= 1 double)
    kmc_host::Ops ops;
    double *d_params = nullptr;  // batched plugins: parameters in device memory
    float *d_X = nullptr, *d_y = nullptr;  // logistic: data
    long long ndata = 0;
    // logistic on tcgen05 (kmc_tc.cuh): bf16 copy of X, X^T y, TMA map of X
    bool tc_ok = false, tc_on = false;  // tensor-core paths are approximate (stated tolerances): always opt-in
    __nv_bfloat16 *d_Xbf = nullptr;
    double *d_xty = nullptr;
    CUtensorMap mapX;
    int nsm = 148;
    int kp = 32;  // logistic on tcgen05: d zero-padded to the GEMM's K (32 or 64)
    // wide Gaussian on tcgen05: matrix A split into 3 bf16 pieces [3][128][128], TMA map
    __nv_bfloat16 *d_Abf = nullptr;
    int fused_variant = 2;       // dense Gaussian, launch_mode 0: 2 = K2G (matrix in TMEM, default), 1 = K2F (matrix in shared memory)
    CUtensorMap mapA;
    double *d_At = nullptr;  // FP64 kernel: A transposed and padded to 128 rows, [d][128]

    bool tc() const { return tc_ok && tc_on; }  // the tcgen05 path is available and opted in
};


struct kmc_sampler_s {
    kmc_density_s *dn = nullptr;
    kmc_emcee_opts opts{};
    long long nw = 0, nhalf = 0, ns = 0;
    int d = 0;
    long long hdone = 0;       // half-steps completed (2 per outer iteration)
    long long sbeg = 0, scnt = 0;  // shard: positions of each half this sampler updates
    long long nl = 0;          // walkers this sampler stores chains for (2*scnt)
    double *x = nullptr, *lp = nullptr, *chain_x = nullptr, *chain_lp = nullptr;
    unsigned *nacc = nullptr;
    unsigned long long *barrier = nullptr;
    unsigned long long bar_base = 0;
    long long *rp_partner = nullptr;
    double *rp_z = nullptr, *rp_u = nullptr;
    long long rp_t0 = 0, rp_niters = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    bool timed = false;
    long long last_launches = 0;
    int nsm = 0;
    unsigned grid = 1, per_cta = 1, block = 32;  // persistent launch geometry
    size_t smem_bytes = 0;
    bool use_smem = false;           // owned state is shared-memory resident (emcee_smem_kernel)
    bool use_bulk = false;           // bulk (TMA) general kernel (emcee_bulk_kernel)
    unsigned long long *scratch = nullptr;  // 4 x 8 bytes for the statistics kernels
    kmc::BatchBuf bb{};                     // batched plugins: proposals of the active shard
    // peer mode
    int npeers = 0, rank = 0;
    const double *peer_x[8] = {};
    unsigned long long *peer_flags[8] = {};
    unsigned long long *flags = nullptr;    // this rank's flag array [8]
    unsigned long long epoch = 0;
    std::vector<void *> ipc_opened;
    kmc_host::BatchScratch bsc;
    // local layout of x / lp / nacc: rows held, offset of half 1, offset of this sampler's slice inside a half
    long long nstate = 0, hoff = 0, loff = 0;
    // push mode (KMC_EXCHANGE_PUSH, kmc_push.cuh): positions + receive ring + chunk flags in one window allocation
    bool push = false, attached = false;
    unsigned char *window = nullptr;
    size_t win_flags = 0, win_recv = 0, win_x = 0, win_bytes = 0;  // byte offsets inside the window (same on every rank)
    unsigned long long *task_ctr = nullptr;
    unsigned *notes = nullptr;  // push exchange: the publisher CTA's inbox (one note per push task)
    int G = 1;
    unsigned chunk = 0, rounds = 0, nchunks = 0, cap = 0, lag = 0;
    double *peer_recv[8] = {};
    int share = 1;  // sub-samplers sharing this device (kmc_emcee_create_multi with a repeated ordinal)
    // Metropolis handle (kmc_metropolis_create): nw = nl = nstate = chains, scnt = chains (one "half"), steps in tdone
    bool metro = false;
    long long tdone = 0;
    std::vector<double> sigma;     // [d] proposal scales: the fused kernel's by-value argument
    double *d_sigma = nullptr;     // batched plugins: the same in device memory
    double *rp_n = nullptr;        // replay normals [steps][chains][d] (rp_u holds the uniforms)
    // correlated proposal (kmc_metropolis_create_chol): y = x + L z
    bool chol = false;
    std::vector<double> chol_packed;  // [d (d + 1) / 2] L by rows: the fused kernel's by-value argument
    double *d_chol = nullptr;         // batched plugins: L [d][d] in device memory
    double *d_z = nullptr;            // batched plugins: the step's normals [chains][d]
};


namespace kmc_host {

// Wire rank r's window (base address as seen from this sampler's device) into the push kernel's peer tables.
inline void push_set_peer(kmc_sampler_s *s, int r, unsigned char *base) {
    s->peer_recv[r] = reinterpret_cast<double *>(base + s->win_recv);
    s->peer_flags[r] = reinterpret_cast<unsigned long long *>(base + s->win_flags);
    s->peer_x[r] = reinterpret_cast<const double *>(base + s->win_x);
}

// Task hand-out of the push kernel.  push_lag > 0: ORDERED, update(c, *) follows push(c + lag, *); push_lag = 0: ordered
// with the library's lag = 5/16 of the chunks (measured on 2 / 4 / 8 B200s with the 2^24-walker 10-D ensemble: the best
// lags were 2048 of 8192, 512 of 2048 and 384 of 1024 chunks -- a flag reaches the consumer ~25 us after its push, and
// everything before and after the overlap window is still useful work: pushes first, updates last); push_lag = -1:
// ADAPTIVE (two counters, an update is taken when its flags are seen set, else a push; returned as lag 0).
inline unsigned push_default_lag(unsigned nchunks, int push_lag) {
    if (push_lag < 0) return 0u;
    unsigned lag = push_lag > 0 ? (unsigned)push_lag : (5u * nchunks + 15u) / 16u;
    if (lag < 1u) lag = 1u;
    return lag < nchunks ? lag : nchunks;
}

// Batched log-density of npts device-resident points with the density's plugin (any plugin), on stream st.
cudaError_t eval_on_device(const kmc_density_s &dn, const double *X, long long npts, double *out, BatchScratch &sc,
                           cudaStream_t st);
// Kernels eval_on_device launches for this density.
int eval_launches(const kmc_density_s &dn);

// Walker-major copy of the stored chains to the host: thetas [nk][ns][d] and logp [nk][ns] (either may be NULL) for
// the stored walkers idx[0, nk), or [0, nk) if idx is NULL, staged through <= 64 MiB.  Synchronises the stream once.
int32_t chain_gather(kmc_sampler_s *s, const unsigned *idx, long long nk, double *thetas, double *logp);

// Complete samples stored so far per walker: the thinning clock after the iterations run (Metropolis: tdone steps;
// emcee: hdone / 2, so an iteration with one half-step left adds no sample).  The store is sample-major, so they are
// its first stored_samples(s) * nl rows; the rest of the ns planned samples hold whatever the block held before.
inline long long stored_samples(const kmc_sampler_s *s) {
    const long long t = s->metro ? s->tdone : s->hdone / 2;
    return kmc::ThinClock<>::at(t, s->opts.nburnin_walker, s->opts.nthin).sidx;
}

// A sampler under construction, deleted by kmc_emcee_destroy: every exit of a create call frees what was allocated.
using SamplerPtr = std::unique_ptr<kmc_sampler_s, int32_t (*)(kmc_sampler_t)>;

// Device state of both samplers, from the sizes the create call set (nstate, nl, ns, scnt): the stream and the timing
// events, x (a push sampler's x already lies in its window), lp, zeroed nacc, the statistics scratch, the chain store,
// the batched plugins' proposal buffers, theta0 and its log-densities.  The caller synchronises the stream once its
// own buffers are set up.
int32_t sampler_init(kmc_sampler_s *s, const double *theta0s);

// kmc_emcee_run of a Metropolis handle (kmc_metro.cu).
int32_t metro_run(kmc_sampler_s *s, long long nsteps);

// The run of both samplers over [done, done + n), n clamped to the `total` steps left (half-steps for emcee, per = 2 of
// them per replay iteration; Metropolis steps, per = 1).  path(t0, t1, launches) enqueues the range, recording ev0 where
// its timed window starts, and reports its kernel launches; the run then closes the window and advances `done`.
template <class Path>
int32_t run_range(kmc_sampler_s *s, long long &done, long long total, long long n, int per, Path &&path) {
    const long long remaining = total - done;
    if (n < 0 || n > remaining) n = remaining;
    s->last_launches = 0;
    s->timed = false;
    if (n <= 0) return KMC_OK;
    const long long t0 = done, t1 = done + n;
    if (s->opts.mode == KMC_MODE_REPLAY && (t0 < per * s->rp_t0 || t1 > per * (s->rp_t0 + s->rp_niters)))
        return fail(KMC_ERR_STATE, "replay draws cover %s [%lld, %lld), asked to run %s [%lld, %lld)",
                    per == 2 ? "iterations" : "steps", s->rp_t0, s->rp_t0 + s->rp_niters, per == 2 ? "half-steps" : "steps",
                    t0, t1);
    CU_TRY(cudaSetDevice(s->opts.device));
    long long launches = 0;
    const int32_t rc = path(t0, t1, launches);
    if (rc != KMC_OK) return rc;
    s->last_launches = launches;
    CU_TRY(cudaEventRecord(s->ev1, s->stream));
    s->timed = true;
    done = t1;
    return KMC_OK;
}

}  // namespace kmc_host
