// kmc_api.cu -- C-ABI of libkissmcmc_cuda.so (see include/kissmcmc_cuda.h).
//
// Host-side runtime of the emcee hot path: handle management, argument checks that mirror
// the reference's asserts (src/samplers.jl:200-205), kernel dispatch over the log-density
// plugin registry, the thinned chain store and result copy-out.  No CPU fallback exists:
// every compute entry point needs a CUDA device.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "kmc_internal.cuh"
#include "kmc_tc.cuh"
#include "kmc_fused_gauss.cuh"
#include "kmc_fused_gauss2.cuh"

namespace kmc_host {

namespace {
thread_local std::string g_err;
}

const std::string &last_error() { return g_err; }

int32_t fail(int32_t code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}

// ------------------------------------------------------------------ device memory cache
// cudaMalloc / cudaFree cost milliseconds once pinned host memory and other contexts are
// mapped; samplers are created and destroyed per emcee() call, so freed blocks are kept in a
// small per-device cache and reused by exact size.  kmc_trim() releases them.
namespace {
struct DevCache {
    std::mutex mu;
    std::multimap<std::pair<int, size_t>, void *> free_blocks;  // (device, bytes) -> ptr
    std::map<void *, std::pair<int, size_t>> live;
    size_t cached_bytes = 0;
    static constexpr size_t kMaxCached = (size_t)2 << 30;  // total kept; kmc_trim() releases everything
    static constexpr size_t kMaxBlock = (size_t)512 << 20;   // larger blocks (long chains) always go back to the driver
} g_cache;
}  // namespace

cudaError_t dev_alloc_raw(void **out, size_t bytes, int device) {
    {
        std::lock_guard<std::mutex> lk(g_cache.mu);
        auto it = g_cache.free_blocks.find({device, bytes});
        if (it != g_cache.free_blocks.end()) {
            *out = it->second;
            g_cache.free_blocks.erase(it);
            g_cache.cached_bytes -= bytes;
            g_cache.live[*out] = {device, bytes};
            return cudaSuccess;
        }
    }
    cudaError_t e = cudaMalloc(out, bytes);
    if (e != cudaSuccess) {  // give cached blocks back and retry once
        cudaGetLastError();
        std::lock_guard<std::mutex> lk(g_cache.mu);
        for (auto &kv : g_cache.free_blocks) cudaFree(kv.second);
        g_cache.free_blocks.clear();
        g_cache.cached_bytes = 0;
        e = cudaMalloc(out, bytes);
    }
    if (e != cudaSuccess) {
        cudaGetLastError();  // the failure is returned here, not left for a later cudaGetLastError check to report
        return e;
    }
    std::lock_guard<std::mutex> lk(g_cache.mu);
    g_cache.live[*out] = {device, bytes};
    return e;
}

void dev_free(void *p) {
    if (!p) return;
    std::lock_guard<std::mutex> lk(g_cache.mu);
    auto it = g_cache.live.find(p);
    if (it == g_cache.live.end()) {
        cudaFree(p);
        return;
    }
    const auto key = it->second;
    g_cache.live.erase(it);
    if (key.second > DevCache::kMaxBlock || g_cache.cached_bytes + key.second > DevCache::kMaxCached) {
        cudaFree(p);
        return;
    }
    g_cache.free_blocks.insert({key, p});
    g_cache.cached_bytes += key.second;
}

namespace {

constexpr int kLogisticMaxD = 512;

bool find_ops(int kind, int d, Ops &o) {
    switch (kind) {
        case kmc::KIND_EXPONENTIAL:
            if (ops_exponential(d, o)) return true;
            if (d > 4096) return false;
            o = Ops();
            o.batch = BATCH_EXP;  // any other dimension: batched half-step with a thread-per-point sum
            o.nparams = 0;
            return true;
        case kmc::KIND_GAUSSIAN:
            if (ops_gaussian(d, o)) return true;
            if (d > kmc::kHugeMaxD) return false;
            o = Ops();
            o.batch = BATCH_GAUSSIAN;  // dense contraction over the active half (d > 128: FP64 from L2, no tensor-core path)
            o.nparams = d + d * d + 1;
            return true;
        case kmc::KIND_LOGISTIC:
            if (d > kLogisticMaxD) return false;  // 32 points' theta in shared memory; tcgen05 path up to d = 64
            o = Ops();
            o.batch = BATCH_LOGISTIC;
            o.nparams = 1;
            return true;
        case kmc::KIND_ROSENBROCK: return ops_rosenbrock(d, o);
        case kmc::KIND_LOGNORMAL: return ops_lognormal(d, o);
        default: return false;
    }
}

int kind_of(const char *name) {
    if (!name) return -1;
    if (!strcmp(name, "exponential")) return kmc::KIND_EXPONENTIAL;
    if (!strcmp(name, "rosenbrock")) return kmc::KIND_ROSENBROCK;
    if (!strcmp(name, "gaussian")) return kmc::KIND_GAUSSIAN;
    if (!strcmp(name, "lognormal")) return kmc::KIND_LOGNORMAL;
    if (!strcmp(name, "logistic")) return kmc::KIND_LOGISTIC;
    return -1;
}

// CTAs of `kern` resident per SM, or 0 if the query fails (its error is cleared).
int occupancy(const void *kern, int block, size_t smem) {
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kern, block, smem) == cudaSuccess) return n;
    cudaGetLastError();
    return 0;
}

// Batched log-density of npts device-resident points (K4 for the batched plugins; stage 2 of
// the batched half-step).  `scratch` holds the logistic partial sums ([chunks][npts]).
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *ptr = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(ptr);
    }
    return fn;
}

// 2-D bf16 row-major [rows][128] tensor, box = [box_rows][64] (128 B), 128-byte swizzle
bool make_map_bf16_k128(CUtensorMap *map, const void *base, unsigned long long rows, unsigned box_rows) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return false;
    const cuuint64_t dims[2] = {128, rows};
    const cuuint64_t strides[1] = {256};
    const cuuint32_t box[2] = {64, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// 2-D bf16 row-major [rows][kp] tensor (kp = 32 or 64), box = [box_rows][kp], swizzle = the row size in bytes
// (64-byte / 128-byte; K-major UMMA operand)
bool make_map_bf16_k(CUtensorMap *map, const void *base, unsigned long long rows, unsigned box_rows, int kp) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return false;
    const cuuint64_t dims[2] = {(cuuint64_t)kp, rows};
    const cuuint64_t strides[1] = {(cuuint64_t)kp * 2};
    const cuuint32_t box[2] = {(cuuint32_t)kp, box_rows};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, kp == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

constexpr int kLogitChunks = 64;

struct TcPlan {
    kmc::tc::LogitParams lp;
    unsigned grid;
};

TcPlan tc_plan(const kmc_density_s &dn, long long npts) {
    TcPlan pl{};
    pl.lp.W = npts;
    pl.lp.N = dn.ndata;
    pl.lp.mtiles = (int)((npts + kmc::tc::BM - 1) / kmc::tc::BM);
    pl.lp.ntiles = (int)((dn.ndata + kmc::tc::BN - 1) / kmc::tc::BN);
    int nch = (dn.nsm * 8 + pl.lp.mtiles - 1) / pl.lp.mtiles;
    nch = std::max(1, std::min(nch, std::min(pl.lp.ntiles, 512)));
    pl.lp.tiles_per_chunk = (pl.lp.ntiles + nch - 1) / nch;
    pl.lp.nchunks = (pl.lp.ntiles + pl.lp.tiles_per_chunk - 1) / pl.lp.tiles_per_chunk;
    pl.lp.wpad = (long long)pl.lp.mtiles * kmc::tc::BM;
    pl.grid = (unsigned)std::min<long long>((long long)pl.lp.mtiles * pl.lp.nchunks, dn.nsm);
    return pl;
}

cudaError_t batch_scratch_reserve(BatchScratch &sc, const kmc_density_s &dn, long long npts) {
    if (dn.ops.batch != BATCH_LOGISTIC) return cudaSuccess;
    const bool tcp = dn.tc();
    const TcPlan pl = tcp ? tc_plan(dn, npts) : TcPlan{};
    if (tcp) {
        const size_t pneed = sizeof(__nv_bfloat16) * kmc::tc::PIECES * (size_t)pl.lp.wpad * dn.kp;
        const cudaError_t e = reserve(sc.pieces, sc.pieces_bytes, pneed, dn.device);
        if (e != cudaSuccess) return e;
    }
    const size_t need = sizeof(double) * (size_t)(tcp ? pl.lp.nchunks : kLogitChunks) * (size_t)npts;
    return reserve(sc.part, sc.bytes, need, dn.device);
}

cudaError_t gauss_pieces_reserve(BatchScratch &sc, const kmc_density_s &dn, long long npts) {
    const long long wpad = ((npts + kmc::tc::BM - 1) / kmc::tc::BM) * kmc::tc::BM;
    const size_t pneed = sizeof(__nv_bfloat16) * kmc::tc::PIECES * (size_t)wpad * kmc::tc::GK;
    return reserve(sc.pieces, sc.pieces_bytes, pneed, dn.device);
}

// The tcgen05 Mahalanobis GEMM on centred bf16 pieces [3][wpad][128] already in sc.pieces.
cudaError_t launch_gauss_tc(const kmc_density_s &dn, BatchScratch &sc, long long npts, double *out, cudaStream_t st) {
    const int d = dn.d;
    kmc::tc::GaussParams gp{};
    gp.W = npts;
    gp.mtiles = (int)((npts + kmc::tc::BM - 1) / kmc::tc::BM);
    gp.wpad = (long long)gp.mtiles * kmc::tc::BM;
    gp.d = d;
    gp.lognorm = dn.params[d + (size_t)d * d];
    gp.out = out;
    CUtensorMap mapC;
    if (!make_map_bf16_k128(&mapC, sc.pieces.get(), (unsigned long long)kmc::tc::PIECES * gp.wpad, kmc::tc::BM))
        return cudaErrorInvalidValue;
    const size_t smem = sizeof(kmc::tc::GaussSmem) + 1024;
    cudaError_t e = cudaFuncSetAttribute(kmc::tc::gaussian_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) return e;
    const unsigned grid = (unsigned)std::min<long long>(gp.mtiles, dn.nsm);
    kmc::tc::gaussian_tc_kernel<<<grid, kmc::tc::kGaussThreads, smem, st>>>(mapC, dn.mapA, gp);
    return cudaGetLastError();
}

cudaError_t launch_batch_logp(const kmc_density_s &dn, const double *X, long long npts, double *out,
                              BatchScratch &sc, cudaStream_t st) {
    const int d = dn.d;
    if (dn.ops.batch == BATCH_GAUSSIAN && dn.tc()) {  // tcgen05 Mahalanobis GEMM
        cudaError_t e = gauss_pieces_reserve(sc, dn, npts);
        if (e != cudaSuccess) return e;
        const long long wpad = ((npts + kmc::tc::BM - 1) / kmc::tc::BM) * kmc::tc::BM;
        const long long ne = wpad * kmc::tc::GK;
        kmc::tc::split_rows128_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(X, dn.d_params, sc.pieces.get(),
                                                                                    npts, wpad, d);
        return launch_gauss_tc(dn, sc, npts, out, st);
    }
    if (dn.ops.batch == BATCH_GAUSSIAN && d > kmc::kWideMaxD) {
        const int dpad = (d + 127) / 128 * 128;
        const size_t per_warp = sizeof(double) * (size_t)d * kmc::kWidePts;
        const int wpb = (int)std::max<size_t>(1, std::min<size_t>(kmc::kWideThreads / 32, (size_t)(200 * 1024) / per_warp));
        const size_t smem = per_warp * wpb;
        cudaError_t e = cudaFuncSetAttribute(kmc::gaussian_huge_logp_kernel,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        const long long ngroups = (npts + kmc::kWidePts - 1) / kmc::kWidePts;
        const unsigned grid = (unsigned)std::min<long long>((ngroups + wpb - 1) / wpb, 2LL * dn.nsm);
        kmc::gaussian_huge_logp_kernel<<<grid, wpb * 32, smem, st>>>(X, out, npts, d, dpad, dn.d_params, dn.d_At);
        return cudaGetLastError();
    }
    if (dn.ops.batch == BATCH_GAUSSIAN) {
        const size_t smem = sizeof(double) * ((size_t)d * 128 + (size_t)(kmc::kWideThreads / 32) * d * kmc::kWidePts);
        cudaError_t e = cudaFuncSetAttribute(kmc::gaussian_wide_logp_kernel,
                                             cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
        const long long ngroups = (npts + kmc::kWidePts - 1) / kmc::kWidePts;
        const int wpb = kmc::kWideThreads / 32;
        const unsigned grid = (unsigned)std::min<long long>((ngroups + wpb - 1) / wpb, dn.nsm);
        kmc::gaussian_wide_logp_kernel<<<grid, kmc::kWideThreads, smem, st>>>(X, out, npts, d, dn.d_params, dn.d_At);
        return cudaGetLastError();
    }
    if (dn.ops.batch == BATCH_EXP) {
        kmc::exponential_wide_logp_kernel<<<(unsigned)((npts + 255) / 256), 256, 0, st>>>(X, out, npts, d);
        return cudaGetLastError();
    }
    if (dn.ops.batch == BATCH_LOGISTIC && dn.tc()) {  // tcgen05 logits GEMM + fused softplus row sums
        cudaError_t e = batch_scratch_reserve(sc, dn, npts);
        if (e != cudaSuccess) return e;
        TcPlan pl = tc_plan(dn, npts);
        pl.lp.part = sc.part.get();
        const int kp = dn.kp;  // d zero-padded to the GEMM's K (32 or 64)
        const long long ne = pl.lp.wpad * kp;
        kmc::tc::split_theta_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(X, sc.pieces.get(), npts, pl.lp.wpad, d,
                                                                                       kp, 1.4426950408889634);
        CUtensorMap mapA;
        if (!make_map_bf16_k(&mapA, sc.pieces.get(), (unsigned long long)kmc::tc::PIECES * pl.lp.wpad, kmc::tc::BM, kp))
            return cudaErrorInvalidValue;
        if (kp == 32) {
            const size_t smem = sizeof(kmc::tc::Smem<32>) + 1024;
            e = cudaFuncSetAttribute(kmc::tc::logistic_tc_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            kmc::tc::logistic_tc_kernel<32><<<pl.grid, kmc::tc::kThreads, smem, st>>>(mapA, dn.mapX, pl.lp);
        } else {
            const size_t smem = sizeof(kmc::tc::Smem<64>) + 1024;
            e = cudaFuncSetAttribute(kmc::tc::logistic_tc_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            kmc::tc::logistic_tc_kernel<64><<<pl.grid, kmc::tc::kThreads, smem, st>>>(mapA, dn.mapX, pl.lp);
        }
        const double sg = dn.params[0];
        kmc::tc::logistic_tc_finish_kernel<<<(unsigned)((npts + 255) / 256), 256, 0, st>>>(
            X, sc.part.get(), dn.d_xty, out, npts, d, pl.lp.nchunks, 0.5 / (sg * sg));
        return cudaGetLastError();
    }
    if (dn.ops.batch == BATCH_LOGISTIC) {
        cudaError_t e = batch_scratch_reserve(sc, dn, npts);
        if (e != cudaSuccess) return e;
        const long long rows = (dn.ndata + kLogitChunks - 1) / kLogitChunks;
        const size_t smem = sizeof(double) * ((size_t)kmc::kLogitTile * d + 8 * kmc::kLogitTile);
        const dim3 grid((unsigned)((npts + kmc::kLogitTile - 1) / kmc::kLogitTile), kLogitChunks);
        if (smem > 48 * 1024) {
            e = cudaFuncSetAttribute(kmc::logistic_logp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        kmc::logistic_logp_kernel<<<grid, 256, smem, st>>>(X, sc.part.get(), npts, d, dn.d_X, dn.d_y, dn.ndata, rows);
        const double sg = dn.params[0];
        kmc::logistic_finish_kernel<<<(unsigned)((npts + 255) / 256), 256, 0, st>>>(X, sc.part.get(), out, npts, d,
                                                                                     kLogitChunks, 0.5 / (sg * sg));
        return cudaGetLastError();
    }
    return cudaErrorInvalidValue;
}

}  // namespace

cudaError_t eval_on_device(const kmc_density_s &dn, const double *X, long long npts, double *out, BatchScratch &sc,
                           cudaStream_t st) {
    if (dn.ops.batch) return launch_batch_logp(dn, X, npts, out, sc, st);
    long long nwl = npts;
    void *args[] = {(void *)&X, (void *)&out, &nwl, (void *)dn.params.data()};
    return cudaLaunchKernel(dn.ops.eval, dim3((unsigned)((npts + 255) / 256)), dim3(256), args, 0, st);
}

int eval_launches(const kmc_density_s &dn) {
    switch (dn.ops.batch) {
        case BATCH_GAUSSIAN: return dn.tc() ? 2 : 1;  // (split + GEMM) or the FP64 kernel
        case BATCH_LOGISTIC: return dn.tc() ? 3 : 2;  // (split + GEMM + finish) or (partial sums + finish)
        default: return 1;
    }
}

void cache_trim() {
    std::lock_guard<std::mutex> lk(g_cache.mu);
    for (auto &kv : g_cache.free_blocks) {
        cudaSetDevice(kv.first.first);
        cudaFree(kv.second);
    }
    g_cache.free_blocks.clear();
    g_cache.cached_bytes = 0;
}

int32_t sampler_init(kmc_sampler_s *s, const double *theta0s) {
    const int d = s->d, dev = s->opts.device;
    CU_TRY(cudaStreamCreateWithFlags(&s->own_stream, cudaStreamNonBlocking));
    s->stream = s->own_stream;
    CU_TRY(cudaEventCreate(&s->ev0));
    CU_TRY(cudaEventCreate(&s->ev1));
    if (!s->x) CU_TRY(dev_alloc(&s->x, sizeof(double) * s->nstate * d, dev));
    CU_TRY(dev_alloc(&s->lp, sizeof(double) * s->nstate, dev));
    CU_TRY(dev_alloc(&s->nacc, sizeof(unsigned) * s->nstate, dev));
    CU_TRY(dev_alloc(&s->scratch, 4 * sizeof(unsigned long long), dev));
    if (s->ns > 0) {
        CU_TRY(dev_alloc(&s->chain_x, sizeof(double) * s->ns * s->nl * d, dev));
        CU_TRY(dev_alloc(&s->chain_lp, sizeof(double) * s->ns * s->nl, dev));
    }
    CU_TRY(cudaMemsetAsync(s->nacc, 0, sizeof(unsigned) * s->nstate, s->stream));
    if (s->push) {  // only this shard's rows: its slice of half 0, then of half 1
        CU_TRY(cudaMemcpyAsync(s->x, theta0s + (size_t)s->sbeg * d, sizeof(double) * s->scnt * d,
                               cudaMemcpyHostToDevice, s->stream));
        CU_TRY(cudaMemcpyAsync(s->x + (size_t)s->scnt * d, theta0s + (size_t)(s->nhalf + s->sbeg) * d,
                               sizeof(double) * s->scnt * d, cudaMemcpyHostToDevice, s->stream));
    } else {  // deep copy
        CU_TRY(cudaMemcpyAsync(s->x, theta0s, sizeof(double) * s->nstate * d, cudaMemcpyHostToDevice, s->stream));
    }
    if (s->dn->ops.batch) {  // per-step buffers of the active shard: proposals, their log-densities, accept uniforms
        CU_TRY(dev_alloc(&s->bb.Y, sizeof(double) * s->scnt * d, dev));
        CU_TRY(dev_alloc(&s->bb.u, sizeof(double) * s->scnt, dev));
        CU_TRY(dev_alloc(&s->bb.p1, sizeof(double) * s->scnt, dev));
    }
    CU_TRY(eval_on_device(*s->dn, s->x, s->nstate, s->lp, s->bsc, s->stream));  // p0 = pdf(theta0), :209-210
    return KMC_OK;
}

int32_t chain_gather(kmc_sampler_s *s, const unsigned *idx, long long nk, double *thetas, double *logp) {
    const long long ns = s->ns, nl = s->nl;
    const int d = s->d;
    // walkers per staging chunk: <= 64 MiB of [wc][ns][d] doubles
    const long long wc = std::min(nk, std::max<long long>(32, (64LL << 20) / (sizeof(double) * ns * d)));
    DevBuf<double> stage;
    CU_TRY(dev_alloc(stage, sizeof(double) * wc * ns * d, s->opts.device));
    auto transpose = idx ? kmc::chain_transpose_kernel<true> : kmc::chain_transpose_kernel<false>;
    const dim3 blk(32, 8);
    for (long long w0 = 0; w0 < nk; w0 += wc) {
        const long long cur = std::min(wc, nk - w0);
        for (int what = 0; what < 2; ++what) {
            double *host = what == 0 ? thetas : logp;
            if (!host) continue;
            const int dd = what == 0 ? d : 1;
            const double *src = what == 0 ? s->chain_x : s->chain_lp;
            for (long long s0 = 0; s0 < ns; s0 += kmc::kTransposeMaxSamples) {
                const long long sc = std::min(kmc::kTransposeMaxSamples, ns - s0);
                const dim3 grd((unsigned)((cur + 31) / 32), (unsigned)((sc + 31) / 32), (unsigned)dd);
                transpose<<<grd, blk, 0, s->stream>>>(src, stage.get(), ns, nl, w0, cur, dd, s0, idx);
            }
            CU_TRY(cudaMemcpyAsync(host + w0 * ns * dd, stage.get(), sizeof(double) * cur * ns * dd,
                                   cudaMemcpyDeviceToHost, s->stream));
        }
    }
    CU_TRY(cudaStreamSynchronize(s->stream));
    CU_TRY(cudaGetLastError());
    return KMC_OK;
}

namespace {

// Half-steps [h0, h1) in p: the burn-in and thinning phase of h0 (returned too), and the barrier epochs used so far.
kmc::ThinClock<> set_range(kmc::RunParams &p, const kmc_sampler_s *s, long long h0, long long h1) {
    p.h0 = h0;
    p.h1 = h1;
    const auto clk = kmc::ThinClock<>::at(h0 >> 1, s->opts.nburnin_walker, p.nthin);
    p.n0 = clk.n;
    p.phase0 = clk.phase;
    p.sidx0 = clk.sidx;
    p.bar_base = s->bar_base;
    return clk;
}

// The emcee run paths.  Each enqueues half-steps [h0, h1) of p, recording ev0 where its timed window starts, advances the
// barrier bookkeeping of a persistent kernel and reports its kernel launches.

// Sharded ensemble, owner-computes pushes (kmc_push.cuh): one persistent kernel for the whole range.
int32_t run_push(kmc_sampler_s *s, kmc::RunParams &p, long long h0, long long h1, long long &launches) {
    if (s->G > 1 && !s->attached)
        return fail(KMC_ERR_STATE, "push exchange: attach the peers' windows first (kmc_emcee_window_attach)");
    kmc::PushParams q{};
    q.recv = reinterpret_cast<double *>(s->window + s->win_recv);
    q.flags = reinterpret_cast<unsigned long long *>(s->window + s->win_flags);
    for (int r = 0; r < s->G; ++r) {
        q.peer_recv[r] = s->peer_recv[r];
        q.peer_flags[r] = s->peer_flags[r];
        q.peer_x[r] = s->peer_x[r];
    }
    q.task_ctr = s->task_ctr;
    q.notes = s->notes;
    q.S = (unsigned)s->scnt;
    q.G = (unsigned)s->G;
    q.rank = (unsigned)s->rank;
    q.chunk = s->chunk;
    q.rounds = s->rounds;
    q.nchunks = s->nchunks;
    q.cap = s->cap;
    q.lag = s->lag;
    q.batch = 1;  // measured on 8 B200s (profiles/r2_call13.log, r2_call14.log): notes posted singly, as soon as the
    q.age = 2;    // newest message is two tasks old, beat every batched / later variant (flag latency gates the consumers)
    set_range(p, s, h0, h1);
    CU_TRY(cudaMemsetAsync(s->task_ctr, 0, 4 * sizeof(unsigned long long), s->stream));
    CU_TRY(cudaEventRecord(s->ev0, s->stream));
    void *args[] = {&p, &q, s->dn->params.data()};
    CU_TRY(cudaLaunchCooperativeKernel(s->dn->ops.run_push, dim3(s->grid), dim3(s->block), args, s->smem_bytes, s->stream));
    s->bar_base += (unsigned long long)(h1 - h0 - 1) * s->grid;
    launches = 1;
    return KMC_OK;
}

// Dense Gaussian on tcgen05, launch_mode 0: the whole range in one persistent fused kernel, K2G (fused_variant 2: the
// matrix resident in TMEM) or K2F (fused_variant 1: the matrix in shared memory).
int32_t run_fused_gauss(kmc_sampler_s *s, kmc::RunParams &p, long long h0, long long h1, long long &launches) {
    kmc_density_s &dn = *s->dn;
    const bool replay = s->opts.mode == KMC_MODE_REPLAY, k2g = dn.fused_variant == 2;
    CU_TRY(cudaEventRecord(s->ev0, s->stream));
    kmc::tc::Fused2Params f2{};
    f2.mu = dn.d_params;
    f2.apieces = reinterpret_cast<const unsigned *>(dn.d_Abf);
    f2.lognorm = dn.params[s->d + (size_t)s->d * s->d];
    f2.d = s->d;
    kmc::tc::FusedParams f1{f2.mu, f2.lognorm, f2.d};
    const void *kern = k2g ? (replay ? (const void *)kmc::tc::gaussian_fused2_kernel<true>
                                     : (const void *)kmc::tc::gaussian_fused2_kernel<false>)
                           : (replay ? (const void *)kmc::tc::gaussian_fused_kernel<true>
                                     : (const void *)kmc::tc::gaussian_fused_kernel<false>);
    const size_t smem = (k2g ? sizeof(kmc::tc::Fused2Smem) : sizeof(kmc::tc::FusedSmem)) + 1024;
    CU_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const long long ntiles = (s->scnt + kmc::tc::BM - 1) / kmc::tc::BM;
    const unsigned grid = (unsigned)std::min<long long>(ntiles, dn.nsm);
    set_range(p, s, h0, h1);
    void *args2[] = {&p, &f2}, *args1[] = {&dn.mapA, &p, &f1};
    CU_TRY(cudaLaunchCooperativeKernel(kern, dim3(grid), dim3(kmc::tc::kFusedThreads), k2g ? args2 : args1, smem, s->stream));
    s->bar_base += (unsigned long long)(h1 - h0 - 1) * grid;
    launches = 1;
    return KMC_OK;
}

// Batched plugins: propose -> batched log-density -> accept, per half-step.  The dense Gaussian on tcgen05 (launch_mode
// 1) writes no Y: the proposals go straight into bf16 pieces and accept recomputes the accepted rows.
int32_t run_batched(kmc_sampler_s *s, kmc::RunParams &p, long long h0, long long h1, long long &launches) {
    kmc_density_s &dn = *s->dn;
    const bool replay = s->opts.mode == KMC_MODE_REPLAY, gtc = dn.ops.batch == BATCH_GAUSSIAN && dn.tc();
    const unsigned grid = (unsigned)((s->scnt * 32 + 255) / 256);
    CU_TRY(cudaEventRecord(s->ev0, s->stream));
    if (gtc) CU_TRY(gauss_pieces_reserve(s->bsc, dn, s->scnt));
    const long long wpad = ((s->scnt + kmc::tc::BM - 1) / kmc::tc::BM) * kmc::tc::BM;
    const unsigned gridp = (unsigned)((wpad * 32 + 255) / 256);
    auto propose = replay ? kmc::propose_kernel<true> : kmc::propose_kernel<false>;
    auto accept = replay ? kmc::accept_kernel<true> : kmc::accept_kernel<false>;
    auto propose_pieces = replay ? kmc::propose_pieces_kernel<true> : kmc::propose_pieces_kernel<false>;
    auto accept_recompute = replay ? kmc::accept_recompute_kernel<true> : kmc::accept_recompute_kernel<false>;
    for (long long h = h0; h < h1; ++h) {
        const auto clk = set_range(p, s, h, h + 1);
        const int store = clk.store() ? 1 : 0;
        if (gtc) {
            propose_pieces<<<gridp, 256, 0, s->stream>>>(p, s->bb, h, s->d, dn.d_params, s->bsc.pieces.get(), wpad);
            CU_TRY(launch_gauss_tc(dn, s->bsc, s->scnt, s->bb.p1, s->stream));
            accept_recompute<<<grid, 256, 0, s->stream>>>(p, s->bb, h, s->d, clk.n, store, clk.sidx);
        } else {
            propose<<<grid, 256, 0, s->stream>>>(p, s->bb, h, s->d);
            CU_TRY(eval_on_device(dn, s->bb.Y, s->scnt, s->bb.p1, s->bsc, s->stream));
            accept<<<grid, 256, 0, s->stream>>>(p, s->bb, h, s->d, clk.n, store, clk.sidx);
        }
    }
    CU_TRY(cudaGetLastError());
    launches = (h1 - h0) * (gtc ? 3 : 2 + eval_launches(dn));
    return KMC_OK;
}

// Fused plugins, launch_mode 1: one walker per thread, one half-step per launch.
int32_t run_per_half(kmc_sampler_s *s, kmc::RunParams &p, long long h0, long long h1, long long &launches) {
    CU_TRY(cudaEventRecord(s->ev0, s->stream));
    const void *kern = s->dn->ops.run[s->opts.mode == KMC_MODE_REPLAY ? 1 : 0][0];
    const int blk = s->dn->ops.block >= 256 ? 256 : s->dn->ops.block;
    p.per_cta = (unsigned)blk;
    const unsigned grid = (unsigned)((s->scnt + blk - 1) / blk);
    void *args[] = {&p, s->dn->params.data()};
    for (long long h = h0; h < h1; ++h) {
        set_range(p, s, h, h + 1);
        CU_TRY(cudaLaunchKernel(kern, dim3(grid), dim3(blk), args, 0, s->stream));
    }
    launches = h1 - h0;
    return KMC_OK;
}

// Fused plugins, launch_mode 0: the whole range in one persistent kernel with the geometry chosen at creation.
int32_t run_persistent(kmc_sampler_s *s, kmc::RunParams &p, long long h0, long long h1, long long &launches) {
    const bool peer = s->npeers >= 1;
    CU_TRY(cudaEventRecord(s->ev0, s->stream));
    const void *kern = s->use_bulk ? s->dn->ops.run_bulk[peer ? 1 : 0]
                       : peer      ? s->dn->ops.run_peer
                                   : s->dn->ops.run[s->opts.mode == KMC_MODE_REPLAY ? 1 : 0][s->use_smem ? 1 : 0];
    set_range(p, s, h0, h1);
    void *args[] = {&p, s->dn->params.data()};
    CU_TRY(cudaLaunchCooperativeKernel(kern, dim3(s->grid), dim3(s->block), args,
                                       (s->use_bulk || (!peer && s->use_smem)) ? s->smem_bytes : 0, s->stream));
    s->bar_base += (unsigned long long)(h1 - h0 - 1) * s->grid * (peer ? 2 : 1);
    if (peer) s->epoch += (unsigned long long)(h1 - h0 - 1);
    launches = 1;
    return KMC_OK;
}

}  // namespace

}  // namespace kmc_host

using namespace kmc_host;

extern "C" {

int32_t kmc_version(void) { return 200; }

const char *kmc_last_error(void) { return last_error().c_str(); }

int32_t kmc_device_count(int32_t *count) {
    if (!count) return fail(KMC_ERR_INVALID, "count is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *count = 0;
        return fail(KMC_ERR_CUDA, "cudaGetDeviceCount failed: %s", cudaGetErrorString(e));
    }
    *count = n;
    return KMC_OK;
}

int32_t kmc_trim(void) {
    cache_trim();
    return KMC_OK;
}

int32_t kmc_density_create(const char *name, int32_t d, const double *params, int64_t nparams,
                           const void *data, int64_t data_bytes, int32_t device,
                           kmc_density_t *out) {
    if (!out) return fail(KMC_ERR_INVALID, "out is NULL");
    *out = nullptr;
    const int kind = kind_of(name);
    if (kind < 0) return fail(KMC_ERR_INVALID, "unknown log-density plugin '%s'", name ? name : "(null)");
    if (d < 1) return fail(KMC_ERR_INVALID, "d must be >= 1");
    if (nparams < 0 || (nparams > 0 && !params)) return fail(KMC_ERR_INVALID, "bad params");
    Ops ops;
    if (!find_ops(kind, d, ops))
        return fail(KMC_ERR_UNSUPPORTED, "no sm_100a kernel for plugin '%s' with d=%d", name, d);
    if (nparams != ops.nparams)
        return fail(KMC_ERR_INVALID, "plugin '%s' with d=%d takes %d parameters, got %lld", name, d,
                    ops.nparams, (long long)nparams);
    // the density under construction, deleted by kmc_density_destroy on every exit but the last
    std::unique_ptr<kmc_density_s, int32_t (*)(kmc_density_t)> h(new kmc_density_s, kmc_density_destroy);
    h->kind = kind;
    h->d = d;
    h->device = device;
    h->ops = ops;
    h->params.assign(std::max<size_t>(std::max<size_t>(1, ops.dn_bytes / sizeof(double)), (size_t)nparams), 0.0);
    if (nparams) memcpy(h->params.data(), params, sizeof(double) * nparams);
    if (kind == kmc::KIND_ROSENBROCK) {  // RN(1/T) for the exact reciprocal-based division (ddiv_by)
        const double T = std::fabs(params[2]);
        h->params[3] = (T > 0x1p-100 && T < 0x1p100) ? 1.0 / params[2] : 0.0;
    }
    if (ops.batch) {  // batched plugins keep parameters (and data) in device memory
        if (nparams) h->params.assign(params, params + nparams);
        CU_TRY(cudaSetDevice(device));
        int nsm = 0;
        cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, device);
        h->nsm = nsm > 0 ? nsm : 148;
        if (nparams) {
            CU_TRY(dev_alloc(&h->d_params, sizeof(double) * nparams, device));
            CU_TRY(cudaMemcpy(h->d_params, params, sizeof(double) * nparams, cudaMemcpyHostToDevice));
        }
        if (ops.batch == BATCH_GAUSSIAN) {  // A^T padded to a multiple of 128 rows for the FP64 kernels
            const size_t dpad = (size_t)(d + 127) / 128 * 128;
            std::vector<double> At((size_t)d * dpad, 0.0);
            for (int i = 0; i < d; ++i)
                for (int j = 0; j < d; ++j) At[(size_t)j * dpad + i] = params[d + (size_t)i * d + j];
            CU_TRY(dev_alloc(&h->d_At, sizeof(double) * At.size(), device));
            CU_TRY(cudaMemcpy(h->d_At, At.data(), sizeof(double) * At.size(), cudaMemcpyHostToDevice));
        }
        if (ops.batch == BATCH_GAUSSIAN && d <= kmc::kWideMaxD) {  // matrix pieces for the tcgen05 Mahalanobis GEMM
            CU_TRY(dev_alloc(&h->d_Abf, sizeof(__nv_bfloat16) * kmc::tc::PIECES * kmc::tc::GN * kmc::tc::GK, device));
            const long long ne = (long long)kmc::tc::GN * kmc::tc::GK;
            kmc::tc::split_rows128_kernel<<<(unsigned)((ne + 255) / 256), 256>>>(h->d_params + d, nullptr, h->d_Abf, d,
                                                                                kmc::tc::GN, d);
            CU_TRY(cudaDeviceSynchronize());
            h->tc_ok = make_map_bf16_k128(&h->mapA, h->d_Abf, (unsigned long long)kmc::tc::PIECES * kmc::tc::GN,
                                          kmc::tc::GN);
        }
        if (ops.batch == BATCH_LOGISTIC) {
            const long long N = data_bytes / (long long)(sizeof(float) * (d + 1));
            if (!data || N < 1 || N * (long long)(sizeof(float) * (d + 1)) != data_bytes)
                return fail(KMC_ERR_INVALID, "logistic needs data = float32 X[N][d] then y[N] (%d+1 floats per row)", d);
            if (!(params[0] > 0.0)) return fail(KMC_ERR_INVALID, "logistic prior_sigma must be > 0");
            h->ndata = N;
            CU_TRY(dev_alloc(&h->d_X, sizeof(float) * N * d, device));
            CU_TRY(dev_alloc(&h->d_y, sizeof(float) * N, device));
            CU_TRY(cudaMemcpy(h->d_X, data, sizeof(float) * N * d, cudaMemcpyHostToDevice));
            CU_TRY(cudaMemcpy(h->d_y, (const float *)data + N * d, sizeof(float) * N, cudaMemcpyHostToDevice));
            // tcgen05 path: d <= 64 (zero-padded to K = 32 or 64) and every X value exactly representable in bf16
            if (d <= 64) {
                h->kp = d <= 32 ? 32 : 64;
                const uint32_t *xb = reinterpret_cast<const uint32_t *>(data);
                bool exact = true;
                for (long long i = 0; i < N * d && exact; ++i) exact = (xb[i] & 0xFFFFu) == 0;
                if (exact) {
                    // X^T (y - 1/2) in FP64: the y_n s_n term and the s_n/2 term of softplus(s) = s/2 + |s|/2 +
                    // log1p(e^-|s|) together are then an exact d-dot (logistic_tc_finish_kernel)
                    std::vector<double> xty(d, 0.0);
                    const float *Xh = (const float *)data, *yh = Xh + N * d;
                    for (long long n = 0; n < N; ++n) {
                        const double yc = (double)yh[n] - 0.5;
                        for (int c = 0; c < d; ++c) xty[c] += yc * (double)Xh[n * d + c];
                    }
                    CU_TRY(dev_alloc(&h->d_Xbf, sizeof(__nv_bfloat16) * N * h->kp, device));
                    CU_TRY(dev_alloc(&h->d_xty, sizeof(double) * d, device));
                    CU_TRY(cudaMemcpy(h->d_xty, xty.data(), sizeof(double) * d, cudaMemcpyHostToDevice));
                    kmc::tc::f32_to_bf16_kernel<<<(unsigned)((N * h->kp + 255) / 256), 256>>>(h->d_X, h->d_Xbf, N, d, h->kp);
                    CU_TRY(cudaDeviceSynchronize());
                    h->tc_ok = make_map_bf16_k(&h->mapX, h->d_Xbf, (unsigned long long)N, kmc::tc::BN, h->kp);
                }
            }
        }
    }
    *out = h.release();
    return KMC_OK;
}

int32_t kmc_density_set_option(kmc_density_t h, const char *key, double value) {
    if (!h || !key) return fail(KMC_ERR_INVALID, "NULL argument");
    if (!strcmp(key, "tensor_cores")) {
        if (value != 0.0 && !h->tc_ok)
            return fail(KMC_ERR_UNSUPPORTED, "this density has no tcgen05 path (dense Gaussian with 16 < d <= 128; logistic "
                                             "with d <= 64 and bf16-representable data)");
        h->tc_on = value != 0.0;
        return KMC_OK;
    }
    if (!strcmp(key, "fused_variant")) {
        if (value != 1.0 && value != 2.0) return fail(KMC_ERR_INVALID, "fused_variant must be 1 (K2F) or 2 (K2G)");
        h->fused_variant = (int)value;
        return KMC_OK;
    }
    return fail(KMC_ERR_INVALID, "unknown option '%s'", key);
}

int32_t kmc_density_get_info(kmc_density_t h, const char *key, double *value) {
    if (!h || !key || !value) return fail(KMC_ERR_INVALID, "NULL argument");
    if (!strcmp(key, "tensor_cores")) {
        *value = h->tc() ? 1.0 : 0.0;
        return KMC_OK;
    }
    if (!strcmp(key, "tensor_cores_available")) {
        *value = h->tc_ok ? 1.0 : 0.0;
        return KMC_OK;
    }
    if (!strcmp(key, "batched")) {
        *value = h->ops.batch;
        return KMC_OK;
    }
    if (!strcmp(key, "fused_variant")) {
        *value = h->fused_variant;
        return KMC_OK;
    }
    return fail(KMC_ERR_INVALID, "unknown info key '%s'", key);
}

int32_t kmc_density_destroy(kmc_density_t h) {
    if (!h) return KMC_OK;
    dev_free(h->d_params);
    dev_free(h->d_X);
    dev_free(h->d_y);
    dev_free(h->d_Xbf);
    dev_free(h->d_xty);
    dev_free(h->d_Abf);
    dev_free(h->d_At);
    delete h;
    return KMC_OK;
}

int32_t kmc_density_eval(kmc_density_t h, const double *thetas, int64_t nw, double *logp_out) {
    if (!h || !thetas || !logp_out || nw < 0) return fail(KMC_ERR_INVALID, "bad argument");
    if (nw == 0) return KMC_OK;
    CU_TRY(cudaSetDevice(h->device));
    DevBuf<double> dx, dl;
    BatchScratch sc;
    CU_TRY(dev_alloc(dx, sizeof(double) * nw * h->d, h->device));
    CU_TRY(dev_alloc(dl, sizeof(double) * nw, h->device));
    CU_TRY(cudaMemcpy(dx.get(), thetas, sizeof(double) * nw * h->d, cudaMemcpyHostToDevice));
    CU_TRY(eval_on_device(*h, dx.get(), nw, dl.get(), sc, nullptr));
    CU_TRY(cudaMemcpy(logp_out, dl.get(), sizeof(double) * nw, cudaMemcpyDeviceToHost));
    CU_TRY(cudaDeviceSynchronize());
    return KMC_OK;
}

int32_t kmc_emcee_destroy(kmc_sampler_t s) {
    if (!s) return KMC_OK;
    cudaSetDevice(s->opts.device);
    if (s->stream) cudaStreamSynchronize(s->stream);  // cached blocks must be idle before reuse
    if (s->push) cudaFree(s->window);  // own allocation (exported through CUDA IPC); x lives inside it
    else dev_free(s->x);
    dev_free(s->task_ctr);
    dev_free(s->notes);
    dev_free(s->lp);
    dev_free(s->chain_x);
    dev_free(s->chain_lp);
    dev_free(s->nacc);
    dev_free(s->barrier);
    dev_free(s->rp_partner);
    dev_free(s->rp_z);
    dev_free(s->rp_u);
    dev_free(s->rp_n);
    dev_free(s->d_sigma);
    dev_free(s->d_chol);
    dev_free(s->d_z);
    dev_free(s->scratch);
    for (void *q : s->ipc_opened) cudaIpcCloseMemHandle(q);
    cudaFree(s->flags);
    dev_free(s->bb.Y);
    dev_free(s->bb.z);
    dev_free(s->bb.u);
    dev_free(s->bb.p1);
    dev_free(s->bb.j);
    if (s->ev0) cudaEventDestroy(s->ev0);
    if (s->ev1) cudaEventDestroy(s->ev1);
    if (s->own_stream) cudaStreamDestroy(s->own_stream);
    delete s;
    return KMC_OK;
}

int32_t kmc_emcee_create(kmc_density_t density, const double *theta0s, int64_t nwalkers, int32_t d,
                         const kmc_emcee_opts *opts, kmc_sampler_t *out) {
    if (!out) return fail(KMC_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (!density || !theta0s || !opts) return fail(KMC_ERR_INVALID, "NULL argument");
    if (d != density->d) return fail(KMC_ERR_INVALID, "d=%d does not match the density (d=%d)", d, density->d);
    // the reference's asserts, src/samplers.jl:200-205
    if (!(opts->a_scale > 1.0)) return fail(KMC_ERR_INVALID, "a_scale must be > 1");
    if (nwalkers < 2 || (nwalkers & 1)) return fail(KMC_ERR_INVALID, "Use an even number of walkers.");
    if (nwalkers < (int64_t)d + 2)
        return fail(KMC_ERR_INVALID, "Use more walkers: at least DOF+2, but better many more.");
    if (opts->nthin < 1) return fail(KMC_ERR_INVALID, "nthin must be >= 1");
    if (opts->niter_walker < 0 || opts->nburnin_walker < 0)
        return fail(KMC_ERR_INVALID, "niter and nburnin must be >= 0");
    if (nwalkers / 2 >= (1LL << 32)) return fail(KMC_ERR_INVALID, "too many walkers");
    if (opts->mode != KMC_MODE_PHILOX && opts->mode != KMC_MODE_REPLAY)
        return fail(KMC_ERR_INVALID, "unknown mode %d", opts->mode);
    if (density->ops.batch && opts->device != density->device)
        return fail(KMC_ERR_INVALID, "the density's parameters / data live on device %d, the sampler was asked for device %d",
                    density->device, opts->device);

    CU_TRY(cudaSetDevice(opts->device));
    SamplerPtr s(new kmc_sampler_s, kmc_emcee_destroy);
    s->dn = density;
    s->opts = *opts;
    s->nw = nwalkers;
    s->nhalf = nwalkers / 2;
    s->d = d;
    s->sbeg = opts->shard_count > 0 ? opts->shard_begin : 0;
    s->scnt = opts->shard_count > 0 ? opts->shard_count : s->nhalf;
    s->nl = 2 * s->scnt;
    if (s->sbeg < 0 || s->sbeg + s->scnt > s->nhalf)
        return fail(KMC_ERR_INVALID, "shard [%lld, %lld) is outside the half-ensemble [0, %lld)", s->sbeg,
                    s->sbeg + s->scnt, (long long)(nwalkers / 2));
    const long long nspan = opts->niter_walker - opts->nburnin_walker;
    s->ns = nspan > 0 ? nspan / opts->nthin : 0;  // :234
    s->push = opts->exchange == KMC_EXCHANGE_PUSH;
    if (opts->exchange != KMC_EXCHANGE_REPLICA && opts->exchange != KMC_EXCHANGE_PUSH)
        return fail(KMC_ERR_INVALID, "unknown exchange %d", opts->exchange);
    if (s->push) {  // owner-computes push exchange: equal shards, fused plugin with 16-byte-multiple rows, Philox draws
        const char *why = nullptr;
        if (opts->shard_count <= 0 || s->nhalf % s->scnt || s->sbeg % s->scnt) why = "equal shards: rank r owns [r*S, (r+1)*S) of each half";
        else if (s->nhalf / s->scnt > kmc::kPushMaxRanks) why = "at most 8 ranks";
        else if (density->ops.batch || !density->ops.run_push) why = "a fused (non-batched) plugin with even d";
        else if (opts->mode != KMC_MODE_PHILOX || opts->launch_mode != 0) why = "Philox draws and launch_mode 0";
        else if (opts->push_chunk < 0 || opts->push_chunk > kmc::kPushMaxChunk) why = "push_chunk within the kernel's maximum";
        else if (opts->push_cap < 0 || opts->push_cap > kmc::kPushMaxCap) why = "push_cap within the kernel's maximum";
        else if (opts->push_lag < -1) why = "push_lag >= -1";
        if (why) return fail(KMC_ERR_UNSUPPORTED, "the push exchange needs %s", why);
        s->G = (int)(s->nhalf / s->scnt);
        s->rank = (int)(s->sbeg / s->scnt);
        // default: a chunk sends ~one task-width of rows per destination (kPushThreads walkers per rank), capped by the
        // kernel's maximum chunk; a ring slot holds the mean hit count + k sigma of its binomial spread (rows past it are
        // read from the owner directly): k = 8 for CTA-wide tasks, 3 for warp-wide ones (their shared memory is tight)
        s->chunk = opts->push_chunk > 0 ? (unsigned)opts->push_chunk
                                        : (unsigned)std::min<long long>(kmc::kPushMaxChunk,
                                                                        (long long)kmc::kPushThreads * std::max(s->G, 1));
        if (s->G == 1 && opts->push_chunk <= 0) s->chunk = kmc::kPushMaxChunk;
        s->chunk = (unsigned)std::min<long long>(s->chunk, std::max<long long>(s->scnt, 1));
        s->rounds = (s->chunk + kmc::kPushThreads - 1) / kmc::kPushThreads;
        s->nchunks = (unsigned)((s->scnt + s->chunk - 1) / s->chunk);
        const double mean_hits = (double)s->chunk / s->G, ksig = kmc::kPushThreads == 32 ? 3.0 : 8.0;
        const unsigned want = (unsigned)(mean_hits + ksig * std::sqrt(mean_hits * (1.0 - 1.0 / s->G)) + 2.0);
        s->cap = opts->push_cap > 0 ? (unsigned)opts->push_cap : std::min<unsigned>(kmc::kPushMaxCap, std::max(want, 16u));
    }
    s->nstate = s->push ? 2 * s->scnt : s->nw;
    s->hoff = s->push ? s->scnt : s->nhalf;
    s->loff = s->push ? 0 : s->sbeg;

    if (s->push) {  // one window: [chunk flags | receive ring | positions], exported as ONE CUDA IPC handle
        auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
        s->win_flags = 0;
        s->win_recv = up(sizeof(unsigned long long) * (size_t)s->G * s->nchunks);
        s->win_x = s->win_recv + up(2 * (size_t)s->G * s->nchunks * (kmc::kPushHeader + sizeof(double) * s->cap * d));
        s->win_bytes = s->win_x + up(sizeof(double) * (size_t)s->nstate * d);
        CU_TRY(cudaMalloc(&s->window, s->win_bytes));
        s->x = reinterpret_cast<double *>(s->window + s->win_x);
    }
    if (const int32_t rc = sampler_init(s.get(), theta0s); rc != KMC_OK) return rc;
    if (s->push) {
        CU_TRY(cudaMemsetAsync(s->window, 0, s->win_recv, s->stream));  // flags = 0: nothing has landed
        push_set_peer(s.get(), s->rank, s->window);
        CU_TRY(dev_alloc(&s->task_ctr, 4 * sizeof(unsigned long long), opts->device));
        if (s->G > 1) {  // the publisher's inbox: one note per push task, epochs only grow
            const size_t nb = sizeof(unsigned) * (size_t)s->nchunks * (s->G - 1);
            CU_TRY(dev_alloc(&s->notes, nb, opts->device));
            CU_TRY(cudaMemsetAsync(s->notes, 0, nb, s->stream));
        }
    }
    CU_TRY(dev_alloc(&s->barrier, sizeof(unsigned long long), opts->device));
    CU_TRY(cudaMemsetAsync(s->barrier, 0, sizeof(unsigned long long), s->stream));
    CU_TRY(cudaMalloc(&s->flags, 8 * sizeof(unsigned long long)));  // own allocation: exported through CUDA IPC
    CU_TRY(cudaMemsetAsync(s->flags, 0, 8 * sizeof(unsigned long long), s->stream));
    if (density->ops.batch) {  // the half-step's stretch factors and partners
        CU_TRY(dev_alloc(&s->bb.z, sizeof(double) * s->scnt, opts->device));
        CU_TRY(dev_alloc(&s->bb.j, sizeof(unsigned) * s->scnt, opts->device));
    }
    CU_TRY(cudaDeviceGetAttribute(&s->nsm, cudaDevAttrMultiProcessorCount, opts->device));
    if (s->push) {  // one persistent kernel, tasks handed out dynamically: as many CTAs as fit
        const void *kp = density->ops.run_push;
        const size_t psm = kmc::push_smem_bytes(d, s->cap);
        CU_TRY(cudaFuncSetAttribute(kp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)psm));
        int occ = 0;
        CU_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kp, kmc::kPushThreads, psm));
        if (occ < 1) return fail(KMC_ERR_CUDA, "the push kernel does not fit on the device");
        s->grid = (unsigned)(occ * s->nsm);
        s->block = kmc::kPushThreads;
        s->smem_bytes = psm;
        s->lag = kmc_host::push_default_lag(s->nchunks, opts->push_lag);
    } else if (!density->ops.batch) {   // persistent launch geometry: every CTA owns per_cta walker positions of each half and
        // every thread the same number of them (block size = per_cta / rounds, warp-rounded)
        const int r = opts->mode == KMC_MODE_REPLAY ? 1 : 0;
        auto geometry = [&](const void *kern, int maxblk, int ctas_per_sm, size_t smem_per_walker, bool &fits) {
            const long long want = (s->scnt + maxblk - 1) / maxblk;
            s->grid = (unsigned)std::min<long long>(want, (long long)ctas_per_sm * s->nsm);
            s->per_cta = (unsigned)((s->scnt + s->grid - 1) / s->grid);
            s->grid = (unsigned)((s->scnt + s->per_cta - 1) / s->per_cta);
            const unsigned rounds = (s->per_cta + maxblk - 1) / maxblk;
            s->block = std::min<unsigned>(maxblk, (((s->per_cta + rounds - 1) / rounds + 31) / 32) * 32);
            s->smem_bytes = (size_t)2 * s->per_cta * smem_per_walker;
            if (s->smem_bytes > 48 * 1024) {
                cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)s->smem_bytes);
                if (e != cudaSuccess) { cudaGetLastError(); fits = false; return rounds; }
            }
            fits = (long long)occupancy(kern, (int)s->block, s->smem_bytes) * s->nsm >= (long long)s->grid;
            return rounds;
        };
        bool fits = false;
        s->use_smem = false;
        if (opts->launch_mode == 0 && density->ops.run[r][1] && opts->shard_count == 0) {  // shared-memory-resident state if it fits
            int max_optin = 0;
            CU_TRY(cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, opts->device));
            const unsigned rounds = geometry(density->ops.run[r][1], kmc::kSmemThreads, kmc::kSmemCtas, density->ops.smem_per_walker, fits);
            s->use_smem = fits && rounds <= (unsigned)kmc::kRounds && s->smem_bytes <= (size_t)max_optin;
        }
        s->use_bulk = !s->use_smem && opts->launch_mode == 0 && r == 0 && density->ops.run_bulk[0];
        if (s->use_bulk) {  // 2 CTAs x 256 threads per SM, rows staged through shared memory
            const void *kb0 = density->ops.run_bulk[0], *kb1 = density->ops.run_bulk[1];
            cudaFuncSetAttribute(kb0, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)density->ops.bulk_smem);
            cudaFuncSetAttribute(kb1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)density->ops.bulk_smem);
            const int occ = occupancy(kb1, kmc::kBulkThreads, density->ops.bulk_smem);
            if (occ < 1) {
                cudaGetLastError();  // and the attribute calls' errors
                s->use_bulk = false;
            } else {
                const long long want = (s->scnt + kmc::kBulkThreads - 1) / kmc::kBulkThreads;
                s->grid = (unsigned)std::min<long long>(want, (long long)occ * s->nsm);
                s->per_cta = (unsigned)((s->scnt + s->grid - 1) / s->grid);
                s->per_cta = ((s->per_cta + 1) / 2) * 2;  // even: group bases stay 16-byte aligned for any even D
                s->grid = (unsigned)((s->scnt + s->per_cta - 1) / s->per_cta);
                s->block = kmc::kBulkThreads;
                s->smem_bytes = density->ops.bulk_smem;
            }
        }
        if (!s->use_smem && !s->use_bulk) {
            // as many CTAs per SM as the kernel's registers allow (at least what it was compiled for)
            int occ = occupancy(density->ops.run[r][0], density->ops.block, 0);
            if (opts->shard_count > 0 && density->ops.run_peer)  // a sharded sampler may switch to the peer kernel
                occ = std::min(occ, occupancy(density->ops.run_peer, density->ops.block, 0));
            geometry(density->ops.run[r][0], density->ops.block, std::max(occ, 1), 0, fits);
            if (!fits) return fail(KMC_ERR_CUDA, "kernel does not fit on the device");
        }
    }
    CU_TRY(cudaStreamSynchronize(s->stream));
    *out = s.release();
    return KMC_OK;
}

int32_t kmc_emcee_set_stream(kmc_sampler_t s, void *cuda_stream) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    CU_TRY(cudaSetDevice(s->opts.device));
    CU_TRY(cudaStreamSynchronize(s->stream));
    s->stream = cuda_stream ? (cudaStream_t)cuda_stream : s->own_stream;
    return KMC_OK;
}

int32_t kmc_emcee_set_replay(kmc_sampler_t s, const int64_t *partner, const double *z, const double *u,
                             int64_t niters) {
    if (!s || !partner || !z || !u || niters < 0) return fail(KMC_ERR_INVALID, "bad argument");
    if (s->metro) return fail(KMC_ERR_STATE, "a Metropolis handle takes its draws through kmc_metropolis_set_replay");
    if (s->opts.mode != KMC_MODE_REPLAY) return fail(KMC_ERR_STATE, "sampler is not in replay mode");
    CU_TRY(cudaSetDevice(s->opts.device));
    CU_TRY(cudaStreamSynchronize(s->stream));
    const long long n = niters * s->nw;
    for (long long i = 0; i < n; ++i)
        if (partner[i] < 0 || partner[i] >= s->nw)
            return fail(KMC_ERR_INVALID, "replay partner %lld at slot %lld is outside [0, nwalkers)",
                        (long long)partner[i], i);
    dev_free(s->rp_partner);
    dev_free(s->rp_z);
    dev_free(s->rp_u);
    s->rp_partner = nullptr;
    s->rp_z = s->rp_u = nullptr;
    s->rp_niters = 0;
    if (n > 0) {
        CU_TRY(dev_alloc(&s->rp_partner, sizeof(long long) * n, s->opts.device));
        CU_TRY(dev_alloc(&s->rp_z, sizeof(double) * n, s->opts.device));
        CU_TRY(dev_alloc(&s->rp_u, sizeof(double) * n, s->opts.device));
        CU_TRY(cudaMemcpy(s->rp_partner, partner, sizeof(long long) * n, cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(s->rp_z, z, sizeof(double) * n, cudaMemcpyHostToDevice));
        CU_TRY(cudaMemcpy(s->rp_u, u, sizeof(double) * n, cudaMemcpyHostToDevice));
    }
    s->rp_t0 = (s->hdone / 2);
    s->rp_niters = niters;
    return KMC_OK;
}

int32_t kmc_emcee_run_half(kmc_sampler_t s, int64_t nhalfsteps) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    if (s->metro) return fail(KMC_ERR_STATE, "a Metropolis handle has no half-steps: use kmc_emcee_run");
    return run_range(s, s->hdone, 2 * s->opts.niter_walker, nhalfsteps, 2,
                     [s](long long hbeg, long long hend, long long &launches) -> int32_t {
        kmc::RunParams p{};
        p.x = s->x;
        p.lp = s->lp;
        p.nacc = s->nacc;
        p.chain_x = s->chain_x;
        p.chain_lp = s->chain_lp;
        p.rp_partner = s->rp_partner;
        p.rp_z = s->rp_z;
        p.rp_u = s->rp_u;
        p.rp_t0 = s->rp_t0;
        p.nw = s->nw;
        p.nhalf = (unsigned)s->nhalf;
        p.shard_begin = (unsigned)s->sbeg;
        p.shard_end = (unsigned)(s->sbeg + s->scnt);
        p.chain_nw = s->nl;
        p.nthin = s->opts.nthin;
        p.ns = s->ns;
        const double a = s->opts.a_scale;
        p.sia = std::sqrt(1.0 / a);
        p.span = std::sqrt(a) - p.sia;
        p.nm1 = (double)(s->d - 1);
        p.nm1f = (float)(s->d - 1);
        p.margin = (float)((p.nm1 + 64.0) * 2e-6);
        p.keys = kmc::philox_keys(s->opts.seed);
        p.id_base[0] = (unsigned)s->opts.walker_id_base;
        p.id_base[1] = (unsigned)(s->opts.walker_id_base + s->nhalf);
        const unsigned nh = (unsigned)s->nhalf;
        p.lemire_t = (unsigned)(0u - nh) % nh;
        p.barrier = s->barrier;
        p.per_cta = s->per_cta;
        if (s->npeers >= 1) {  // set_peers was called (a single rank exercises the bulk-copy gathers alone)
            if (s->opts.mode == KMC_MODE_REPLAY || s->dn->ops.batch || s->opts.launch_mode != 0 || !s->dn->ops.run_peer)
                return fail(KMC_ERR_UNSUPPORTED, "peer mode needs a fused (non-batched) plugin, Philox draws and launch_mode 0");
            // The ranks meet at a flag barrier BETWEEN the half-steps of one launch only: a second launch could gather from a
            // peer that is still writing the last half-step of the first.  The pull mode therefore runs the whole job in ONE
            // launch (the push exchange, kmc_emcee_window_*, has no such restriction).
            if (s->npeers > 1 && (hbeg != 0 || hend != 2 * s->opts.niter_walker))
                return fail(KMC_ERR_STATE, "peer (pull) mode runs the whole job in one launch: call kmc_emcee_run(s, -1) once");
            for (int r = 0; r < s->npeers; ++r) {
                p.peer_x[r] = s->peer_x[r];
                p.peer_flags[r] = s->peer_flags[r];
            }
            p.npeers = s->npeers;
            p.rank = s->rank;
            p.epoch_base = s->epoch;
        }
        if (s->push) return run_push(s, p, hbeg, hend, launches);
        if (s->dn->ops.batch == BATCH_GAUSSIAN && s->dn->tc() && s->opts.launch_mode == 0)
            return run_fused_gauss(s, p, hbeg, hend, launches);
        if (s->dn->ops.batch) return run_batched(s, p, hbeg, hend, launches);
        if (s->opts.launch_mode == 1) return run_per_half(s, p, hbeg, hend, launches);
        return run_persistent(s, p, hbeg, hend, launches);
    });
}

int32_t kmc_emcee_run(kmc_sampler_t s, int64_t niters) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    if (s->metro) return metro_run(s, niters);
    if (s->hdone & 1) return fail(KMC_ERR_STATE, "an outer iteration is half done: finish it with kmc_emcee_run_half");
    return kmc_emcee_run_half(s, niters < 0 ? -1 : 2 * niters);
}

int32_t kmc_emcee_ipc_export(kmc_sampler_t s, void *handle_x, void *handle_flags) {
    if (!s || !handle_x || !handle_flags) return fail(KMC_ERR_INVALID, "NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handles are 64 bytes");
    if (s->metro) return fail(KMC_ERR_STATE, "Metropolis chains are independent: nothing to exchange");
    CU_TRY(cudaSetDevice(s->opts.device));
    if (s->push) return fail(KMC_ERR_STATE, "a push-exchange sampler exports its window (kmc_emcee_window_export)");
    CU_TRY(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t *>(handle_x), s->x));
    CU_TRY(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t *>(handle_flags), s->flags));
    return KMC_OK;
}

int32_t kmc_emcee_set_peers(kmc_sampler_t s, const void *handles_x, const void *handles_flags, int32_t nranks,
                            int32_t rank) {
    if (!s || !handles_x || !handles_flags) return fail(KMC_ERR_INVALID, "NULL argument");
    if (s->metro) return fail(KMC_ERR_STATE, "Metropolis chains are independent: nothing to exchange");
    if (nranks < 1 || nranks > 8 || rank < 0 || rank >= nranks) return fail(KMC_ERR_INVALID, "bad rank / nranks (max 8)");
    if (s->push) return fail(KMC_ERR_STATE, "a push-exchange sampler attaches windows (kmc_emcee_window_attach)");
    if (s->scnt * nranks != s->nhalf || s->sbeg != (long long)rank * s->scnt)
        return fail(KMC_ERR_INVALID, "peer mode needs equal shards: rank r owns [r*S, (r+1)*S) of each half");
    CU_TRY(cudaSetDevice(s->opts.device));
    const cudaIpcMemHandle_t *hx = reinterpret_cast<const cudaIpcMemHandle_t *>(handles_x);
    const cudaIpcMemHandle_t *hf = reinterpret_cast<const cudaIpcMemHandle_t *>(handles_flags);
    for (int r = 0; r < nranks; ++r) {
        if (r == rank) {
            s->peer_x[r] = s->x;
            s->peer_flags[r] = s->flags;
            continue;
        }
        void *px = nullptr, *pf = nullptr;
        CU_TRY(cudaIpcOpenMemHandle(&px, hx[r], cudaIpcMemLazyEnablePeerAccess));
        s->ipc_opened.push_back(px);
        CU_TRY(cudaIpcOpenMemHandle(&pf, hf[r], cudaIpcMemLazyEnablePeerAccess));
        s->ipc_opened.push_back(pf);
        s->peer_x[r] = static_cast<const double *>(px);
        s->peer_flags[r] = static_cast<unsigned long long *>(pf);
    }
    s->npeers = nranks;
    s->rank = rank;
    return KMC_OK;
}

int32_t kmc_emcee_window_export(kmc_sampler_t s, void *handle) {
    if (!s || !handle) return fail(KMC_ERR_INVALID, "NULL argument");
    if (s->metro) return fail(KMC_ERR_STATE, "Metropolis chains are independent: nothing to exchange");
    if (!s->push) return fail(KMC_ERR_STATE, "not a push-exchange sampler (opts.exchange = KMC_EXCHANGE_PUSH)");
    CU_TRY(cudaSetDevice(s->opts.device));
    CU_TRY(cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t *>(handle), s->window));
    return KMC_OK;
}

int32_t kmc_emcee_window_attach(kmc_sampler_t s, const void *handles, int32_t nranks, int32_t rank) {
    if (!s || !handles) return fail(KMC_ERR_INVALID, "NULL argument");
    if (s->metro) return fail(KMC_ERR_STATE, "Metropolis chains are independent: nothing to exchange");
    if (!s->push) return fail(KMC_ERR_STATE, "not a push-exchange sampler (opts.exchange = KMC_EXCHANGE_PUSH)");
    if (nranks != s->G || rank != s->rank)
        return fail(KMC_ERR_INVALID, "the sampler's shard is rank %d of %d, got rank %d of %d", s->rank, s->G, rank, nranks);
    CU_TRY(cudaSetDevice(s->opts.device));
    const cudaIpcMemHandle_t *hw = reinterpret_cast<const cudaIpcMemHandle_t *>(handles);
    for (int r = 0; r < nranks; ++r) {
        if (r == rank) {
            push_set_peer(s, r, s->window);
            continue;
        }
        void *pw = nullptr;
        CU_TRY(cudaIpcOpenMemHandle(&pw, hw[r], cudaIpcMemLazyEnablePeerAccess));
        s->ipc_opened.push_back(pw);
        push_set_peer(s, r, static_cast<unsigned char *>(pw));
    }
    s->attached = true;
    return KMC_OK;
}

int32_t kmc_emcee_device_ptrs(kmc_sampler_t s, void **x, void **logp, void **naccept) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    if (x) *x = s->x;
    if (logp) *logp = s->lp;
    if (naccept) *naccept = s->nacc;
    return KMC_OK;
}

int32_t kmc_emcee_sync(kmc_sampler_t s) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    CU_TRY(cudaSetDevice(s->opts.device));
    CU_TRY(cudaStreamSynchronize(s->stream));
    return KMC_OK;
}

int32_t kmc_emcee_last_run_ms(kmc_sampler_t s, double *ms, int64_t *launches) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    if (launches) *launches = s->last_launches;
    if (ms) *ms = 0.0;
    if (!s->timed) return KMC_OK;
    CU_TRY(cudaSetDevice(s->opts.device));
    CU_TRY(cudaEventSynchronize(s->ev1));
    float f = 0.f;
    CU_TRY(cudaEventElapsedTime(&f, s->ev0, s->ev1));
    if (ms) *ms = f;
    return KMC_OK;
}

int32_t kmc_emcee_progress(kmc_sampler_t s, int64_t *iters_done, double *naccept_mean, double *naccept_std,
                           int64_t *outliers) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    CU_TRY(cudaSetDevice(s->opts.device));
    unsigned long long *sum = s->scratch, *outl = s->scratch + 1;
    double *ssq = reinterpret_cast<double *>(s->scratch + 2);
    CU_TRY(cudaMemsetAsync(s->scratch, 0, 4 * sizeof(unsigned long long), s->stream));
    const long long nst = s->nstate;  // the whole ensemble, or this shard's walkers for a push-exchange sampler
    const unsigned grid = (unsigned)std::min<long long>((nst + 255) / 256, 1184);
    kmc::nacc_sum_kernel<<<grid, 256, 0, s->stream>>>(s->nacc, nst, sum);
    unsigned long long hsum = 0, houtl = 0;
    double hssq = 0.0;
    CU_TRY(cudaMemcpyAsync(&hsum, sum, sizeof hsum, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    const double mean = (double)hsum / (double)nst;  // :276
    kmc::nacc_moment_kernel<<<grid, 256, 0, s->stream>>>(s->nacc, nst, mean, -1.0, ssq, nullptr);
    CU_TRY(cudaMemcpyAsync(&hssq, ssq, sizeof hssq, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    const double sd = std::sqrt(hssq / (double)(nst - 1));  // :277 sqrt(var(naccept))
    kmc::nacc_moment_kernel<<<grid, 256, 0, s->stream>>>(s->nacc, nst, mean, 2.0 * sd, nullptr, outl);  // :278
    CU_TRY(cudaMemcpyAsync(&houtl, outl, sizeof houtl, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    CU_TRY(cudaGetLastError());
    if (iters_done) *iters_done = s->metro ? s->tdone : (s->hdone / 2);
    if (naccept_mean) *naccept_mean = mean;
    if (naccept_std) *naccept_std = sd;
    if (outliers) *outliers = (int64_t)houtl;
    return KMC_OK;
}

int32_t kmc_emcee_nsamples(kmc_sampler_t s, int64_t *ns) {
    if (!s || !ns) return fail(KMC_ERR_INVALID, "NULL argument");
    *ns = s->ns;
    return KMC_OK;
}

int32_t kmc_emcee_nlocal(kmc_sampler_t s, int64_t *nl) {
    if (!s || !nl) return fail(KMC_ERR_INVALID, "NULL argument");
    *nl = s->nl;
    return KMC_OK;
}

int32_t kmc_emcee_copy_results(kmc_sampler_t s, double *thetas, double *logp, double *accept_ratio) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    CU_TRY(cudaSetDevice(s->opts.device));
    CU_TRY(cudaStreamSynchronize(s->stream));
    const long long nl = s->nl;
    if (s->ns > 0 && (thetas || logp))
        if (const int32_t rc = chain_gather(s, nullptr, nl, thetas, logp); rc != KMC_OK) return rc;
    if (accept_ratio) {  // this sampler's walkers: its slice of half 0, then of half 1 (Metropolis: every chain)
        std::vector<unsigned> h(nl);
        if (s->metro) {
            CU_TRY(cudaMemcpy(h.data(), s->nacc, sizeof(unsigned) * nl, cudaMemcpyDeviceToHost));
        } else {
            CU_TRY(cudaMemcpy(h.data(), s->nacc + s->loff, sizeof(unsigned) * s->scnt, cudaMemcpyDeviceToHost));
            CU_TRY(cudaMemcpy(h.data() + s->scnt, s->nacc + s->hoff + s->loff, sizeof(unsigned) * s->scnt,
                              cudaMemcpyDeviceToHost));
        }
        const double den = (double)(s->opts.niter_walker - s->opts.nburnin_walker);  // :291
        for (long long w = 0; w < nl; ++w) accept_ratio[w] = (double)h[w] / den;
    }
    return KMC_OK;
}

int32_t kmc_emcee_chain_moments(kmc_sampler_t s, double *mean, double *var, int64_t *count) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    const long long nrows = s->ns * s->nl;
    const int d = s->d;
    if (count) *count = nrows;
    if (nrows < 1) return fail(KMC_ERR_STATE, "no samples stored");
    CU_TRY(cudaSetDevice(s->opts.device));
    DevBuf<double> sums;
    CU_TRY(dev_alloc(sums, sizeof(double) * 2 * d, s->opts.device));
    std::vector<double> h(2 * d), shift(d);
    CU_TRY(cudaMemsetAsync(sums.get(), 0, sizeof(double) * 2 * d, s->stream));
    const unsigned grid = (unsigned)std::min<long long>((nrows * d + 255) / 256, 148 * 8);
    kmc::chain_moments_kernel<<<grid, 256, sizeof(double) * 2 * d, s->stream>>>(s->chain_x, nrows, d, sums.get());
    CU_TRY(cudaMemcpyAsync(h.data(), sums.get(), sizeof(double) * 2 * d, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaMemcpyAsync(shift.data(), s->chain_x, sizeof(double) * d, cudaMemcpyDeviceToHost, s->stream));
    CU_TRY(cudaStreamSynchronize(s->stream));
    const double n = (double)nrows;
    for (int c = 0; c < d; ++c) {
        if (mean) mean[c] = shift[c] + h[c] / n;
        if (var) var[c] = nrows > 1 ? (h[d + c] - h[c] * h[c] / n) / (n - 1.0) : 0.0;
    }
    return KMC_OK;
}

int32_t kmc_emcee_copy_state(kmc_sampler_t s, double *theta, double *logp, int64_t *naccept) {
    if (!s) return fail(KMC_ERR_INVALID, "NULL sampler");
    CU_TRY(cudaSetDevice(s->opts.device));
    CU_TRY(cudaStreamSynchronize(s->stream));
    const long long nst = s->nstate;  // push exchange: the rows this shard holds (its slice of half 0, then of half 1)
    if (theta) CU_TRY(cudaMemcpy(theta, s->x, sizeof(double) * nst * s->d, cudaMemcpyDeviceToHost));
    if (logp) CU_TRY(cudaMemcpy(logp, s->lp, sizeof(double) * nst, cudaMemcpyDeviceToHost));
    if (naccept) {
        std::vector<unsigned> h(nst);
        CU_TRY(cudaMemcpy(h.data(), s->nacc, sizeof(unsigned) * nst, cudaMemcpyDeviceToHost));
        for (long long w = 0; w < nst; ++w) naccept[w] = h[w];
    }
    return KMC_OK;
}

}  // extern "C"
