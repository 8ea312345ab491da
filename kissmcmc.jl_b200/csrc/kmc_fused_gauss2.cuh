// kmc_fused_gauss2.cuh -- K2G: the fused dense-Gaussian half-step (K2F, kmc_fused_gauss.cuh) with the MATRIX as the
// TMEM-resident A operand of the tcgen05 GEMM.  The DEFAULT fused kernel of the tensor-core dense Gaussian in launch_mode 0
// (kmc_density_s::fused_variant = 2); set_option("fused_variant", 1) selects K2F.
//
// Why.  K2F keeps the three matrix pieces (96 KB) and one tile of walker pieces (96 KB) in shared memory, so a tile's
// phases are serialised (no room for a second walker-piece buffer) and every SS-mode MMA reads 7.5 KB of operands from
// shared memory (~95 cycles per 128x112x16 MMA against a 56-cycle tensor floor; profiles/r1_k2f_phase_cycles.log).
// Here the roles of the operands are swapped:
//
//     D[i][w] = sum_k  M[i][k] * C[w][k]          i = output dimension (M of the MMA, 128 TMEM lanes)
//                                                 w = walker of the tile (N of the MMA, <= 128 columns)
//
//   A operand = matrix pieces, written ONCE per kernel into TMEM columns [0,192) (tcgen05.st: lane = row i, two bf16
//               per 32-bit column) and read from there by every MMA (tcgen05.mma ... [d_tmem], [a_tmem], b_desc ...)
//   B operand = walker pieces in shared memory, K-major SWIZZLE_128B exactly as K2F builds them -- now DOUBLE-BUFFERED
//               (2 x 96 KB), so the GEMM of tile t runs while all warps build tile t+1
//   D         = two accumulators of 128 columns (TMEM columns [192,448)): lane i holds y_i of every walker of the tile
//
// Pipeline of a CTA over its tiles k = 0..T-1 of one half-step (T = 2 for BASELINE.json configs[2]):
//     P1(k)  proposals -> pieces c[k&1]            all 16 warps
//     MMA(k) issued by warp 0, commit -> mma_done[k&1]
//     E(k-1) warps 0-3: wait mma_done[(k-1)&1], |y|^2 per walker, accept test    | warps 4-7: draws of tile k+1
//     P3(k-1) write-back of accepted rows          all 16 warps
// so MMA(k) is hidden behind E(k-1), P3(k-1) and P1(k+1).
//
// |y|^2 per walker is a sum over TMEM LANES (i), not columns: each of warps 0-3 squares its 32 lanes' values and
// transposes-and-adds them with a 5-stage shuffle butterfly (31 SHFL + 31 FADD per 32 walkers), the four warps' partial
// sums meet in shared memory and are added in fixed order.  FP32 tree instead of K2F's column-sequential sum: the two
// variants agree to ~1e-7 |y|^2, not bit for bit (both are inside the stated tolerance 1e-5 (1 + |y|^2) of the
// tensor-core Gaussian path; the FP64 kernel is the exact default).
#pragma once
#include "kmc_fused_gauss.cuh"
#ifndef KMC_K2G_POLL_ACQ
#define KMC_K2G_POLL_ACQ 1  // the grid barrier is polled by an idle warp with acquire loads: 18.63 -> 18.26 us per half-step
#endif

namespace kmc {
namespace tc {

constexpr int kRowBufs = 3;            // per-row draw arrays: tile k uses buffer k % 3 (E(k-1) | draws(k+1) | P1(k))
constexpr unsigned kTmemA = 0;         // matrix pieces: piece pc at columns 64*pc .. 64*pc+63
constexpr unsigned kTmemD = 192;       // accumulators: buffer b at columns 192 + 128*b
constexpr unsigned kWorkHalfWarps = 2 * (kFusedThreads / 32 - 1);  // warps 1-15 gather / write back; warp 0 issues MMAs

struct __align__(1024) Fused2Smem {
    unsigned char c[2][PIECES][GPIECE_BYTES];  // walker pieces (B operand), double-buffered
    unsigned long long mma_done[2];
    unsigned tmem_base;
    double z[kRowBufs][BM], u[kRowBufs][BM];
    unsigned j[kRowBufs][BM];
    float q[kRowBufs][BM];
    alignas(16) double mu[GK];
    float part[4][BM];                 // per-warp partial |y|^2 (over the warp's 32 output dimensions) per walker
    unsigned nlist[kRowBufs];
    unsigned char list[kRowBufs][BM];
    unsigned char acc[kRowBufs][BM];
};

struct Fused2Params {
    const double *mu;          // [d] (device)
    const unsigned *apieces;   // matrix pieces [3][128 rows i][64 words] = bf16 pairs (k even | k odd << 16), row-major
    double lognorm;
    int d;
};

__device__ __forceinline__ void tmem_st32(unsigned taddr, const unsigned (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,"
        "%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};" ::"r"(taddr),
        "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
        "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
        "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
        "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}

// D[tmem] (+)= A[tmem] . B[smem]^T for a converged warp (see tc_mma_elect)
__device__ __forceinline__ void tc_mma_ts_elect(unsigned tmem_d, unsigned tmem_a, unsigned long long bdesc, unsigned idesc,
                                                unsigned accumulate, unsigned leader) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(tmem_d),
        "r"(tmem_a), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
}

template <bool REPLAY>
__global__ void __launch_bounds__(kFusedThreads, 1)
gaussian_fused2_kernel(const RunParams p, const Fused2Params fp) {
    extern __shared__ unsigned char smem_raw[];
    Fused2Smem &sm = *reinterpret_cast<Fused2Smem *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = tid >> 5;
    const int d = fp.d;

    if (tid < GK) sm.mu[tid] = tid < d ? fp.mu[tid] : 0.0;
    if (tid == 0) {
#pragma unroll
        for (int b = 0; b < kRowBufs; ++b) sm.nlist[b] = 0u;
        mbar_init(&sm.mma_done[0], 1);
        mbar_init(&sm.mma_done[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&sm.tmem_base))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem = __shfl_sync(0xffffffffu, sm.tmem_base, 0);

    // the matrix: once per CTA, global -> registers -> TMEM (lane = output dimension i, 64 columns per piece)
    if (warp < 4) {
        const unsigned i = warp * 32 + lane;
#pragma unroll 1
        for (int pc = 0; pc < PIECES; ++pc)
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                const uint4 *src = reinterpret_cast<const uint4 *>(fp.apieces + ((size_t)pc * GN + i) * (GK / 2) + half * 32);
                unsigned v[32];
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const uint4 w = src[e];
                    v[4 * e] = w.x;
                    v[4 * e + 1] = w.y;
                    v[4 * e + 2] = w.z;
                    v[4 * e + 3] = w.w;
                }
                tmem_st32(tmem + ((unsigned)(warp * 32) << 16) + kTmemA + pc * 64 + half * 32, v);
            }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();

    // balanced tiles as in K2F: every CTA gets the same number of tiles per half-step, a tile holds tr <= 128 walkers
    const unsigned W = p.shard_end - p.shard_begin;
    const unsigned waves = ((W + BM - 1) / BM + gridDim.x - 1) / gridDim.x;
    const unsigned tr = min((unsigned)BM, (W + waves * gridDim.x - 1) / (waves * gridDim.x));
    const unsigned ntiles = (W + tr - 1) / tr;
    const unsigned T = ntiles > blockIdx.x ? (ntiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0u;  // tiles of this CTA
    const unsigned nwcols = (tr + 15u) & ~15u;  // N of the MMA: walkers of a tile, rounded up to the instruction's step
    const int nk = (d + 15) / 16;               // k-steps that hold data
    const unsigned half16 = lane >> 4, ck = lane & 15;
    unsigned mph = 0;                           // bit b: phase of mma_done[b]
    ThinClock<> clk{p.n0, p.phase0, p.sidx0};
    unsigned long long target = p.bar_base;

#ifdef KMC_K2F_PROF
    long long pt[6] = {0, 0, 0, 0, 0, 0}, pc0 = clock64();
#define K2G_TICK(i) do { const long long c_ = clock64(); pt[i] += c_ - pc0; pc0 = c_; } while (0)
#else
#define K2G_TICK(i) do { } while (0)
#endif

    for (long long h = p.h0; h < p.h1; ++h) {
        const unsigned batch = (unsigned)(h & 1);
        const bool store = clk.store();
        const size_t a0 = batch ? (size_t)p.nhalf : 0;

        // draws (src/samplers.jl:250,:252,:260) of one tile: one thread per walker row, into row buffer rb
        auto tile_draws = [&](long long hs, unsigned tl, unsigned rb, unsigned r) {
            const unsigned w = tl * tr + r;
            if (r < tr && w < W) {
                unsigned j;
                double z, u;
                step_draws<REPLAY>(p, hs, p.shard_begin + w, j, z, u);
                sm.z[rb][r] = z;
                sm.u[rb][r] = u;
                sm.j[rb][r] = j;
                sm.q[rb][r] = filter_q<REPLAY>(p, z, u);
            }
        };
        if (h == p.h0) {  // later half-steps: made in the shadow of the grid barrier
            if (tid < BM) {
                if (T > 0) tile_draws(h, blockIdx.x, 0, tid);
            } else if (tid < 2 * BM) {
                if (T > 1) tile_draws(h, blockIdx.x + gridDim.x, 1, tid - BM);
            }
            __syncthreads();
        }

        // -------------------------------------------------- E(kk): |y|^2, log-density, accept test of tile kk (warps 0-3)
        auto epilogue = [&](unsigned kk) {  // warps 4-11
            const unsigned b = kk & 1, rb = kk % kRowBufs;
            const unsigned w0 = (blockIdx.x + kk * gridDim.x) * tr;
            const int ew = warp - 4;        // 0..7: warps 4-7 reduce columns [0,64), warps 8-11 columns [64,128)
            const int quarter = warp & 3;   // the TMEM lane quarter this warp may read (output dimensions 32q .. 32q+31)
            const int r = (ew & 3) * 32 + lane;  // the walker row of the accept test (warps 4-7)
            double p0 = 0.0;  // current log-density: in flight while the squares are reduced
            if (ew < 4 && (unsigned)r < tr && w0 + r < W) p0 = p.lp[a0 + p.shard_begin + w0 + r];
            mbar_wait(&sm.mma_done[b], (mph >> b) & 1u);
            __syncwarp();
            tc_fence_after();
            const unsigned dbase = tmem + ((unsigned)(quarter * 32) << 16) + kTmemD + b * BM;
            const unsigned cb0 = (unsigned)(ew >> 2) * 64u;
#pragma unroll
            for (unsigned cc = 0; cc < 64; cc += 32) {
                const unsigned cb = cb0 + cc;
                if (cb < tr) {  // warp-uniform
                    unsigned v[32];
                    tmem_ld32(dbase + cb, v);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    float s[32];
#pragma unroll
                    for (int e = 0; e < 32; ++e) {
                        const float y = cb + e < nwcols ? __uint_as_float(v[e]) : 0.0f;  // columns past the MMA's N are stale
                        s[e] = y * y;
                    }
                    // transpose-and-add over the warp's 32 lanes (output dimensions): lane l ends with column cb + l
#pragma unroll
                    for (int hh = 16; hh >= 1; hh >>= 1) {
                        const bool up = (lane & hh) != 0;
#pragma unroll
                        for (int e = 0; e < hh; ++e) {
                            const float send = up ? s[e] : s[e + hh];
                            const float keep = up ? s[e + hh] : s[e];
                            s[e] = keep + __shfl_xor_sync(0xffffffffu, send, hh);
                        }
                    }
                    sm.part[quarter][cb + lane] = s[0];
                }
            }
            tc_fence_before();
            asm volatile("bar.sync 1, 256;" ::: "memory");  // warps 4-11 only
            const unsigned w = w0 + r;
            if (ew < 4 && (unsigned)r < tr && w < W) {
                const float ssf = ((sm.part[0][r] + sm.part[1][r]) + sm.part[2][r]) + sm.part[3][r];
                const unsigned i = p.shard_begin + w;
                const size_t k = a0 + i;
                const double p1 = fp.lognorm - 0.5 * (double)ssf;
                const double tt = (p1 - p0) + (double)sm.q[rb][r] * 0.6931471805599453;  // :260, FP32 filter of K1
                const bool acc = accept_decide(
                    tt, p0, p.margin, [&] { return accept_exact<false>(p.nm1, sm.z[rb][r], p1, p0, sm.u[rb][r]); });
                sm.acc[rb][r] = acc ? 1 : 0;
                if (acc || store) sm.list[rb][atomicAdd(&sm.nlist[rb], 1u)] = (unsigned char)r;
                if (acc) {
                    p.lp[k] = p1;
                    if (!(batch == 1 && clk.burnin_end())) atomicAdd(p.nacc + k, 1u);
                }
                if (batch == 1 && clk.burnin_end()) {  // :285-288
                    p.nacc[i] = 0u;
                    p.nacc[(size_t)p.nhalf + i] = 0u;
                }
                if (store) __stcs(p.chain_lp + chain_row(p, clk.sidx, batch, i), acc ? p1 : p0);
            }
        };

        // -------------------------------------------------- P3(kk): accepted rows (and the chain) of tile kk, all warps
        auto writeback = [&](unsigned kk) {  // warps 1-15 (warp 0 only issues MMAs)
            const unsigned rb = kk % kRowBufs;
            const unsigned w0 = (blockIdx.x + kk * gridDim.x) * tr;
            const unsigned nl = warp == 0 ? 0u : sm.nlist[rb];
            for (unsigned l = (warp - 1) * 2 + half16; l < nl; l += kWorkHalfWarps)
                fused_writeback_row(p, sm, rb, sm.list[rb][l], w0, a0, d, ck, batch, store, clk.sidx);
        };

        K2G_TICK(0);
        for (unsigned k = 0; k <= T; ++k) {
            if (k < T) {
                const unsigned b = k & 1, rb = k % kRowBufs;
                const unsigned w0 = (blockIdx.x + k * gridDim.x) * tr;
                if (tid == 8 * 32) sm.nlist[rb] = 0u;  // last used by tile k-3, whose P3 ended two barriers ago
                // ---------------------------------------------- P1(k): proposals -> swizzled bf16 pieces c[b]  (as K2F)
                {
                    const unsigned hw = (warp - 1) * 2 + half16;  // 30 working half-warps: rows hw, hw+30, ... (warp 0 only issues MMAs)
                    auto row_live = [&](unsigned r) { return r < tr && w0 + r < W; };
                    auto row_load = [&](unsigned r, double2 (&xa)[4], double2 (&xb)[4]) {
                        const unsigned i = p.shard_begin + w0 + r;
                        fused_row_load(p.x + (a0 + i) * d, p.x + (size_t)sm.j[rb][r] * d, true, d, ck, xa, xb);
                    };
                    auto row_emit = [&](unsigned r, const double2 (&xa)[4], const double2 (&xb)[4]) {
                        const double zz = sm.z[rb][r];
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int c = 2 * (ck + 16 * e);
                            const double2 m = *reinterpret_cast<const double2 *>(sm.mu + c);  // zero past d
                            const double v0 = stretch_coord(xb[e].x, xa[e].x, zz) - m.x;  // :255, centred
                            const double v1 = stretch_coord(xb[e].y, xa[e].y, zz) - m.y;
                            unsigned pk[PIECES];
                            split3_pair(v0, v1, pk);
                            const unsigned cp = ck + 16 * e;
                            const unsigned off = sw128_chunk_offset(r, cp >> 2) + ((cp & 3) << 2);
#pragma unroll
                            for (int pc = 0; pc < PIECES; ++pc) *reinterpret_cast<unsigned *>(sm.c[b][pc] + off) = pk[pc];
                        }
                    };
                    if (warp != 0) {
                        double2 xa0[4], xb0[4], xa1[4], xb1[4];
#ifdef KMC_K2G_ROWMAP4
                        // Rows of the two half-warps of a warp differ by 4: with the 128-byte swizzle their 64-byte store
                        // groups then fall into complementary halves of the 32 banks (rows r and r+1 share a half three
                        // times out of four: 2-way conflicts on the STS.32 of the piece stores).  Slot m of warp w' is
                        // n = w' + 15 m -> row 8 (n / 4) + n % 4 + 4 * (half-warp); every row < 152 exactly once.
                        auto slot_row = [&](unsigned m) {
                            const unsigned nn = (unsigned)(warp - 1) + 15u * m;
                            return 8u * (nn >> 2) + (nn & 3u) + 4u * half16;
                        };
                        const unsigned r0 = slot_row(0), r1 = slot_row(1), r2 = slot_row(2), r3 = slot_row(3), r4 = slot_row(4);
#else
                        constexpr unsigned S = kWorkHalfWarps;
                        const unsigned r0 = hw, r1 = hw + S, r2 = hw + 2 * S, r3 = hw + 3 * S, r4 = hw + 4 * S;
#endif
                        const bool l0 = row_live(r0), l1 = row_live(r1), l2 = row_live(r2), l3 = row_live(r3), l4 = row_live(r4);
                        if (l0) row_load(r0, xa0, xb0);
                        if (l1) row_load(r1, xa1, xb1);
                        if (l0) row_emit(r0, xa0, xb0);
                        if (l2) row_load(r2, xa0, xb0);
                        if (l1) row_emit(r1, xa1, xb1);
                        if (l3) row_load(r3, xa1, xb1);
                        if (l2) row_emit(r2, xa0, xb0);
                        if (l4) row_load(r4, xa0, xb0);
                        if (l3) row_emit(r3, xa1, xb1);
                        if (l4) row_emit(r4, xa0, xb0);
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic smem writes -> tensor-core proxy
                __syncthreads();
                K2G_TICK(1);
                // ---------------------------------------------- MMA(k): whole warp 0, elected lane as a predicate
                if (warp == 0) {
                    tc_fence_after();
                    const unsigned leader = elect_one() ? 1u : 0u;
                    const unsigned idesc = idesc_bf16_f32(BM, (int)nwcols);  // M = 128 output dimensions, N = walkers
                    unsigned long long dc[PIECES];
#pragma unroll
                    for (int pc = 0; pc < PIECES; ++pc) dc[pc] = smem_desc_sw128(smem_u32(sm.c[b][pc]));
                    const unsigned dtm = tmem + kTmemD + b * BM;
                    const int pc_c[6] = {2, 0, 1, 1, 0, 0};  // [walker piece, matrix piece], smallest products first
                    const int pc_a[6] = {0, 2, 1, 0, 1, 0};
#pragma unroll
                    for (int pr = 0; pr < 6; ++pr) {
#pragma unroll
                        for (int kq = 0; kq < GK / 16; ++kq) {
                            if (kq >= nk) break;
                            const unsigned long long off16 =
                                (unsigned long long)(((kq >> 2) * (GPIECE_BYTES / 2) + (kq & 3) * 32) >> 4);
                            tc_mma_ts_elect(dtm, tmem + kTmemA + pc_a[pr] * 64 + kq * 8, dc[pc_c[pr]] + off16, idesc,
                                            (pr | kq) ? 1u : 0u, leader);
                        }
                    }
                    tc_commit_elect(&sm.mma_done[b], leader);
                }
                K2G_TICK(2);
            }
            if (k >= 1) {
                if (warp >= 4 && warp < 12) {
                    epilogue(k - 1);
                } else if (warp >= 12) {  // the draws of tile k+1 while warps 4-11 reduce tile k-1
                    if (k + 1 < T) tile_draws(h, blockIdx.x + (k + 1) * gridDim.x, (k + 1) % kRowBufs, (warp - 12) * 32 + lane);
                }
                mph ^= 1u << ((k - 1) & 1);
                __syncthreads();
                K2G_TICK(3);
                writeback(k - 1);
                K2G_TICK(4);
            }
        }
        if (batch == 1) clk.advance(store, p.nthin);
        if (h + 1 < p.h1) {  // the reference's join between the two half-ensemble sweeps (:248/:273)
            target += gridDim.x;
            __syncthreads();
            if (gridDim.x > 1 && tid == 0) barrier_arrive(p.barrier);
            // in the barrier's shadow (independent of the other CTAs): the next half-step's first two tiles' draws
            if (tid >= 32 && tid < 32 + BM) {
                if (T > 0) tile_draws(h + 1, blockIdx.x, 0, tid - 32);
            } else if (tid >= 32 + BM && tid < 32 + 2 * BM) {
                if (T > 1) tile_draws(h + 1, blockIdx.x + gridDim.x, 1, tid - 32 - BM);
            }
#if KMC_K2G_POLL_ACQ
            if (gridDim.x > 1 && tid == (int)blockDim.x - 32) barrier_wait_acquire(p.barrier, target);  // an idle warp
#else
            if (gridDim.x > 1 && tid == 0) barrier_wait(p.barrier, target);
#endif
            __syncthreads();
        }
        K2G_TICK(5);
    }
#ifdef KMC_K2F_PROF
    if (tid == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1))
        printf("K2G cta %d cycles: draws %lld P1 %lld mma-issue %lld epilogue %lld P3 %lld barrier %lld (half-steps %lld)\n",
               (int)blockIdx.x, pt[0], pt[1], pt[2], pt[3], pt[4], pt[5], (long long)(p.h1 - p.h0));
#endif

    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

}  // namespace tc
}  // namespace kmc
