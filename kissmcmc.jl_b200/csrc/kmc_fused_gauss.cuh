// kmc_fused_gauss.cuh -- K2F: the whole stretch-move half-step of the dense Gaussian plugin
// (BASELINE.json configs[2], 16 < d <= 128) as ONE persistent tcgen05 kernel.
//
// One CTA per SM, 512 threads, cooperative launch over a whole range of half-steps (grid barrier
// between half-steps like emcee_run_kernel).  The matrix pieces A (3 x 32 KB bf16, SWIZZLE_128B)
// are loaded once by TMA and stay in shared memory.  Per 128-walker tile:
//
//   P1  all 16 warps, 16 lanes per walker (two walkers in flight per half-warp), 8 columns per lane (the draws,
//       src/samplers.jl:250,:252,:260, were made one thread per walker while the previous tile's GEMM ran):
//       gather x_j (one contiguous 8d-byte row) and x_k, proposal y = xj + z(xk - xj) (:255) in FP64,
//       centre, split into three bf16 pieces and store each 16-byte chunk DIRECTLY into the swizzled
//       K-major UMMA tile in shared memory (chunk index XOR row%8 inside each 8 x 128 B atom) --
//       the proposal never goes to global memory.   fence.proxy.async + bar.sync
//   P2  one thread issues the 48 tcgen05.mma (6 piece pairs x 8 k-steps, M=128 N=128 K=16, FP32 in
//       TMEM) and commits to an mbarrier; warps 0-3 (thread = walker row) read the accumulator with
//       tcgen05.ld, reduce |y|^2 over the first d columns, form logp and run the exact FP64 accept
//       test (:260), update logp / accept counter / thinned logp chain
//   P3  all warps: accepted walkers (and all, when the iteration is stored) recompute y with the
//       same three IEEE operations and write x (:261) / the chain (:268-272)
//
// Traffic per half-step ~ read x_k, x_j once + rewrite accepted rows: close to the algorithmic
// 24d+24 bytes per walker-step, instead of ~3x that for the three-kernel pipeline.
#pragma once
#include "kmc_batched.cuh"
#include "kmc_tc.cuh"

namespace kmc {
namespace tc {

constexpr int kFusedThreads = 512;

struct __align__(1024) FusedSmem {
    unsigned char a[PIECES][GPIECE_BYTES];  // matrix pieces (B operand), resident
    unsigned char c[PIECES][GPIECE_BYTES];  // centred proposal pieces (A operand) of the current tile
    unsigned long long afull, mma_done;
    unsigned tmem_base;
    double z[2][BM], u[2][BM];   // per-row draws, double-buffered by tile parity (P3 of tile t overlaps P1 of tile t+1)
    unsigned j[2][BM];
    alignas(16) double mu[GK];   // the mean, zero-padded to 128 columns (read as double2)
    float q[2][BM];              // FP32 accept-filter term of the draw (filter_q), NaN = exact path
    unsigned nlist[2];           // rows of the tile that P3 has to touch (accepted, or all when the iteration is stored)
    unsigned char list[2][BM];
    unsigned char acc[2][BM];
};

struct FusedParams {
    const double *mu;  // [d] (device)
    double lognorm;
    int d;
};

// byte offset of the 16-byte chunk (row r, chunk index ck in 0..15 = 8 bf16 columns each) inside a
// piece stored as [2 k-halves][128 rows][128 B] with the 128-byte swizzle
__device__ __forceinline__ bool elect_one() {
    unsigned pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

__device__ __forceinline__ unsigned sw128_chunk_offset(unsigned r, unsigned ck) {
    const unsigned kh = ck >> 3, c8 = ck & 7;
    return kh * (GPIECE_BYTES / 2) + (r >> 3) * 1024 + (r & 7) * 128 + ((c8 ^ (r & 7)) << 4);
}

// Columns 2 cp, 2 cp + 1 (column pairs cp = ck + 16 e, e = 0..3) of a walker's own row xk and, when load_j, of its partner's
// row xj (an L2 load: other CTAs write it), zero past d.  Even d: one 16-byte load per column pair.
__device__ __forceinline__ void fused_row_load(const double *xk, const double *xj, bool load_j, int d, unsigned ck,
                                               double2 (&xa)[4], double2 (&xb)[4]) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int c = 2 * (ck + 16 * e);
        xa[e] = make_double2(0.0, 0.0);
        xb[e] = make_double2(0.0, 0.0);
        if ((d & 1) == 0) {
            if (c < d) {
                xa[e] = *reinterpret_cast<const double2 *>(xk + c);
                if (load_j) xb[e] = __ldcg(reinterpret_cast<const double2 *>(xj + c));
            }
        } else {
            if (c < d) {
                xa[e].x = xk[c];
                if (load_j) xb[e].x = __ldcg(xj + c);
            }
            if (c + 1 < d) {
                xa[e].y = xk[c + 1];
                if (load_j) xb[e].y = __ldcg(xj + c + 1);
            }
        }
    }
}

// P3 of listed row rr of the tile whose first walker is w0: an accepted row recomputes its proposal with the same three
// operations as P1 (:255, same bits) and writes it back (:261); in a stored iteration the row goes to the chain (:268-272).
// A half-warp per row, lane ck owns the column pairs of fused_row_load.
template <class Smem>
__device__ __forceinline__ void fused_writeback_row(const RunParams &p, const Smem &sm, unsigned rb, unsigned rr, unsigned w0,
                                                    size_t a0, int d, unsigned ck, unsigned batch, bool store, long long sidx) {
    const bool accr = sm.acc[rb][rr] != 0;
    const unsigned i = p.shard_begin + w0 + rr;
    double *xk = p.x + (a0 + i) * d;
    double2 xa[4], xb[4];
    fused_row_load(xk, p.x + (size_t)sm.j[rb][rr] * d, accr, d, ck, xa, xb);
    const double z = sm.z[rb][rr];
    const size_t o = store ? chain_row(p, sidx, batch, i) : 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const int c = 2 * (ck + 16 * e);
        const double v0 = accr ? stretch_coord(xb[e].x, xa[e].x, z) : xa[e].x;
        const double v1 = accr ? stretch_coord(xb[e].y, xa[e].y, z) : xa[e].y;
        if ((d & 1) == 0) {  // even d: rows are 16-byte aligned, one 16-byte store per column pair
            if (c < d) {
                if (accr) *reinterpret_cast<double2 *>(xk + c) = make_double2(v0, v1);
                if (store) __stcs(reinterpret_cast<double2 *>(p.chain_x + o * d + c), make_double2(v0, v1));
            }
        } else {
            if (c < d) {
                if (accr) xk[c] = v0;
                if (store) __stcs(p.chain_x + o * d + c, v0);
            }
            if (c + 1 < d) {
                if (accr) xk[c + 1] = v1;
                if (store) __stcs(p.chain_x + o * d + c + 1, v1);
            }
        }
    }
}

template <bool REPLAY>
__global__ void __launch_bounds__(kFusedThreads, 1)
gaussian_fused_kernel(const __grid_constant__ CUtensorMap mapA, const RunParams p, const FusedParams fp) {
    extern __shared__ unsigned char smem_raw[];
    FusedSmem &sm = *reinterpret_cast<FusedSmem *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = tid >> 5;
    const int d = fp.d;

    if (tid < GK) sm.mu[tid] = tid < d ? fp.mu[tid] : 0.0;
    if (tid == 0) {
        sm.nlist[0] = sm.nlist[1] = 0u;
        mbar_init(&sm.afull, 1);
        mbar_init(&sm.mma_done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 128;" ::"r"(smem_u32(&sm.tmem_base))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    // lane-0 shuffle: tells ptxas the TMEM base is warp-uniform, so the MMA issue loop keeps it in a uniform register
    // instead of an ELECT + R2UR waterfall per tcgen05.mma (the issue stream, not the tensor pipe, was the bound)
    const unsigned tmem = __shfl_sync(0xffffffffu, sm.tmem_base, 0);
    if (tid == 0) {  // the matrix: once per CTA
        mbar_expect_tx(&sm.afull, PIECES * GPIECE_BYTES);
        for (int pc = 0; pc < PIECES; ++pc)
            for (int kh = 0; kh < 2; ++kh)
                tma_load_2d(sm.a[pc] + kh * (GPIECE_BYTES / 2), &mapA, kh * 64, pc * GN, &sm.afull);
    }
    mbar_wait(&sm.afull, 0);

    // Tiles are balanced over the grid: every CTA gets the same number of tiles per half-step and a tile holds
    // tr <= 128 walkers (2^15 active walkers on 148 CTAs: 296 tiles of 111 rows instead of 256 of 128, of which 40
    // CTAs would get one and 108 two).  A row of the GEMM depends on its own walker only, so the tiling changes no bit.
    const unsigned W = p.shard_end - p.shard_begin;
    const unsigned waves = ((W + BM - 1) / BM + gridDim.x - 1) / gridDim.x;
    const unsigned tr = min((unsigned)BM, (W + waves * gridDim.x - 1) / (waves * gridDim.x));  // walkers per tile
    const unsigned ntiles = (W + tr - 1) / tr;
    const int nk = (d + 15) / 16;        // k-steps (and 16-column groups of the output) that hold data
    const unsigned half16 = lane >> 4;   // which of the warp's two walkers
    const unsigned ck = lane & 15;       // 16-byte chunk = columns 8*ck .. 8*ck+7
    unsigned mma_phase = 0, tpar = 0;  // tpar: parity of the tile counter of this CTA
    ThinClock<> clk{p.n0, p.phase0, p.sidx0};
    unsigned long long target = p.bar_base;
#ifdef KMC_K2F_PROF
    long long pt[6] = {0, 0, 0, 0, 0, 0}, pc0 = clock64();
#define K2F_TICK(i) do { const long long c_ = clock64(); pt[i] += c_ - pc0; pc0 = c_; } while (0)
#else
#define K2F_TICK(i) do { } while (0)
#endif

    for (long long h = p.h0; h < p.h1; ++h) {
        const unsigned batch = (unsigned)(h & 1);
        const bool store = clk.store();
        const size_t a0 = batch ? (size_t)p.nhalf : 0;

        // draws (src/samplers.jl:250,:252,:260) of one tile: one thread per walker row, into parity `par`
        auto tile_draws = [&](long long hs, unsigned tl, unsigned par, unsigned r) {
            const unsigned w = tl * tr + r;
            if (r < tr && w < W) {
                unsigned j;
                double z, u;
                step_draws<REPLAY>(p, hs, p.shard_begin + w, j, z, u);
                sm.z[par][r] = z;
                sm.u[par][r] = u;
                sm.j[par][r] = j;
                sm.q[par][r] = filter_q<REPLAY>(p, z, u);
            }
        };
        // the first tile's draws of this half-step were made in the shadow of the previous grid barrier
        if (h == p.h0) {
            if (blockIdx.x < ntiles && tid < BM) tile_draws(h, blockIdx.x, tpar, tid);
            __syncthreads();
        }
        K2F_TICK(0);
        for (unsigned tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const unsigned w0 = tile * tr;
            // ------------------------------------------------ P1: proposals -> swizzled bf16 pieces
            // lane handles column pairs cp = ck + 16 e (columns 2cp, 2cp+1), e = 0..3: every load instruction of
            // a half-warp reads 256 contiguous bytes of the row.  Half-warp hw owns rows hw, hw+32, hw+64, hw+96 of
            // the tile; the loads of the next row are issued before the math of the current one (two register
            // buffers), so the L2 latency and the LSU work of one row hide behind the FP64 / conversion work of another.
            {
                const unsigned hw = warp * 2 + half16;
                auto row_live = [&](unsigned r) { return r < tr && w0 + r < W; };
                auto row_load = [&](unsigned r, double2 (&xa)[4], double2 (&xb)[4]) {
                    const unsigned i = p.shard_begin + w0 + r;
                    fused_row_load(p.x + (a0 + i) * d, p.x + (size_t)sm.j[tpar][r] * d, true, d, ck, xa, xb);
                };
                auto row_emit = [&](unsigned r, const double2 (&xa)[4], const double2 (&xb)[4]) {
                    const double zz = sm.z[tpar][r];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int c = 2 * (ck + 16 * e);
                        const double2 m = *reinterpret_cast<const double2 *>(sm.mu + c);  // zero past d
                        // :255, centred; columns past d were loaded as zeros and stay zero
                        const double v0 = stretch_coord(xb[e].x, xa[e].x, zz) - m.x;
                        const double v1 = stretch_coord(xb[e].y, xa[e].y, zz) - m.y;
                        unsigned pk[PIECES];
                        split3_pair(v0, v1, pk);
                        const unsigned cp = ck + 16 * e;  // column pair -> 4 bytes inside chunk cp/4
                        const unsigned off = sw128_chunk_offset(r, cp >> 2) + ((cp & 3) << 2);
#pragma unroll
                        for (int pc = 0; pc < PIECES; ++pc) *reinterpret_cast<unsigned *>(sm.c[pc] + off) = pk[pc];
                    }
                };
                // rows past the tile are skipped: whatever the buffer holds there only reaches accumulator rows nobody reads
                double2 xa0[4], xb0[4], xa1[4], xb1[4];
                const bool l0 = row_live(hw), l1 = row_live(hw + 32), l2 = row_live(hw + 64), l3 = row_live(hw + 96);
                if (l0) row_load(hw, xa0, xb0);
                if (l1) row_load(hw + 32, xa1, xb1);
                if (l0) row_emit(hw, xa0, xb0);
                if (l2) row_load(hw + 64, xa0, xb0);
                if (l1) row_emit(hw + 32, xa1, xb1);
                if (l3) row_load(hw + 96, xa1, xb1);
                if (l2) row_emit(hw + 64, xa0, xb0);
                if (l3) row_emit(hw + 96, xa1, xb1);
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic smem writes -> tensor-core proxy
            __syncthreads();
            K2F_TICK(1);
            // ------------------------------------------------ P2: tcgen05 GEMM, epilogue, accept
            if (warp == 0) {
                // The WHOLE warp runs the issue loop, converged: every operand (descriptors, TMEM address, instruction
                // descriptor) is warp-uniform and stays in uniform registers, and the one elected lane is a predicate on
                // the tcgen05 instructions themselves.  Issued from inside `if (tid == 0)` each MMA cost an ELECT /
                // BRA.U.ANY waterfall and ~18 instructions (~100 cycles against the 56-cycle tensor floor of a
                // 128x112x16 MMA: the issue stream, not the tensor pipe, paced the GEMM).  A descriptor of a later
                // k-step is the piece's descriptor plus a compile-time constant in its 16-byte address field.
                tc_fence_after();
                const unsigned leader = elect_one() ? 1u : 0u;
                // only the first ceil(d/16) k-steps and ceil(d/16)*16 output columns: the rest are zero padding
                // (adding +0 products changes no bit, so this equals the full 128x128x128 product)
                const unsigned idesc = idesc_bf16_f32(BM, nk * 16);
                unsigned long long dc[PIECES], da[PIECES];
#pragma unroll
                for (int pc = 0; pc < PIECES; ++pc) {
                    dc[pc] = smem_desc_sw128(smem_u32(sm.c[pc]));
                    da[pc] = smem_desc_sw128(smem_u32(sm.a[pc]));
                }
                const int pc_c[6] = {2, 0, 1, 1, 0, 0};
                const int pc_a[6] = {0, 2, 1, 0, 1, 0};
#pragma unroll
                for (int pr = 0; pr < 6; ++pr) {
#pragma unroll
                    for (int k = 0; k < GK / 16; ++k) {
                        if (k >= nk) break;
                        const unsigned long long off16 = (unsigned long long)(((k >> 2) * (GPIECE_BYTES / 2) + (k & 3) * 32) >> 4);
                        tc_mma_elect(tmem, dc[pc_c[pr]] + off16, da[pc_a[pr]] + off16, idesc, (pr | k) ? 1u : 0u, leader);
                    }
                }
                tc_commit_elect(&sm.mma_done, leader);
            }
            if (warp < 4) {
                double p0 = 0.0;  // current log-density: fetched while the GEMM runs
                if ((unsigned)(warp * 32 + lane) < tr && w0 + warp * 32 + lane < W)
                    p0 = p.lp[a0 + p.shard_begin + w0 + warp * 32 + lane];
                mbar_wait(&sm.mma_done, mma_phase);
                K2F_TICK(5);
                __syncwarp();  // lane 0 came here from the MMA issue: converge before the .aligned TMEM loads
                tc_fence_after();
                const int r = warp * 32 + lane;
                double ss = 0.0;
#pragma unroll 1
                for (int cb = 0; cb < GN; cb += 32) {
                    if (cb >= d) break;
                    unsigned v[32];
                    tmem_ld32(tmem + ((unsigned)(warp * 32) << 16) + cb, v);
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    float part = 0.0f;
#pragma unroll
                    for (int e = 0; e < 32; ++e) {
                        const float y = cb + e < nk * 16 ? __uint_as_float(v[e]) : 0.0f;  // columns past the MMA's N are stale
                        part = fmaf(y, y, part);
                    }
                    ss += (double)part;
                }
                tc_fence_before();
                const unsigned w = w0 + r;
                if ((unsigned)r < tr && w < W) {
                    const unsigned i = p.shard_begin + w;
                    const size_t k = a0 + i;
                    const double p1 = fp.lognorm - 0.5 * ss;
                    // :260 -- the FP32 filter of kmc_kernels.cuh decides exactly like the FP64 expression whenever
                    // |tt| is above its rigorous margin; everything else takes the FP64 expression itself
                    const double tt = (p1 - p0) + (double)sm.q[tpar][r] * 0.6931471805599453;
                    bool acc;
                    if (tt > (double)p.margin) acc = true;
                    else if (tt < -(double)p.margin) acc = false;
                    else acc = accept_exact<false>(p.nm1, sm.z[tpar][r], p1, p0, sm.u[tpar][r]);
                    sm.acc[tpar][r] = acc ? 1 : 0;
                    if (acc || store) sm.list[tpar][atomicAdd(&sm.nlist[tpar], 1u)] = (unsigned char)r;
                    if (acc) {
                        p.lp[k] = p1;
                        if (!(batch == 1 && clk.burnin_end())) atomicAdd(p.nacc + k, 1u);  // fire-and-forget; only this thread touches the counter
                    }
                    if (batch == 1 && clk.burnin_end()) {  // :285-288
                        p.nacc[i] = 0u;
                        p.nacc[(size_t)p.nhalf + i] = 0u;
                    }
                    if (store) __stcs(p.chain_lp + chain_row(p, clk.sidx, batch, i), acc ? p1 : p0);
                }
            }
            else if (warp < 8) {  // idle during the GEMM: the NEXT tile's draws, into the other parity
                if (tile + gridDim.x < ntiles) tile_draws(h, tile + gridDim.x, tpar ^ 1, (warp - 4) * 32 + lane);
            } else if (tid == 8 * 32) {
                sm.nlist[tpar ^ 1] = 0u;  // the previous tile's P3 finished before the barrier that closed this tile's P1
            }
            mma_phase ^= 1;
            __syncthreads();
            K2F_TICK(2);
            // ------------------------------------------------ P3: accepted rows (and the chain)
            // No barrier after P3: the next tile's P1 only writes sm.c (free since the MMA completed) and the
            // OTHER parity of the per-row arrays; the bar.sync after that P1 orders everything else.
            // One listed row per half-warp at a time (two in flight, or a load/compute pipeline as in P1, spill at the
            // 128-register cap of a 512-thread CTA and were measured slower: 44 and 36 us per half-step against 21).
            const unsigned nl = sm.nlist[tpar];
            for (unsigned l0 = warp * 2 + half16; l0 < nl; l0 += 2 * (kFusedThreads / 32)) {
                double2 xa[1][4], xb[1][4];
                unsigned rr[1];
                bool live[1], accr[1];
#pragma unroll
                for (int t = 0; t < 1; ++t) {
                    const unsigned l = l0 + t * 2 * (kFusedThreads / 32);
                    live[t] = l < nl;
                    rr[t] = live[t] ? sm.list[tpar][l] : 0u;
                    accr[t] = live[t] && sm.acc[tpar][rr[t]] != 0;
                    if (!live[t]) continue;
                    const double *xk = p.x + (a0 + p.shard_begin + w0 + rr[t]) * d;
                    const double *xj = p.x + (size_t)sm.j[tpar][rr[t]] * d;
                    fused_row_load(xk, xj, accr[t], d, ck, xa[t], xb[t]);
                }
#pragma unroll
                for (int t = 0; t < 1; ++t) {
                    if (!live[t]) continue;
                    const unsigned i = p.shard_begin + w0 + rr[t];
                    double *xk = p.x + (a0 + i) * d;
                    const double z = sm.z[tpar][rr[t]];
                    const size_t o = store ? chain_row(p, clk.sidx, batch, i) : 0;
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int c = 2 * (ck + 16 * e);
                        const double v0 = accr[t] ? stretch_coord(xb[t][e].x, xa[t][e].x, z) : xa[t][e].x;  // :255, same bits
                        const double v1 = accr[t] ? stretch_coord(xb[t][e].y, xa[t][e].y, z) : xa[t][e].y;
                        if ((d & 1) == 0) {  // even d: rows are 16-byte aligned, one 16-byte store per column pair
                            if (c < d) {
                                if (accr[t]) *reinterpret_cast<double2 *>(xk + c) = make_double2(v0, v1);                  // :261
                                if (store) __stcs(reinterpret_cast<double2 *>(p.chain_x + o * d + c), make_double2(v0, v1));  // :268-272
                            }
                        } else {
                            if (c < d) {
                                if (accr[t]) xk[c] = v0;
                                if (store) __stcs(p.chain_x + o * d + c, v0);
                            }
                            if (c + 1 < d) {
                                if (accr[t]) xk[c + 1] = v1;
                                if (store) __stcs(p.chain_x + o * d + c + 1, v1);
                            }
                        }
                    }
                }
            }
            tpar ^= 1;
            K2F_TICK(3);
        }
        if (batch == 1) clk.advance(store, p.nthin);
        if (h + 1 < p.h1) {  // the reference's join between the two half-ensemble sweeps (:248/:273)
            target += gridDim.x;
            __syncthreads();
            if (gridDim.x > 1 && tid == 0) barrier_arrive(p.barrier);
            // in the barrier's shadow (independent of the other CTAs): the next half-step's first tile's draws, into
            // the parity the next tile uses (the last tile's P3, which read the other parity, ended before the bar.sync)
            if (blockIdx.x < ntiles && tid >= 32 && tid < 32 + BM) tile_draws(h + 1, blockIdx.x, tpar, tid - 32);
            if (gridDim.x > 1 && tid == 0) barrier_wait(p.barrier, target);
            __syncthreads();
        }
        K2F_TICK(4);
    }
#ifdef KMC_K2F_PROF
    if (tid == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1))
        printf("K2F cta %d cycles: draws %lld P1 %lld mma %lld epilogue %lld P3 %lld barrier %lld (half-steps %lld)\n", (int)blockIdx.x,
               pt[0], pt[1], pt[5], pt[2], pt[3], pt[4], (long long)(p.h1 - p.h0));
#endif

    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 128;" ::"r"(tmem) : "memory");
}

}  // namespace tc
}  // namespace kmc
