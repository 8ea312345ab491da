// kmc_tc.cuh -- tcgen05 (5th-gen tensor core) log-density kernels for sm_100a.
//
// K3  logistic_tc_kernel: the walkers x data logits GEMM of Bayesian logistic regression
//     (BASELINE.json configs[3]) fused with its softplus row reduction.
//
//       S[w][n] = theta_w . x_n          [W x 32] . [32 x N]   (N ~ 1e6 streamed, W = active half)
//       out[w]  = sum_n ( |S[w][n]|/2 + log1p(exp(-|S[w][n]|)) )   = sum_n softplus(S) - sum_n S/2
//
//     The caller adds the exact FP64 terms  theta.(X^T (y - 1/2))  and the prior (logistic_tc_finish_kernel).
//
//   * operands: X is bf16 (the plugin requires bf16-representable data, checked at creation, so
//     this is exact); theta (FP64) is split into three bf16 pieces hi+mid+lo (24 significant
//     bits).  bf16 x bf16 products are exact in FP32, the accumulation is FP32 in TMEM, so a
//     logit carries an absolute error of a few 2^-24 sum_k |theta_k x_nk| and the N rows add
//     theirs up.  Bound per point, derived in tests/test_tc_error_model.py (u = 2^-24,
//     m = ceil(d/16)):  |R_tc - R| <= u [(0.5 + 1.05 m) sum_n sum_k |theta_k x_nk|
//     + 8.5 sum_n |theta . x_n|] + 5 u N  <=  13.2 u sum_n sum_k |theta_k x_nk| + 5 u N;
//     a difference of two points, the sum of their bounds.  It grows with the logit scale:
//     ~1.3 per point at the bench problem (d = 32, N = 1e6, theta*), ~13 with the data drawn
//     from 16 theta*; on the bench problem a B200 shows ~3e-2 (a common offset) per point and
//     2e-3 on differences.
//   * one CTA per SM, persistent over work items (walker tile of 128, chunk of data tiles):
//       warp 0     TMA producer: A = 3 theta pieces [128 x 32] once per item, B = X tile
//                  [256 x 32] per stage (4 stages), SWIZZLE_64B K-major, mbarrier complete_tx
//       warp 1     MMA issuer: one elected thread, 6 x tcgen05.mma.cta_group::1.kind::f16
//                  (M=128, N=256, K=16) per tile = 3 pieces x 2 k-steps, lo piece first;
//                  tcgen05.commit frees the smem stage and publishes the accumulator
//       warps 2-17 epilogue: tcgen05.ld 32x32b.x32 from the double-buffered TMEM accumulator
//                  (2 x 256 columns = all 512); per logit one MUFU ex2, one FFMA (running product of
//                  1 + 2^-|s'|, one lg2 per 32 columns) and one FADD (sum of |s'|); FP32 partial
//                  per 32 columns, FP64 running sum per row, tail columns masked
//   * every mbarrier wait has a watchdog (trap after ~2 s) so a bad descriptor cannot hang the GPU.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>

#include "kmc_device.cuh"

namespace kmc {
namespace tc {

constexpr int BM = 128, BN = 256, STAGES = 4, ACC = 2, PIECES = 3;  // K of the logistic GEMM is a template parameter: 32 or 64
#ifndef KMC_K3_EPI
#define KMC_K3_EPI 16
#endif
constexpr int kEpiWarps = KMC_K3_EPI;            // 8 or 16: 2 or 4 epilogue warps per scheduler
constexpr int kEpiParts = kEpiWarps / 4;         // column parts of the accumulator (a warp owns 32 rows x BN/kEpiParts columns)
constexpr int kEpiCols = BN / kEpiParts;
constexpr int kThreads = 32 * (2 + kEpiWarps);
// d is zero-padded to BK = 32 (64-byte rows, SWIZZLE_64B) or, for 32 < d <= 64, to BK = 64 (128-byte rows, SWIZZLE_128B)
template <int BK>
struct __align__(1024) Smem {
    static constexpr int kABytes = BM * BK * 2;  // 8 / 16 KB per theta piece
    static constexpr int kBBytes = BN * BK * 2;  // 16 / 32 KB per X tile
    unsigned char a[PIECES][kABytes];
    unsigned char b[STAGES][kBBytes];
    unsigned long long full[STAGES], empty[STAGES], tfull[ACC], tempty[ACC], afull, aempty;
    unsigned tmem_base;
    double comb[kEpiParts - 1][BM];
};

__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(unsigned long long *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity) {
    const unsigned a = smem_u32(bar);
    const long long t0 = clock64();
    unsigned done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(a), "r"(parity)
            : "memory");
        if (!done && clock64() - t0 > 4000000000LL) __trap();  // watchdog: never hang the device
    }
}
__device__ __forceinline__ void tma_load_2d(void *dst, const CUtensorMap *map, int x, int y, unsigned long long *bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"((unsigned long long)map), "r"(smem_u32(bar)), "r"(x), "r"(y)
        : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(unsigned long long *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
// D[tmem] (+)= A[smem] . B[smem]^T, kind::f16 (bf16 in, fp32 accumulate), issued by one thread
__device__ __forceinline__ void tc_mma(unsigned tmem_d, unsigned long long adesc, unsigned long long bdesc,
                                       unsigned idesc, unsigned accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// The same two instructions for a converged warp: every lane executes the asm with warp-uniform operands, only the
// elected lane (leader != 0) issues.  No divergent branch around the instruction, so ptxas keeps the operands in
// uniform registers instead of an ELECT / BRA.U.ANY waterfall per MMA.
__device__ __forceinline__ void tc_mma_elect(unsigned tmem_d, unsigned long long adesc, unsigned long long bdesc,
                                             unsigned idesc, unsigned accumulate, unsigned leader) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "setp.ne.b32 q, %5, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate), "r"(leader)
        : "memory");
}
__device__ __forceinline__ void tc_commit_elect(unsigned long long *bar, unsigned leader) {
    asm volatile(
        "{\n\t.reg .pred q;\n\t"
        "setp.ne.b32 q, %1, 0;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)),
        "r"(leader)
        : "memory");
}

// K-major operand tile with 64-byte rows (32 bf16), SWIZZLE_64B: 8-row groups are 512 B apart
// (SBO), LBO unused (1), descriptor version 1 (sm_100), layout type 4.  cute/arch/mma_sm100_desc.hpp.
__device__ __forceinline__ unsigned long long smem_desc_sw64(unsigned addr) {
    unsigned long long d = 0;
    d |= (unsigned long long)((addr >> 4) & 0x3FFF);
    d |= (unsigned long long)1 << 16;            // leading byte offset (ignored for swizzled K-major)
    d |= (unsigned long long)(512 >> 4) << 32;   // stride byte offset: 8 rows x 64 B
    d |= (unsigned long long)1 << 46;            // version
    d |= (unsigned long long)4 << 61;            // SWIZZLE_64B
    return d;
}
// K-major operand tile with 128-byte rows (64 bf16), SWIZZLE_128B: 8-row groups are 1024 B apart.
__device__ __forceinline__ unsigned long long smem_desc_sw128(unsigned addr) {
    unsigned long long d = 0;
    d |= (unsigned long long)((addr >> 4) & 0x3FFF);
    d |= (unsigned long long)1 << 16;
    d |= (unsigned long long)(1024 >> 4) << 32;  // 8 rows x 128 B
    d |= (unsigned long long)1 << 46;
    d |= (unsigned long long)2 << 61;            // SWIZZLE_128B
    return d;
}
template <int BK>
__device__ __forceinline__ unsigned long long smem_desc_k(unsigned addr) {
    if constexpr (BK == 32) return smem_desc_sw64(addr);
    else return smem_desc_sw128(addr);
}
// kind::f16 instruction descriptor: D = F32, A = B = BF16, both K-major, M = 128, N = 256.
__host__ __device__ constexpr unsigned idesc_bf16_f32(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(n >> 3) << 17) | ((unsigned)(m >> 4) << 24);
}

// 2^-|s|: one MUFU.EX2 (the abs / neg fold into the operand modifiers)
__device__ __forceinline__ float ex2_neg_abs(float s) {
    float t;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(t) : "f"(-fabsf(s)));
    return t;
}

// The same function on the FMA / ALU pipes (no MUFU): 2^-a = 2^-i * 2^(i-a), i = round(a) taken from the low mantissa
// bits of a + 1.5*2^23, 2^x on [-1/2, 1/2] as a degree-5 polynomial (max relative error 2.0e-7, MUFU.EX2: 2.4e-7), the
// exponent subtracted as an integer.  Every KMC_K3_POLY-th column of the epilogue takes this path so that the XU pipe
// (16 lanes/clk/SM, the bound of the all-MUFU epilogue) and the issue slots are loaded evenly.
#ifndef KMC_K3_POLY
#define KMC_K3_POLY 4
#endif
__device__ __forceinline__ float ex2_neg_abs_poly(float s) {
    const float a = fminf(fabsf(s), 126.0f);
    const float r = a + 12582912.0f;
    const float x = (r - 12582912.0f) - a;
    float q = 0.0013266970636323094f;
    q = fmaf(q, x, 0.009675459936261177f);
    q = fmaf(q, x, 0.05550742521882057f);
    q = fmaf(q, x, 0.24022121727466583f);
    q = fmaf(q, x, 0.6931469440460205f);
    q = fmaf(q, x, 1.0000001192092896f);
    return __int_as_float(__float_as_int(q) - (__float_as_int(r) << 23));
}
// column j of a 32-column chunk (j is a compile-time constant after unrolling)
__device__ __forceinline__ float ex2_neg_abs_col(float s, int j) {
    constexpr int P = KMC_K3_POLY > 0 ? KMC_K3_POLY : 1;
    if (KMC_K3_POLY > 0 && j % P == P - 1) return ex2_neg_abs_poly(s);
    return ex2_neg_abs(s);
}

// 32 consecutive FP32 columns of this thread's TMEM lane -> registers (asynchronous until wait::ld)
__device__ __forceinline__ void tmem_ld32(unsigned taddr, unsigned (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}

struct LogitParams {
    long long W;          // points (rows of theta)
    long long N;          // data rows
    int mtiles;           // ceil(W / 128)
    int nchunks;          // data chunks (work items per m-tile)
    int tiles_per_chunk;  // data tiles of 256 rows per chunk
    int ntiles;           // ceil(N / 256)
    long long wpad;       // rows per theta piece in the piece buffer (mtiles * 128)
    double *part;         // [nchunks][W] partial sums of softplus
};

template <int BK>
__global__ void __launch_bounds__(kThreads, 1)
logistic_tc_kernel(const __grid_constant__ CUtensorMap mapA, const __grid_constant__ CUtensorMap mapX,
                   const LogitParams p) {
    static_assert(BK == 32 || BK == 64, "K-major rows of 64 or 128 bytes");
    extern __shared__ unsigned char smem_raw[];
    using SmemT = Smem<BK>;
    constexpr int kABytes = SmemT::kABytes, kBBytes = SmemT::kBBytes;
    SmemT &sm = *reinterpret_cast<SmemT *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&sm.full[s], 1);
            mbar_init(&sm.empty[s], 1);
        }
        for (int a = 0; a < ACC; ++a) {
            mbar_init(&sm.tfull[a], 1);
            mbar_init(&sm.tempty[a], kEpiWarps);
        }
        mbar_init(&sm.afull, 1);
        mbar_init(&sm.aempty, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {  // TMEM: all 512 columns (2 accumulators of 256)
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&sm.tmem_base))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem = sm.tmem_base;
    const int nitems = p.mtiles * p.nchunks;

    if (warp == 0) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            unsigned stage = 0, phase = 0, aphase = 0;
            for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
                const int mt = item % p.mtiles, ch = item / p.mtiles;
                mbar_wait(&sm.aempty, aphase ^ 1);  // MMA finished with the previous item's theta tile
                mbar_expect_tx(&sm.afull, PIECES * kABytes);
                for (int pc = 0; pc < PIECES; ++pc)
                    tma_load_2d(sm.a[pc], &mapA, 0, (int)(pc * p.wpad + (long long)mt * BM), &sm.afull);
                aphase ^= 1;
                const int t0 = ch * p.tiles_per_chunk, t1 = min(p.ntiles, t0 + p.tiles_per_chunk);
                for (int t = t0; t < t1; ++t) {
                    mbar_wait(&sm.empty[stage], phase ^ 1);
                    mbar_expect_tx(&sm.full[stage], kBBytes);
                    tma_load_2d(sm.b[stage], &mapX, 0, t * BN, &sm.full[stage]);  // rows past N are zero-filled
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            constexpr unsigned idesc = idesc_bf16_f32(BM, BN);
            unsigned stage = 0, phase = 0, aphase = 0, acc = 0, accphase = 0;
            for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
                const int ch = item / p.mtiles;
                mbar_wait(&sm.afull, aphase);
                aphase ^= 1;
                tc_fence_after();
                const int t0 = ch * p.tiles_per_chunk, t1 = min(p.ntiles, t0 + p.tiles_per_chunk);
                for (int t = t0; t < t1; ++t) {
                    mbar_wait(&sm.tempty[acc], accphase ^ 1);  // epilogue drained this accumulator
                    mbar_wait(&sm.full[stage], phase);         // X tile landed
                    tc_fence_after();
                    const unsigned d = tmem + acc * BN;
                    const unsigned bbase = smem_u32(sm.b[stage]);
#pragma unroll
                    for (int pc = PIECES - 1; pc >= 0; --pc) {  // lo, mid, hi: small terms first
                        const unsigned abase = smem_u32(sm.a[pc]);
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k)  // 32 bytes per k-step inside the swizzled row
                            tc_mma(d, smem_desc_k<BK>(abase + k * 32), smem_desc_k<BK>(bbase + k * 32), idesc,
                                   (pc != PIECES - 1 || k != 0) ? 1u : 0u);
                    }
                    tc_commit(&sm.empty[stage]);  // smem stage reusable once these MMAs retire
                    tc_commit(&sm.tfull[acc]);    // accumulator ready for the epilogue
                    if (++stage == STAGES) {
                        stage = 0;
                        phase ^= 1;
                    }
                    if (++acc == ACC) {
                        acc = 0;
                        accphase ^= 1;
                    }
                }
                tc_commit(&sm.aempty);  // theta tile reusable once the item's MMAs retire
            }
        }
    } else {
        // ===================== epilogue: softplus + row sums =====================
        const int ew = warp - 2;            // 0..7
        const int quarter = warp & 3;       // TMEM lanes this warp may access: 32*quarter .. +31
        const int colpart = ew >> 2;        // which kEpiCols columns of the accumulator
        const int row = quarter * 32 + lane;
        unsigned acc = 0, accphase = 0;
        for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
            const int mt = item % p.mtiles, ch = item / p.mtiles;
            const int t0 = ch * p.tiles_per_chunk, t1 = min(p.ntiles, t0 + p.tiles_per_chunk);
            double rowsum = 0.0;
            for (int t = t0; t < t1; ++t) {
                mbar_wait(&sm.tfull[acc], accphase);
                tc_fence_after();
                const long long nvalid = p.N - (long long)t * BN;  // columns of this tile that are real data
                // chunks of 32 columns; the TMEM load of chunk c+1 is in flight while chunk c is reduced.  (Carrying the
                // prefetch across the tile boundary was measured slower: 1326 vs 1098 us per half-step -- the wait loop
                // inside the unrolled chunk code costs the compiler its MUFU / FMA interleaving.)
                unsigned v[2][32];
                const unsigned tbase = tmem + ((unsigned)(quarter * 32) << 16) + acc * BN + colpart * kEpiCols;
                tmem_ld32(tbase, v[0]);
#pragma unroll
                for (int c = 0; c < kEpiCols / 32; ++c) {
                    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                    if (c + 1 < kEpiCols / 32) tmem_ld32(tbase + (c + 1) * 32, v[(c + 1) & 1]);
                    const int col0 = colpart * kEpiCols + c * 32;
                    const unsigned *vv = v[c & 1];
                    // softplus(s) = s/2 + |s|/2 + log1p(e^-|s|).  The s/2 term is linear in theta and lives in the exact
                    // FP64 d-dot of the finish kernel; the logits arrive in log2 units (theta was scaled by log2 e before
                    // the split), so the rest is  ln2 * ( |s'|/2 + lg2(1 + 2^-|s'|) ).  The 32 logarithms of a chunk are
                    // taken as ONE lg2 of the running product of (1 + t), t in (0,1] -- at most 2^16 per chain, no
                    // overflow: one MUFU (ex2) + one FFMA + one FADD per logit instead of two MUFU + ~7 FMA-pipe slots.
                    float pa = 1.0f, pb = 1.0f, sa = 0.0f, sb = 0.0f;
                    if (nvalid >= col0 + 32) {
#pragma unroll
                        for (int j = 0; j < 32; j += 2) {
                            const float s0 = __uint_as_float(vv[j]), s1 = __uint_as_float(vv[j + 1]);
                            const float t0 = ex2_neg_abs_col(s0, j), t1 = ex2_neg_abs_col(s1, j + 1);
                            pa = fmaf(pa, t0, pa);
                            pb = fmaf(pb, t1, pb);
                            sa += fabsf(s0);
                            sb += fabsf(s1);
                        }
                    } else {
#pragma unroll
                        for (int j = 0; j < 32; j += 2) {
                            const float s0 = __uint_as_float(vv[j]), s1 = __uint_as_float(vv[j + 1]);
                            if (col0 + j < nvalid) {
                                pa = fmaf(pa, ex2_neg_abs_col(s0, j), pa);
                                sa += fabsf(s0);
                            }
                            if (col0 + j + 1 < nvalid) {
                                pb = fmaf(pb, ex2_neg_abs_col(s1, j + 1), pb);
                                sb += fabsf(s1);
                            }
                        }
                    }
                    float lg;
                    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(pa * pb));
                    rowsum += (double)fmaf(0.5f, sa + sb, lg);  // log2 units; scaled by ln 2 at the store
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&sm.tempty[acc]);
                if (++acc == ACC) {
                    acc = 0;
                    accphase ^= 1;
                }
            }
            // combine the column parts of each row in fixed order, then one store per (chunk, row)
            asm volatile("bar.sync 1, %0;" ::"r"(kEpiWarps * 32));
            if (colpart > 0) sm.comb[colpart - 1][row] = rowsum;
            asm volatile("bar.sync 1, %0;" ::"r"(kEpiWarps * 32));
            if (colpart == 0) {
                const long long w = (long long)mt * BM + row;
#pragma unroll
                for (int k = 0; k < kEpiParts - 1; ++k) rowsum += sm.comb[k][row];
                if (w < p.W) p.part[(size_t)ch * p.W + w] = rowsum * 0.6931471805599453;
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// theta (FP64, d columns) -> three bf16 pieces hi + mid + lo, rows padded with zeros to wpad, columns to kp.
__global__ void split_theta_kernel(const double *__restrict__ TH, __nv_bfloat16 *__restrict__ out, long long W,
                                   long long wpad, int d, int kp, double scale) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= wpad * kp) return;
    const long long w = e / kp;
    const int c = (int)(e - w * kp);
    double r = (w < W && c < d) ? TH[w * d + c] * scale : 0.0;  // scale = log2 e: the GEMM delivers the logits in log2 units
#pragma unroll
    for (int pc = 0; pc < PIECES; ++pc) {
        const __nv_bfloat16 h = __double2bfloat16(r);
        out[(size_t)pc * wpad * kp + e] = h;
        r -= (double)__bfloat162float(h);
    }
}

// X (float32 [n][d]) -> bf16 [n][kp], columns zero-padded
__global__ void f32_to_bf16_kernel(const float *__restrict__ in, __nv_bfloat16 *__restrict__ out, long long n, int d,
                                   int kp) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n * kp) return;
    const long long r = e / kp;
    const int c = (int)(e - r * kp);
    out[e] = __float2bfloat16(c < d ? in[r * d + c] : 0.0f);
}

// logp = theta . (X^T (y - 1/2)) - sum_n (|s_n|/2 + log1p(e^-|s_n|)) - |theta|^2 / (2 sigma^2)
//      = theta . (X^T y) - sum_n softplus(s_n) - prior;   xty holds X^T (y - 1/2); chunks summed in fixed order.
__global__ void logistic_tc_finish_kernel(const double *__restrict__ TH, const double *__restrict__ part,
                                          const double *__restrict__ xty, double *__restrict__ out, long long W, int d,
                                          int nchunks, double inv2s2) {
    const long long w = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    double sp = 0.0;
    for (int k = 0; k < nchunks; ++k) sp += part[(size_t)k * W + w];
    double dot = 0.0, nn = 0.0;
    for (int c = 0; c < d; ++c) {
        const double t = TH[w * d + c];
        dot = fma(t, xty[c], dot);
        nn = fma(t, t, nn);
    }
    out[w] = dot - sp - nn * inv2s2;
}

// ======================================================================================
// K2  gaussian_tc_kernel: batched Mahalanobis form of the dense Gaussian plugin
//     (BASELINE.json configs[2], d <= 128):   y_w = A (x_w - mu),   out[w] = lognorm - 0.5 |y_w|^2
//
//   GEMM  [W x KP] . [KP x NP]^T  with KP = NP = 128 (d zero-padded), M tile = 128 walkers.
//   Both operands are FP64 on the host side and are split into three bf16 pieces each; the six
//   piece pairs whose product is above 2^-24 relative are accumulated in FP32 in TMEM, smallest
//   first:  (lo,hi) (hi,lo) (mid,mid) (mid,hi) (hi,mid) (hi,hi)   [C piece, A piece].
//   Stated tolerance vs the FP64 kernel: |logp_tc - logp_fp64| <= 1e-5 * (1 + |y|^2); the bound derived
//   from the arithmetic (tests/test_tc_error_model.py), P = |A| |x - mu|:
//   21 u sum_i |y_i| P_i + 16 u |y|^2 + (21 u)^2 |P|^2 / 2, u = 2^-24.
//
//   smem: A pieces 3 x 32 KB resident for the whole kernel + C pieces 3 x 32 KB per walker tile,
//   each piece = 2 k-halves of [128 rows x 128 B], SWIZZLE_128B K-major (TMA box 64 x 128).
//   warp 0 TMA, warp 1 MMA (48 x tcgen05.mma M=128 N=128 K=16 per tile), warps 2-5 epilogue
//   (tcgen05.ld, sum of squares of the first d columns), accumulators double-buffered in TMEM.
constexpr int GK = 128, GN = 128, GPIECE_BYTES = 2 * BM * 128;  // 32 KB
constexpr int kGaussThreads = 32 * (2 + 4);

struct __align__(1024) GaussSmem {
    unsigned char a[PIECES][GPIECE_BYTES];  // matrix A pieces [k-half][128 n-rows][128 B]
    unsigned char c[PIECES][GPIECE_BYTES];  // centred walker pieces [k-half][128 m-rows][128 B]
    unsigned long long afull, cfull, cempty, tfull[ACC], tempty[ACC];
    unsigned tmem_base;
};


struct GaussParams {
    long long W;      // points
    int mtiles;       // ceil(W / 128)
    long long wpad;   // mtiles * 128: rows per piece in the C piece buffer
    int d;
    double lognorm;
    double *out;      // [W]
};

__global__ void __launch_bounds__(kGaussThreads, 1)
gaussian_tc_kernel(const __grid_constant__ CUtensorMap mapC, const __grid_constant__ CUtensorMap mapA,
                   const GaussParams p) {
    extern __shared__ unsigned char smem_raw[];
    GaussSmem &sm = *reinterpret_cast<GaussSmem *>(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        mbar_init(&sm.afull, 1);
        mbar_init(&sm.cfull, 1);
        mbar_init(&sm.cempty, 1);
        for (int a = 0; a < ACC; ++a) {
            mbar_init(&sm.tfull[a], 1);
            mbar_init(&sm.tempty[a], 4);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(&sm.tmem_base))
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const unsigned tmem = sm.tmem_base;

    if (warp == 0) {
        if (lane == 0) {
            mbar_expect_tx(&sm.afull, PIECES * GPIECE_BYTES);  // the matrix: once per CTA
            for (int pc = 0; pc < PIECES; ++pc)
                for (int kh = 0; kh < 2; ++kh)
                    tma_load_2d(sm.a[pc] + kh * (GPIECE_BYTES / 2), &mapA, kh * 64, pc * GN, &sm.afull);
            unsigned cphase = 0;
            for (int mt = blockIdx.x; mt < p.mtiles; mt += gridDim.x) {
                mbar_wait(&sm.cempty, cphase ^ 1);
                mbar_expect_tx(&sm.cfull, PIECES * GPIECE_BYTES);
                for (int pc = 0; pc < PIECES; ++pc)
                    for (int kh = 0; kh < 2; ++kh)
                        tma_load_2d(sm.c[pc] + kh * (GPIECE_BYTES / 2), &mapC, kh * 64,
                                    (int)(pc * p.wpad + (long long)mt * BM), &sm.cfull);
                cphase ^= 1;
            }
        }
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr unsigned idesc = idesc_bf16_f32(BM, GN);
            // (C piece, A piece): 0 = hi, 1 = mid, 2 = lo; smallest products first
            const int pc_c[6] = {2, 0, 1, 1, 0, 0};
            const int pc_a[6] = {0, 2, 1, 0, 1, 0};
            unsigned cphase = 0, acc = 0, accphase = 0;
            mbar_wait(&sm.afull, 0);
            for (int mt = blockIdx.x; mt < p.mtiles; mt += gridDim.x) {
                mbar_wait(&sm.tempty[acc], accphase ^ 1);
                mbar_wait(&sm.cfull, cphase);
                cphase ^= 1;
                tc_fence_after();
                const unsigned d = tmem + acc * GN;
#pragma unroll
                for (int pr = 0; pr < 6; ++pr) {
                    const unsigned cb = smem_u32(sm.c[pc_c[pr]]), ab = smem_u32(sm.a[pc_a[pr]]);
#pragma unroll
                    for (int k = 0; k < GK / 16; ++k) {
                        const unsigned off = (k >> 2) * (GPIECE_BYTES / 2) + (k & 3) * 32;  // k-half, then 32 B per k-step
                        tc_mma(d, smem_desc_sw128(cb + off), smem_desc_sw128(ab + off), idesc, (pr | k) ? 1u : 0u);
                    }
                }
                tc_commit(&sm.cempty);
                tc_commit(&sm.tfull[acc]);
                if (++acc == ACC) {
                    acc = 0;
                    accphase ^= 1;
                }
            }
        }
    } else {
        const int quarter = warp & 3;
        const int row = quarter * 32 + lane;
        unsigned acc = 0, accphase = 0;
        for (int mt = blockIdx.x; mt < p.mtiles; mt += gridDim.x) {
            mbar_wait(&sm.tfull[acc], accphase);
            tc_fence_after();
            double ss = 0.0;
#pragma unroll 1
            for (int cb = 0; cb < GN; cb += 32) {
                if (cb >= p.d) break;
                unsigned v[32];
                const unsigned taddr = tmem + ((unsigned)(quarter * 32) << 16) + acc * GN + cb;
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                    "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
                    "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                    : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
                      "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
                      "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]),
                      "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]),
                      "=r"(v[30]), "=r"(v[31])
                    : "r"(taddr)
                    : "memory");
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                float part = 0.0f;  // padded columns are exact zeros (zero rows of the matrix pieces)
#pragma unroll
                for (int j = 0; j < 32; ++j) {
                    const float y = __uint_as_float(v[j]);
                    part = fmaf(y, y, part);
                }
                ss += (double)part;
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&sm.tempty[acc]);
            if (++acc == ACC) {
                acc = 0;
                accphase ^= 1;
            }
            const long long w = (long long)mt * BM + row;
            if (w < p.W) p.out[w] = p.lognorm - 0.5 * ss;
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem) : "memory");
}

// rows of (X - mu) (FP64, d columns) -> three bf16 pieces, rows padded to wpad, columns to 128.
// mu == nullptr: no centring (used for the matrix A itself, rows = d).
__global__ void split_rows128_kernel(const double *__restrict__ X, const double *__restrict__ mu,
                                     __nv_bfloat16 *__restrict__ out, long long rows, long long rpad, int d) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= rpad * GK) return;
    const long long r = e / GK;
    const int c = (int)(e % GK);
    double v = (r < rows && c < d) ? X[r * d + c] - (mu ? mu[c] : 0.0) : 0.0;
    if (mu) {  // points: the split every proposal kernel uses (kmc_device.cuh), so all paths agree bit for bit
        unsigned pk[3];
        split3_pair(v, 0.0, pk);
#pragma unroll
        for (int pc = 0; pc < PIECES; ++pc) out[(size_t)pc * rpad * GK + e] = __ushort_as_bfloat16((unsigned short)pk[pc]);
        return;
    }
#pragma unroll
    for (int pc = 0; pc < PIECES; ++pc) {  // the matrix (once per density): round-to-nearest pieces of the FP64 value
        const __nv_bfloat16 h = __double2bfloat16(v);
        out[(size_t)pc * rpad * GK + e] = h;
        v -= (double)__bfloat162float(h);
    }
}

}  // namespace tc
}  // namespace kmc
