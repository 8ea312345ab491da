// kmc_push.cuh -- the sharded ensemble (one ensemble over G GPUs, SURVEY.md section 8e) as ONE persistent kernel
// per GPU with OWNER-COMPUTES PUSHES of the partner rows over NVLink.
//
// Replaces, across GPUs, the reference's shared-memory read of the passive half inside the threaded sweep
// (src/samplers.jl:246-273, partner read at :255): rank r updates positions [r*S, (r+1)*S) of each half and holds
// ONLY those rows (x[2][S][D]); the partner row of an active walker lives on rank (partner position / S).
//
// The draws are counter-based (Philox keyed by the global walker index, kmc_device.cuh), so the OWNER of a passive
// shard can enumerate, without any index round trip, which of its rows every other rank's active walkers will ask for
// (SURVEY.md section 7.2(9)(i)).  Per half-step every rank runs two kinds of tasks, handed out to its CTAs from two
// atomic counters (pushes in chunk order, update groups in chunk order):
//
//   push(c, dest)   enumerate the partner draws of chunk c (`chunk` <= 1024 consecutive active walkers, `rounds` rounds
//                   of 256) of rank `dest`; the hits in my passive shard are gathered (one bulk copy per row), PACKED
//                   in walker order behind a 16-byte header (the message row at which each round starts) in shared
//                   memory and sent as ONE bulk store (cp.async.bulk shared -> peer global, 16 + rows*8D bytes, 10-30 KB)
//                   into dest's receive ring slot (half-step parity, source = me, chunk c); when the store has
//                   completed, the "chunk ready" flag (source, c) in dest's memory is set to h+1 (release, system scope).
//   update(c, g)    the stretch-move step of round g (256 walkers) of my chunk c: the walker-step's own draws give every
//                   walker's owner and its rank among the round's walkers with that owner; header[g] + rank is its row
//                   in the owner's message.  Waits for the G-1 chunk flags, then one group of the bulk kernel's loop
//                   (kmc_kernels.cuh, emcee_bulk_kernel): own rows in one bulk load, partner rows gathered from the
//                   local receive ring (remote owner), the local passive shard (own rows) or, for the rare row past
//                   the ring slot's capacity, straight from the owner's memory; accept / chain store; ACCEPTED rows are
//                   written back from registers (the update side is bound by its DRAM traffic).
//
// Two hand-outs (PushParams::lag): ORDERED (the default) -- one counter, the pushes of chunk c, then the update groups
// of chunk c - lag; the next task id is ONE atomic issued at the start of the current task, so handing out costs nothing;
// a flag reaches its consumer ~25 us after its push, `lag` chunks of other work cover that.  ADAPTIVE (lag = 0) -- two
// counters; a CTA takes the next update group if that group's flags are seen set, else the next push, and only when no
// push is left an update it has to wait for (no tuning, but three dependent L2 round trips per task: measured 7 % slower
// at 8 GPUs).  There is no cross-GPU barrier at all -- a consumer starts as soon as ITS chunk's rows have landed -- and one local
// grid barrier per half-step (random rows of the whole shard are read by the next half-step's pushes).
//
// Nothing a push does is waited for where it is issued (thread 0 is the CTA's "sender"):
//   * the row gathers of push t land while the CTA works on its NEXT task; the sender issues the bulk store of push t
//     at that task's service point (after its enumeration);
//   * the store's completion is not waited for either: at a later task, once `cp.async.bulk.wait_group kPushAge` says
//     the store is complete, the sender posts a NOTE (release at GPU scope) in local memory;
//   * the system-scope release that the remote flag needs is not paid by the workers at all: with tens of megabytes
//     queued on the link a `fence.acq_rel.sys` takes ~8 us (measured: a quarter of the kernel when every CTA fenced for
//     its own flags).  ONE CTA per GPU, the publisher, takes no tasks: it sweeps the notes (acquire, GPU scope), and per
//     sweep pays one system-scope fence for all the flags it then sets in the peers' memory.  The chain worker's stores
//     -> release.gpu note -> publisher's acquire.gpu -> fence.sys -> flag -> consumer's acquire.sys orders the rows
//     before the consumer's reads.
//
// Why there is no deadlock: pushes wait for nothing (only for the link to drain their previous message); all CTAs are
// co-resident (cooperative launch); a CTA never blocks while it holds an un-noted completed store; ORDERED: give
// push(c, *) level c and update(c, *) level c + lag + 1/2 -- tasks are taken in level order and a task only ever waits
// for strictly lower levels on other GPUs; ADAPTIVE: a CTA blocks on a flag only when its rank has no push left to hand
// out, so every rank's pushes complete whatever its updates do.  Why two ring
// parities suffice: rank q can only push for half-step h+2 after it finished update h+1, which needs every rank's
// pushes of h+1, which a rank sends only after its update h.
//
// Exactness: every walker-step is the same arithmetic on the same draws as the single-GPU kernels, so a sharded run is
// bit-identical to the single-GPU run of the same ensemble (tests/test_gpu_push.py).
#pragma once
#ifdef KMC_PUSH_PROF
#include <cstdio>
#endif
#include "kmc_kernels.cuh"

namespace kmc {

#ifndef KMC_PUSH_THREADS
#define KMC_PUSH_THREADS 256
#endif
#ifndef KMC_PUSH_CTAS
#define KMC_PUSH_CTAS (KMC_PUSH_THREADS == 32 ? 20 : 3)
#endif
constexpr int kPushThreads = KMC_PUSH_THREADS;
constexpr int kPushWarps = kPushThreads / 32;
// T = 256 (the build default): a task is a CTA of 8 warps (chunks of up to 4 rounds, barriers between its phases).
// T = 32 (-DKMC_PUSH_THREADS=32): a task is ONE WARP (chunks of up to 8 rounds), ~20 independent task streams per SM
// instead of 3.  Measured SLOWER (2 B200s, 2^24 x 10-D: 0.59-0.63 vs 0.47 ms per half-step, profiles/r2_summary.md): the
// update groups run at the memory system's pace either way (~17 cycles per walker-step and SM, like the single-GPU bulk
// kernel), so more streams only add per-task overhead.
constexpr int kPushMaxRounds = kPushThreads == 32 ? 8 : 1024 / kPushThreads;  // rounds of T walkers per chunk
constexpr int kPushMaxChunk = kPushMaxRounds * kPushThreads;
constexpr int kPushMaxRanks = 8;
constexpr int kPushSlots = kPushMaxRounds * kPushWarps;  // (round, warp) slots of a chunk <= one warp's lanes (prefix by shuffles)
constexpr int kPushPublishers = kPushThreads == 32 ? 8 : 1;  // CTAs that publish flags instead of taking tasks
constexpr int kPushFifo = 8;    // flags whose store is issued but which are not published yet
#ifndef KMC_PUSH_BATCH
#define KMC_PUSH_BATCH 1
#endif
constexpr unsigned kPushBatch = KMC_PUSH_BATCH;  // flags published per system-scope fence
#ifndef KMC_PUSH_AGE
#define KMC_PUSH_AGE 3
#endif
constexpr unsigned kPushAge = KMC_PUSH_AGE;      // a flag is published once its store is this many commits old
static_assert(kPushSlots <= 32, "the slot prefix is one warp's shuffle scan");

struct PushParams {
    double *recv;               // local receive ring [2 parities][G sources][nchunks][cap][D]
    unsigned long long *flags;  // local chunk flags [G sources][nchunks]: h+1 once the rows for half-step h have landed
    double *peer_recv[kPushMaxRanks];
    unsigned long long *peer_flags[kPushMaxRanks];
    const double *peer_x[kPushMaxRanks];  // x[2][S][D] of every rank (capacity-overflow fallback reads)
    unsigned long long *task_ctr;          // [2 half-step parities][push, update] task counters (zeroed by the host)
    unsigned *notes;                       // [nchunks * (G-1)] per push task: epoch of its completed store (publisher's inbox)
    unsigned S;        // shard size: positions of each half per rank
    unsigned G, rank;  // ranks, my rank
    unsigned chunk;    // walkers per chunk (<= 1024)
    unsigned rounds;   // ceil(chunk / kPushThreads)
    unsigned nchunks;  // ceil(S / chunk)
    unsigned cap;      // rows per ring slot (<= kPushMaxCap)
    unsigned lag;      // > 0: ORDERED hand-out from one counter, update(c, *) follows push(c + lag, *); 0: ADAPTIVE
    unsigned batch;    // notes posted per GPU-scope fence (>= 1)
    unsigned age;      // a store is taken for complete once it is this many commits old (1..3)
};
constexpr int kPushMaxCap = kPushThreads == 32 ? 64 : 384;  // rows: the message buffer is header + cap * 8D bytes of shared memory
constexpr int kPushHeader = 4 * kPushMaxRounds;  // bytes: the message row at which each round of the chunk starts (u32 each)
static_assert(kPushHeader % 16 == 0, "bulk copies move multiples of 16 bytes");

// The sender's state: touched by thread 0 only, kept in shared memory so that it costs the other 255 threads no registers.
struct PushSender {
    double *dst;                     // the push whose gathers are in flight and whose store is not issued yet
    unsigned task;                   // its push task id (names the note and the flag)
    unsigned pending, bytes;
    unsigned gphase;                 // phase of gbar
    unsigned ncommit;                // tasks this CTA has started (the sender's clock)
    unsigned msg_commit, pad0;       // the clock when the newest message store was issued
    unsigned fhead, ftail;           // fifo[fhead..ftail): flags of issued stores that are not published yet
};

// Dynamic shared memory: own rows [T][D] | partner rows [T][D] | message (header + cap rows) | sender | barriers |
// flag queue | hit counts and prefixes.
constexpr size_t push_smem_bytes(int D, unsigned cap) {
    return (size_t)2 * kPushThreads * D * 8 + kPushHeader + (size_t)cap * D * 8 + sizeof(PushSender) +
           sizeof(unsigned long long) * (4 + kPushFifo) +
           sizeof(unsigned) * (2 * kPushSlots * kPushMaxRanks + kPushMaxRanks + kPushFifo);
}

// The partner draw alone (src/samplers.jl:250): the owner side of a push needs nothing else of the walker-step.
__device__ __forceinline__ unsigned partner_pos(const RunParams &p, long long h, unsigned i) {
    const unsigned long long t = (unsigned long long)(h >> 1);
    const unsigned batch = (unsigned)(h & 1);
    const unsigned walker = p.id_base[batch] + i;
    const Philox4 r = philox4x32_10(walker, (unsigned)t, (unsigned)(t >> 32), batch, p.keys);
    unsigned hi, lo;
    mul_wide(r.r0, p.nhalf, hi, lo);
    if (lo < p.lemire_t) hi = lemire_retry(p.keys, walker, (unsigned)t, (unsigned)(t >> 32), batch, p.nhalf, p.lemire_t);
    return hi;  // position inside the passive half
}

__device__ __forceinline__ unsigned long long flag_peek(const unsigned long long *flag) {
    unsigned long long cur;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(cur) : "l"(flag) : "memory");
    return cur;
}

// no ordering: only to CHOOSE a task (the update itself re-checks with acquire semantics before it reads the ring)
__device__ __forceinline__ unsigned long long flag_peek_relaxed(const unsigned long long *flag) {
    unsigned long long cur;
    asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(cur) : "l"(flag) : "memory");
    return cur;
}

__device__ __forceinline__ void flag_wait(const unsigned long long *flag, unsigned long long v) {
    long long t0 = 0;
    unsigned spins = 0;
    while (flag_peek(flag) < v) {
        if ((++spins & 0x3FFu) == 0) {  // watchdog (~10 s): a missing peer must not hang the GPU
            if (t0 == 0) t0 = clock64();
            else if (clock64() - t0 > 20000000000LL) __trap();
        }
    }
}

template <template <int> class Dn, int D>
__global__ void __launch_bounds__(kPushThreads, KMC_PUSH_CTAS) emcee_push_kernel(const RunParams p, const PushParams q,
                                                                                  const Dn<D> dn) {
    static_assert(D % 2 == 0, "rows must be multiples of 16 bytes");
    extern __shared__ __align__(128) unsigned char push_smem[];
    constexpr unsigned T = kPushThreads, ROWB = D * 8;
    double *ownb = reinterpret_cast<double *>(push_smem);  // [T][D] own rows of an update group
    double *xpart = ownb + T * D;                          // [T][D] partner rows of an update group
    unsigned char *msg = reinterpret_cast<unsigned char *>(xpart + T * D);  // header + packed rows of a push
    PushSender *snd = reinterpret_cast<PushSender *>(msg + kPushHeader + (size_t)q.cap * ROWB);
    unsigned long long *ldbar = reinterpret_cast<unsigned long long *>(snd + 1);  // loads of an update group
    unsigned long long *gbar = ldbar + 1;                 // row gathers of the push that owns the message buffer
    unsigned long long *next_slot = ldbar + 3;            // broadcast of the next task id
    unsigned long long *fifo = ldbar + 4;                 // [kPushFifo] sender's queue: push task ids of issued stores
    unsigned *cnt = reinterpret_cast<unsigned *>(ldbar + 4 + kPushFifo);  // [kPushSlots][kPushMaxRanks] hits per slot, owner
    unsigned *pre = cnt + kPushSlots * kPushMaxRanks;     // exclusive prefix of cnt over the slots, per owner
    unsigned *tot = pre + kPushSlots * kPushMaxRanks;     // [kPushMaxRanks] totals
    unsigned *fidx = tot + kPushMaxRanks;                 // [kPushFifo] (spare)

    const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned S = q.S, me = q.rank, G = q.G, R = q.rounds;
    const unsigned NP = q.nchunks * (G - 1);  // push tasks per half-step: (chunk, destination)
    const unsigned NU = q.nchunks * R;        // update tasks per half-step: (chunk, round of T walkers)
    const bool ordered = q.lag > 0;           // one counter, fixed order: pushes of chunk c, then the update groups of chunk c - lag
    const unsigned per_c = G - 1 + R;
    const unsigned long long NT_dense = (unsigned long long)q.nchunks * per_c;  // every push and every update group once
    // the last kPushPublishers CTAs publish flags and take no tasks (each its slice of the push tasks' notes)
    const bool use_pub = G > 1 && gridDim.x > (unsigned)kPushPublishers;
    const bool is_pub = use_pub && blockIdx.x >= gridDim.x - kPushPublishers;
    if (tid == 0) {
        kbar_init(ldbar, 1);
        kbar_init(gbar, 1);
        snd->pending = snd->gphase = snd->ncommit = snd->msg_commit = snd->fhead = snd->ftail = 0u;
    }
    __syncthreads();
    unsigned ldphase = 0;

    // ------------------------------------------------------------------ the sender (thread 0)
    // The only bulk async-groups of this thread are the message stores, one per push, in order.
    // snd->pending: a push whose gathers are in flight into `msg` and whose store is not issued yet.
    // fifo[fhead..ftail): push task ids of issued stores whose notes are not posted yet; snd->ncommit counts the CTA's
    // tasks (a clock), snd->msg_commit is its value when the newest store was issued.
    // issue the bulk store of the pending push (its gathers have landed by now: they were issued a task ago)
    auto service = [&]() {
        if (!snd->pending) return;
        kbar_wait(gbar, snd->gphase & 1u);
        snd->gphase ^= 1u;
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the header (generic proxy) -> bulk store
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(snd->dst),
                     "r"((unsigned)__cvta_generic_to_shared(msg)), "r"(snd->bytes)
                     : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        snd->msg_commit = snd->ncommit;
        const unsigned ft = snd->ftail;
        fifo[ft % kPushFifo] = snd->task;
        snd->ftail = ft + 1;
        snd->pending = 0;
    };
    // post the notes (or, without a publisher, set the flags) of the stores that are complete.  A message drains into
    // NVLink at the link's pace and completion can only be WAITED for, so by default only what can be had without
    // blocking is taken: everything but the newest store (wait_group 1), or everything once the newest store is `age`
    // tasks old (wait_group 0 then returns at once, barring a congested link).
    auto publish = [&](bool all, unsigned long long ready) {
        unsigned fhead = snd->fhead;
        const unsigned ftail = snd->ftail;
        if (fhead == ftail) return;
        unsigned upto;
        if (all || snd->ncommit - snd->msg_commit >= q.age || ftail - fhead >= kPushFifo - 1) {
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
            upto = ftail;
        } else {
            if (ftail - fhead < 1 + q.batch) return;
            asm volatile("cp.async.bulk.wait_group 1;" ::: "memory");
            upto = ftail - 1;
        }
        // wait_group made the completed stores' writes visible to this thread (completion of a bulk async-group implies
        // the generic-async proxy fence); the release fence then orders them before the note / flag for every observer.
        // No fence.proxy.async here: it would also wait for the YOUNGER message that is still draining into the link
        // (measured: ~20k cycles per publish, a quarter of the kernel).
        if (use_pub) {  // hand the completed stores to the publisher CTA: release at GPU scope is all a worker pays
            asm volatile("fence.acq_rel.gpu;" ::: "memory");
            for (; fhead != upto; ++fhead)
                asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(q.notes + (unsigned)fifo[fhead % kPushFifo]),
                             "r"((unsigned)ready)
                             : "memory");
        } else {  // a grid too small for a publisher: set the remote flags directly
            asm volatile("fence.acq_rel.sys;" ::: "memory");
            for (; fhead != upto; ++fhead) {
                const unsigned tp = (unsigned)fifo[fhead % kPushFifo], pcn = tp / (G - 1);
                unsigned long long *fl = q.peer_flags[(me + 1 + (tp - pcn * (G - 1))) % G] + (size_t)me * q.nchunks + pcn;
                asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(fl), "l"(ready) : "memory");
            }
        }
        snd->fhead = fhead;
    };
    // before the message buffer is overwritten: the previous message has left shared memory
    auto msg_free = [&]() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); };

    // The next task of this CTA, chosen by warp 0 (all 32 lanes call it; the result is valid in lane 0):
    // kind << 32 | id, kind 0 = push, 1 = update, 2 = nothing left.  An update group whose chunk's flags are all set
    // is preferred (lanes peek the G-1 flags in parallel); else a push; else an update that will have to wait.
    auto pick = [&](unsigned par, unsigned long long ready) -> unsigned long long {
        unsigned long long *pc = q.task_ctr + 2 * par, *uc = pc + 1;
        // lane 30 reads the push counter, lane 31 the update counter (one round trip for both)
        unsigned long long cv = 0;
        if (lane >= 30) cv = *reinterpret_cast<volatile unsigned long long *>(lane == 31 ? uc : pc);
        const unsigned long long up = __shfl_sync(0xffffffffu, cv, 31), pp = __shfl_sync(0xffffffffu, cv, 30);
        bool late = false;
        if (up < NU && lane < G && lane != me)
            late = flag_peek_relaxed(q.flags + (size_t)lane * q.nchunks + (unsigned)up / R) < ready;
        const bool ok = up < NU && !__any_sync(0xffffffffu, late);
        unsigned long long res = 2ULL << 32;
        if (lane == 0) {
            bool done = false;
            if (ok) {  // claim exactly the group whose flags were seen set (compare-and-swap: a later group might not be ready,
                       // and a CTA must never block on a flag while its rank still has pushes to hand out)
                if (atomicCAS(uc, up, up + 1ULL) == up) {
                    res = (1ULL << 32) | up;
                    done = true;
                }
            }
            if (!done && pp < NP) {
                const unsigned long long t = atomicAdd(pc, 1ULL);
                if (t < NP) {
                    res = t;
                    done = true;
                }
            }
            if (!done) {
                const unsigned long long t = atomicAdd(uc, 1ULL);
                if (t < NU) res = (1ULL << 32) | t;
            }
        }
        return res;
    };

    // ORDERED hand-out: ONE atomic per task.  The sequence "pushes of chunk index c, then the update groups of chunk c - lag"
    // has three regions -- c < lag: pushes only; lag <= c < nchunks: pushes and updates; nchunks <= c < nchunks + lag:
    // updates only -- numbered densely, so no sequence number is wasted on a slot that holds no task (a CTA that had to
    // skip the 7 empty push slots between two updates of the tail paid 7 dependent atomics for one task).
    // Returns kind << 32 | id like pick().
    auto take = [&](unsigned par, unsigned long long ready) -> unsigned long long {
        if (!ordered) return pick(par, ready);
        unsigned long long res = 2ULL << 32;
        if (lane == 0) {
            const unsigned long long v = atomicAdd(q.task_ctr + 2 * par, 1ULL);
            const unsigned long long lenA = (unsigned long long)q.lag * (G - 1);
            const unsigned long long lenB = (unsigned long long)(q.nchunks - q.lag) * per_c;
            if (v < lenA) {
                res = v;  // push(c, slot) with id = c * (G-1) + slot = v
            } else if (v < lenA + lenB) {
                const unsigned w = (unsigned)(v - lenA), c = q.lag + w / per_c, slot = w % per_c;
                if (slot + 1 < G) res = (unsigned long long)(c * (G - 1) + slot);
                else res = (1ULL << 32) | (unsigned long long)((c - q.lag) * R + (slot - (G - 1)));
            } else if (v < NT_dense) {
                res = (1ULL << 32) | (unsigned long long)((q.nchunks - q.lag) * R + (unsigned)(v - lenA - lenB));
            }
        }
        return res;
    };

#ifdef KMC_PUSH_PROF  // thread 0's cycles per phase (experiment builds only)
    long long pt[10] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, pc0 = clock64();
    unsigned npush = 0, nupd = 0;
#define PUSH_TICK(i) do { const long long c_ = clock64(); pt[i] += c_ - pc0; pc0 = c_; } while (0)
#else
#define PUSH_TICK(i) do { } while (0)
#endif
    ThinClock<> clk{p.n0, p.phase0, p.sidx0};
    unsigned long long target = p.bar_base;
    unsigned long long next = 0;

    for (long long h = p.h0; h < p.h1; ++h) {
        const unsigned batch = (unsigned)(h & 1);
        const bool store = clk.store();
        const bool reset = (batch == 1) && clk.burnin_end();
        const size_t act = batch ? (size_t)S : 0;         // first local row of the active half
        const size_t pas = batch ? 0 : (size_t)S;         // first local row of the passive half
        const unsigned par = (unsigned)(h & 1);           // ring parity
        const unsigned long long ready = (unsigned long long)h + 1;
        const size_t slot_bytes = kPushHeader + (size_t)q.cap * ROWB;  // one ring slot: header + cap rows
        if (is_pub) {
            // ---------------------------------------------------------------- the publisher: notes -> remote flags
            // note[tp] == epoch: the store of push task tp has completed (written by its sender with release.gpu).
            // Every thread sweeps its share with relaxed loads, pays ONE system-scope fence for what it found, sets the
            // flags in the peers' memory and marks the notes done, until all NP flags of the half-step are out.
            unsigned *cntp = reinterpret_cast<unsigned *>(next_slot);
            if (tid == 0) *cntp = 0u;
            __syncthreads();
            const unsigned pubi = blockIdx.x - (gridDim.x - kPushPublishers);             // this publisher's slice of the notes
            const unsigned plo = (unsigned)((unsigned long long)NP * pubi / kPushPublishers);
            const unsigned phi = (unsigned)((unsigned long long)NP * (pubi + 1) / kPushPublishers);
            const unsigned want = (unsigned)ready, done_mark = want | 0x80000000u;
            long long t0 = 0;
            unsigned spins = 0;
            for (;;) {
                unsigned found = 0;
                for (unsigned seg = plo; seg < phi; seg += 32 * T) {  // segments of 32 notes per thread
                    unsigned mask = 0;
#pragma unroll 4
                    for (unsigned k = 0; k < 32; ++k) {
                        const unsigned tp = seg + k * T + tid;
                        if (tp < phi) {
                            unsigned v;  // relaxed: the fence below is the acquire for everything the sweep saw
                            asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(q.notes + tp) : "memory");
                            if (v == want) mask |= 1u << k;
                        }
                    }
                    if (mask == 0) continue;
                    // acquire for the notes seen (their senders released at GPU scope) and release for the flags below
                    asm volatile("fence.acq_rel.sys;" ::: "memory");
                    found += __popc(mask);
                    for (; mask; mask &= mask - 1) {
                        const unsigned tp = seg + (__ffs(mask) - 1) * T + tid, pcn = tp / (G - 1);
                        unsigned long long *fl = q.peer_flags[(me + 1 + (tp - pcn * (G - 1))) % G] + (size_t)me * q.nchunks + pcn;
                        asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(fl), "l"(ready) : "memory");
                        asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(q.notes + tp), "r"(done_mark) : "memory");
                    }
                }
                if (found) atomicAdd(cntp, found);
                __syncthreads();
                const unsigned total = *reinterpret_cast<volatile unsigned *>(cntp);
                __syncthreads();
                if (total >= phi - plo) break;
                if ((++spins & 0x3FFu) == 0) {  // watchdog: a lost sender must not hang the GPU
                    if (t0 == 0) t0 = clock64();
                    else if (clock64() - t0 > 40000000000LL) __trap();
                }
            }
            next = 2ULL << 32;
        } else {
            if (warp == 0) {
                if (tid == 0 && blockIdx.x == 0) {  // the other parity's counters are idle during this half-step: reset them
                    q.task_ctr[2 * (par ^ 1)] = 0ULL;
                    q.task_ctr[2 * (par ^ 1) + 1] = 0ULL;
                }
                const unsigned long long first = take(par, ready);
                if (lane == 0) *next_slot = first;
            }
            __syncthreads();
            next = *next_slot;
        }

        while ((next >> 32) < 2) {
            const unsigned kind = (unsigned)(next >> 32), t = (unsigned)next;
            unsigned long long nxt = 0;
            if (ordered && warp == 0) nxt = take(par, ready);  // one atomic, no dependence on flags: issued first, used last
            PUSH_TICK(9);
            if (tid == 0) {
                snd->ncommit += 1;
                publish(false, ready);  // notes for the stores that are complete by now
            }
            PUSH_TICK(3);
            if (kind == 0) {
                // ------------------------------------------------------------ push(c, dest)
                const unsigned c = t / (G - 1), slot = t - c * (G - 1);
                {
                    PUSH_TICK(9);
                    const unsigned dest = (me + 1 + slot) % G;
                    const unsigned i0 = dest * S + c * q.chunk;  // first active walker (position in its half) of the chunk
                    const unsigned lim = min(q.chunk, S - c * q.chunk);
                    unsigned lrow[kPushMaxRounds], rk[kPushMaxRounds];
#pragma unroll
                    for (int g = 0; g < kPushMaxRounds; ++g) {
                        lrow[g] = 0xFFFFFFFFu;
                        rk[g] = 0;
                        unsigned nh = 0;
                        if (g < (int)R) {
                            const unsigned off = g * T + tid;
                            bool hit = false;
                            if (off < lim) {
                                const unsigned pl = partner_pos(p, h, i0 + off) - me * S;  // < S iff the partner is mine
                                hit = pl < S;
                                if (hit) lrow[g] = pl;
                            }
                            const unsigned bl = __ballot_sync(0xffffffffu, hit);
                            rk[g] = __popc(bl & ((1u << lane) - 1u));
                            nh = __popc(bl);
                        }
                        if (lane == 0) cnt[g * kPushWarps + warp] = nh;
                    }
                    __syncthreads();
                    PUSH_TICK(1);
                    if (warp == 0) {
                        const unsigned v = lane < (unsigned)kPushSlots ? cnt[lane] : 0u;
                        unsigned incl = v;
#pragma unroll
                        for (int o = 1; o < kPushSlots; o <<= 1) {
                            const unsigned u = __shfl_up_sync(0xffffffffu, incl, o);
                            if ((int)lane >= o) incl += u;
                        }
                        if (lane < (unsigned)kPushSlots) pre[lane] = incl - v;
                        if (lane == kPushSlots - 1) tot[0] = incl;
                        if (lane == 0) {  // the sender: the previous push goes out, then the message buffer is free again
                            service();
                            msg_free();
                        }
                        __syncwarp();
                        if (lane < (unsigned)kPushSlots && (lane % kPushWarps) == 0)  // header: the row at which each round starts
                            reinterpret_cast<unsigned *>(msg)[lane / kPushWarps] = incl - v;
                    }
                    __syncthreads();
                    PUSH_TICK(0);
                    if (warp == 0) {  // the next task: its counter reads, flag peeks and atomic run while the other warps
                        if (!ordered) nxt = pick(par, ready);  // issue their row gathers
                        PUSH_TICK(4);
                    }
                    const unsigned nsend = min(tot[0], q.cap);
                    if (tid == 0) kbar_expect_tx(gbar, nsend * ROWB);
#pragma unroll
                    for (int g = 0; g < kPushMaxRounds; ++g) {
                        if (lrow[g] != 0xFFFFFFFFu) {
                            const unsigned pi = pre[g * kPushWarps + warp] + rk[g];
                            if (pi < q.cap)
                                bulk_row_g2s(msg + kPushHeader + (size_t)pi * ROWB, p.x + (pas + lrow[g]) * D, ROWB, gbar);
                        }
                    }
                    if (tid == 0) {  // sent at the next service point
                        snd->pending = 1;
                        snd->bytes = kPushHeader + nsend * ROWB;
                        snd->dst = reinterpret_cast<double *>(reinterpret_cast<unsigned char *>(q.peer_recv[dest]) +
                                                              (((size_t)par * G + me) * q.nchunks + c) * slot_bytes);
                        snd->task = t;
                    }
                    PUSH_TICK(2);
#ifdef KMC_PUSH_PROF
                    ++npush;
#endif
                }
            } else if ((t % R) * T < min(q.chunk, S - (t / R) * q.chunk)) {
                // ------------------------------------------------------------ update(cu, g): one group of T walkers
                PUSH_TICK(9);
                const unsigned cu = t / R, g = t - cu * R;
                const unsigned l0 = cu * q.chunk + g * T;     // first local position of the group
                const unsigned rows = min(T, min(q.chunk, S - cu * q.chunk) - g * T);
                const unsigned l = l0 + tid;
                const bool live = tid < rows;
                // the walker-step's draws (:250, :252, :260 uniform); the partner's owner and the walker's rank among the
                // round's walkers with the same owner = its row in that owner's message, after header[g]
                DrawRec dr;
                dr.j = 0;
                dr.z = 0.0;
                dr.q = 0.f;
                unsigned owner = 0xFFu, prow = 0, rkw = 0;
                if (live) {
                    unsigned j;
                    double z, u;
                    step_draws<false>(p, h, me * S + l, j, z, u);
                    dr.z = z;
                    dr.q = filter_q<false>(p, z, u);
                    const unsigned pl = j >= p.nhalf ? j - p.nhalf : j;  // position inside the passive half
                    owner = pl / S;
                    prow = pl - owner * S;
                }
                for (unsigned o = 0; o < G; ++o) {
                    const unsigned bl = __ballot_sync(0xffffffffu, owner == o);
                    if (owner == o) rkw = __popc(bl & ((1u << lane) - 1u));
                    if (lane == 0) cnt[warp * kPushMaxRanks + o] = __popc(bl);
                }
                __syncthreads();
                PUSH_TICK(5);
                if (warp == 0) {
                    for (unsigned o = 0; o < G; ++o) {
                        const unsigned v = lane < (unsigned)kPushWarps ? cnt[lane * kPushMaxRanks + o] : 0u;
                        unsigned incl = v;
#pragma unroll
                        for (int k = 1; k < kPushWarps; k <<= 1) {
                            const unsigned u = __shfl_up_sync(0xffffffffu, incl, k);
                            if ((int)lane >= k) incl += u;
                        }
                        if (lane < (unsigned)kPushWarps) pre[lane * kPushMaxRanks + o] = incl - v;
                    }
                    if (lane == 0) service();
                    // every source's rows of this chunk must have landed in my ring (flags are set after the stores).
                    // No flag of mine may stay unpublished while I wait for somebody else's (two CTAs on two GPUs could
                    // otherwise wait for each other's deferred flags): publish everything before blocking.
                    const bool need = lane < G && lane != me;
                    const unsigned long long *fl = q.flags + (size_t)(need ? lane : 0) * q.nchunks + cu;
                    const bool late = need && flag_peek(fl) < ready;
                    if (__any_sync(0xffffffffu, late)) {
                        if (lane == 0) publish(true, ready);
                        if (late) flag_wait(fl, ready);
                    }
                    __syncwarp();
                    PUSH_TICK(6);
                }
                __syncthreads();
                asm volatile("fence.proxy.async;" ::: "memory");  // acquired peer writes -> this thread's bulk gathers
                if (tid == 0) {
                    kbar_expect_tx(ldbar, rows * ROWB * 2);
                    bulk_row_g2s(ownb, p.x + (act + l0) * D, rows * ROWB, ldbar);
                }
                if (live) {
                    const double *src;
                    if (owner == me) {
                        src = p.x + (pas + prow) * D;
                    } else {
                        const unsigned char *slotp = reinterpret_cast<const unsigned char *>(q.recv) +
                                                     (((size_t)par * G + owner) * q.nchunks + cu) * slot_bytes;
                        const unsigned pi = __ldcg(reinterpret_cast<const unsigned *>(slotp) + g) +
                                            pre[warp * kPushMaxRanks + owner] + rkw;
                        if (pi < q.cap) src = reinterpret_cast<const double *>(slotp + kPushHeader + (size_t)pi * ROWB);
                        else src = q.peer_x[owner] + (pas + prow) * D;  // past the slot's capacity: read the owner
                    }
                    bulk_row_g2s(xpart + (size_t)tid * D, src, ROWB, ldbar);
                }
                const size_t k = act + l;
                const double lpk = live ? p.lp[k] : 0.0;
                if (warp == 0) {  // the next task, chosen while this group's rows are on their way
                    PUSH_TICK(7);
                    if (!ordered) nxt = pick(par, ready);
                    PUSH_TICK(4);
                }
                kbar_wait(ldbar, ldphase);
                ldphase ^= 1;
                if (live) {
                    double xk[D], xj[D], y[D];
#pragma unroll
                    for (int cc = 0; cc < D; cc += 2) {
                        const double2 a2 = *reinterpret_cast<const double2 *>(ownb + (size_t)tid * D + cc);
                        const double2 b2 = *reinterpret_cast<const double2 *>(xpart + (size_t)tid * D + cc);
                        xk[cc] = a2.x;
                        xk[cc + 1] = a2.y;
                        xj[cc] = b2.x;
                        xj[cc + 1] = b2.y;
                    }
                    const double z = dr.z;
#pragma unroll
                    for (int cc = 0; cc < D; ++cc) y[cc] = stretch_coord(xj[cc], xk[cc], z);  // :255
                    const double p1 = dn.logpdf(y);                                          // :257
                    const double tt = (p1 - lpk) + (double)dr.q * 0.6931471805599453;       // :260
                    bool acc;
                    if (tt > (double)p.margin) acc = true;
                    else if (tt < -(double)p.margin) acc = false;
                    else acc = accept_slow<false, false>(p, h, me * S + l, z, p1, lpk);
                    if (acc) {  // :261-265: only accepted rows are written (the kernel is bound by its DRAM traffic)
                        store_row<D>(p.x + k * D, y);
                        p.lp[k] = p1;
                        if (!reset) p.nacc[k] += 1u;
                    }
                    if (reset) {  // :285-288 burn-in counters are discarded (both halves of this position)
                        p.nacc[l] = 0u;
                        p.nacc[(size_t)S + l] = 0u;
                    }
                    if (store) chain_store<D>(p, chain_row(p, clk.sidx, batch, me * S + l), acc, y, xk, p1, lpk);
                }
                PUSH_TICK(7);
#ifdef KMC_PUSH_PROF
                ++nupd;
#endif
            } else if (warp == 0 && !ordered) {  // a round past the end of a ragged last chunk: nothing to do but to move on
                nxt = pick(par, ready);
            }
            __syncthreads();  // everyone has read `next` of this iteration before it is overwritten
            if (tid == 0) *next_slot = nxt;
            __syncthreads();
            next = *next_slot;
            PUSH_TICK(8);
        }

        if (batch == 1) clk.advance(store, p.nthin);
        PUSH_TICK(9);
        if (tid == 0) {  // all of this CTA's messages are complete: the last notes go out
            service();
            publish(true, ready);
            asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
        }
        asm volatile("fence.proxy.async;" ::: "memory");  // this thread's row stores (generic proxy) before anybody's bulk gathers
        PUSH_TICK(3);
        if (h + 1 < p.h1) {  // the reference's join between the two sweeps (:248/:273), local to this GPU
            target += gridDim.x;
            __syncthreads();
            if (gridDim.x > 1) {
                if (tid == 0) {
                    barrier_arrive(p.barrier);
                    barrier_wait(p.barrier, target);
                }
                __syncthreads();
            }
            asm volatile("fence.proxy.async;" ::: "memory");  // acquired row stores -> this thread's bulk gathers
        }
        PUSH_TICK(9);
    }
#ifdef KMC_PUSH_PROF
    if (tid == 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x / 2))
        printf("push rank %u cta %d: pushes %u update groups %u | cycles: sender %lld enum %lld gather-issue %lld | "
               "draws %lld scan+flags %lld group %lld | handoff %lld publish %lld pick %lld barrier+other %lld\n",
               me, (int)blockIdx.x, npush, nupd, pt[0], pt[1], pt[2], pt[5], pt[6], pt[7], pt[8], pt[3], pt[4], pt[9]);
#endif
}

}  // namespace kmc
