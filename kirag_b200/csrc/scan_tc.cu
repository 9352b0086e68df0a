// scan_tc.cu — the bf16 tcgen05 filter scan: the hot loop of the search.
//
// What it replaces: the inner loop of faiss.IndexFlatIP.search (reference call
// site /root/reference/retriever/index.py:47) — blocked sgemm of a query block
// against corpus blocks followed by a per-query heap/reservoir update.  Here
// the contraction runs on the 5th-generation tensor cores and the
// "does this score enter the running top-k'" test is fused into the
// accumulator read-out, so the score matrix never exists in memory.
//
// One kernel (scan_tc_pair_kernel): two CTAs on the two SMs of a TPC form a cluster and issue
// one tcgen05.mma.cta_group::2 of M=256 corpus rows (one 128-row tile per CTA) x N=PQ queries x
// K=16 per K-step.  Each CTA stages its own corpus tile and HALF of the query operand (PQ/2 rows).
// Data flow per CTA (persistent, one cluster per SM pair):
//   warp 0   producer : cp.async.bulk (TMA engine, SASS UBLKCP) of 16 KB shadow
//                       blocks [128 corpus rows x 64 k] into an N-stage ring;
//                       blocks are stored in HBM as the exact SWIZZLE_128B
//                       K-major shared-memory image, so each copy is one
//                       contiguous 16 KB read.  Streamed variant: the stage also
//                       holds this CTA's half of the query block
//   warp 1   leader   : MMA issuer, bf16 in, fp32 accumulate in TMEM; two
//                       accumulator stages so the read-out of tile t overlaps
//                       the MMAs of tile t+1
//            peer     : forwarder (tells the leader that the peer's stage is full)
//   warps 2+  filter  : tcgen05.ld 32x32b -> thread = one corpus row, registers
//                       = scores against 32 queries; compare with tau[q] (held in
//                       registers, fetched one work item ahead); survivors are
//                       appended to the per-query candidate buffer
// Warps 0 and 1 run their loops with all 32 lanes on warp-uniform values and predicate
// only the issuing instructions on elect.sync (see elect_one); one lane polls the mbarriers.
//
// Instantiations (scan_tc_pick):
//   <= 64 queries   64-query tile, resident (32 queries = 64 KB per CTA at d = 1024, 10-stage ring)  HBM-bound
//   <= 128 queries  128-query tile, resident (64 queries = 128 KB per CTA at d = 1024, 6-stage ring) HBM-bound
//   larger          streamed 256-query tiles (16 KB corpus + 16 KB query half per stage)             tensor-bound
// The 64- and 128-query tiles are streamed instead (query half-block in every stage) when the resident
// query half leaves too short a ring: d > 2048 at <= 64 queries, d > 1280 at <= 128 queries.
//
// Roofline: HBM for small query batches (algorithmic bytes = rows * d * 2 per
// launch, streamed exactly once), tensor pipe for large ones (2 * rows * nq * d
// flops per launch).
#include "common.cuh"
#include <cstdio>

namespace kirag {

constexpr int kMaxStages = 12;
constexpr int kBlockBytes = kTileRows * 128;  // one [128 x 64] bf16 block = 16 KB
constexpr int kSmemLimit = 227 * 1024;

// ------------------------------------------------------------------ PTX ----
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a protocol bug must not hang the GPU — trap after ~4 s.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity, int tag) {
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 8000000000LL) {
            printf("kirag scan_tc: mbarrier wait timed out (tag %d, block %d, thread %d, parity %u)\n", tag,
                   blockIdx.x, threadIdx.x, parity);
            __trap();
        }
    }
}
// Wait of a whole (converged) warp on one barrier: ONE lane polls, the others park at the warp barrier.  All 32 lanes
// polling costs 32 shared-memory barrier reads per try_wait; in an HBM-bound scan that traffic sits next to the
// filter warps' accumulator read-out (same-box A/B, profiles/r02_ab/r3f_ab.log: 6.1 -> 6.5 ms at 8 queries).
__device__ __forceinline__ void mbar_wait_warp(uint64_t* bar, uint32_t parity, int tag, int lane) {
    if (lane == 0) mbar_wait(bar, parity, tag);
    __syncwarp();
}
// One lane of the (converged) warp.  The producer / MMA / forwarder warps run their loops with ALL lanes on warp-uniform
// values and only predicate the issuing instructions on this: ptxas then keeps smem addresses, descriptors and
// barrier addresses in uniform registers.  With a single active thread (`if (lane == 0)`) it cannot prove uniformity
// and wraps every tcgen05.mma / bulk copy in an ELECT + 5x R2UR.BROADCAST waterfall: ncu (r2m, B = 4096) showed the MMA
// thread busy issuing ~115 instructions per k-block for ~480 of the 512 tensor cycles the four MMAs take.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ uint64_t policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar,
                                         uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `p` (a local shared-memory object) in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_rank(const void* p, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    // default semantics (release at CTA scope): a cluster-scope release costs a ~1k-cycle fence per
    // arrive, which serialised the forwarder; the data being signalled was written by the async
    // proxy and its arrival is already ordered by the local mbarrier that was waited on
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
__device__ __forceinline__ void tmem_alloc2(uint32_t* holder_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(holder_smem)),
                 "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc2(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16_2cta(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on the barrier at this shared-memory offset in every CTA of the cluster whose rank bit is set in `mask`
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar, uint16_t mask) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
        ::"r"(smem_u32(bar)), "h"(mask)
        : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ uint32_t tmem_ld1(uint32_t taddr) {
    uint32_t r;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr) : "memory");
    return r;
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// SWIZZLE_128B, K-major shared-memory matrix descriptor (sm_100 format):
//   [0,14) start address >> 4 | [16,30) LBO >> 4 (unused for swizzled K-major, 1)
//   [32,46) SBO >> 4 = 1024 B between 8-row groups | [46,48) version = 1 | [61,64) layout = 2
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3ffffu) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// kind::f16 instruction descriptor: D fp32, A/B bf16, both K-major, N>>3 at [17,23), M>>4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

struct ScanArgs {
    const uint8_t* shadow;   // corpus bf16 blocks
    const uint8_t* qshadow;  // query bf16 blocks, half tiles of PQ/2 rows
    int64_t n_rows;
    int d;
    int64_t nq;
    int64_t tile_lo, tile_hi, n_tiles, tile_mult;
    const float* tau;  // [round_up(nq, 256)], +inf in the pad
    Cand* cand;        // [nq, cap]
    int* cnt;          // [nq]
    int cap;
    int n_stages;
    int q_dep;         // 1: the query shadow is written by the kernel right before this one in the chain
                       // (level 0): the producer must pdl_wait() too; 0: only the filter warps wait
    float* dump;      // optional [n_rows, dump_ld] dense approx scores (debug / tests)
    int64_t dump_ld;
};

// ---------------------------------------------------------------- filter ----
// One thread = one corpus row; a warp owns NG groups of 32 query columns of the accumulator.
// Pass 1 reads every group from TMEM and keeps only a 32-bit "score >= tau[q]" mask per group.
// If nothing passed (the common case after the first levels) the accumulator is released at once.
// Otherwise lane c plays "owner of query column c" in every group: one ballot per column, then the
// counters of ALL groups are bumped by NG independent atomic instructions (one round trip in
// total, not one per group), and pass 2 re-reads from TMEM only the groups that have survivors
// and stores (score, row) at the reserved slots.
// The thresholds of this warp's columns live in registers (lane l holds tau of column g*32 + l, fetched through L2
// once per query tile, one work item ahead) and are broadcast by shuffles.  tau must not be read through L1 / the
// non-coherent path: it is rewritten by the previous kernel of a programmatically chained launch; and it must not be
// loaded inside the filter loop at all: with the memory system saturated by the corpus stream an L2 hit takes ~3000
// cycles while the accumulator is held (16 % on the HBM-bound variants in round 1, the bound of the streamed 2-CTA
// kernel at the ridge in round 2).
__device__ __forceinline__ uint32_t pass_mask(const ScanArgs& a, const uint32_t (&v)[32], int64_t q0, int64_t row,
                                              bool row_ok, float mytau) {
    uint32_t pass = 0;
#pragma unroll
    for (int c = 0; c < 32; ++c) {
        const float t = __shfl_sync(0xffffffffu, mytau, c);
        pass |= (__uint_as_float(v[c]) >= t ? 1u : 0u) << c;
    }
    if (!row_ok) pass = 0;
    if (a.dump && row_ok) {
#pragma unroll
        for (int c = 0; c < 32; ++c)
            if (q0 + c < a.nq) a.dump[row * a.dump_ld + q0 + c] = __uint_as_float(v[c]);
    }
    return pass;
}

// After the first levels survivors are rare (a row beats tau[q] for ~k'*growth of millions of rows),
// so a thread almost never has more than a few per work item: they are parked in a 4-entry
// per-thread register list (Stash).  The accumulator is released right after the last TMEM read;
// the slots are then reserved with independent atomics (all entries, all lanes, in flight
// together) and the (score, row) pairs are stored one work item LATER, after the next item's TMEM
// pass — the atomic round trip is never exposed to the tensor pipe.  A group in which some thread
// would overflow its list (the dense first levels) is appended immediately instead.
constexpr int kStash = 4;
struct Stash {
    uint32_t sv[kStash];  // score bits
    int sc[kStash];       // query column inside this warp's column range
    int slot[kStash];     // reserved buffer slot (valid after stash_reserve)
    int n;
    int64_t q0;
    int32_t row;
};
__device__ __forceinline__ void stash_clear(Stash& st) {
    st.n = 0;
    st.q0 = 0;
    st.row = 0;
#pragma unroll
    for (int j = 0; j < kStash; ++j) { st.sv[j] = 0; st.sc[j] = 0; st.slot[j] = -1; }
}
__device__ __forceinline__ void stash_reserve(const ScanArgs& a, Stash& st) {
#pragma unroll
    for (int j = 0; j < kStash; ++j) {
        st.slot[j] = -1;
        if (st.n > j && st.q0 + st.sc[j] < a.nq) st.slot[j] = atomicAdd(a.cnt + st.q0 + st.sc[j], 1);
    }
}
__device__ __forceinline__ void stash_store(const ScanArgs& a, const Stash& st) {
#pragma unroll
    for (int j = 0; j < kStash; ++j) {
        if (st.n > j && st.slot[j] >= 0 && st.slot[j] < a.cap) {
            Cand cd;
            cd.s = __uint_as_float(st.sv[j]);
            cd.id = st.row;
            a.cand[(st.q0 + st.sc[j]) * (int64_t)a.cap + st.slot[j]] = cd;
        }
    }
}

// 32x32 bit-matrix transpose across the warp: in, lane r holds word A[r] (bit c = A[r][c]); out,
// lane c holds the word whose bit r is A[r][c].  Five shuffle rounds instead of 32 ballots.
__device__ __forceinline__ uint32_t warp_transpose_bits(uint32_t x, int lane) {
#pragma unroll
    for (int s = 0; s < 5; ++s) {
        const int j = 16 >> s;
        const uint32_t m = (s == 0) ? 0x0000ffffu : (s == 1) ? 0x00ff00ffu : (s == 2) ? 0x0f0f0f0fu
                         : (s == 3) ? 0x33333333u : 0x55555555u;
        const uint32_t t = __shfl_xor_sync(0xffffffffu, x, j);
        x = (lane & j) ? ((x & ~m) | ((t & ~m) >> j)) : ((x & m) | ((t & m) << j));
    }
    return x;
}

// v[c] for a per-lane dynamic c: five rounds of pairwise selects (16 + 8 + 4 + 2 + 1), registers only
__device__ __forceinline__ uint32_t select32(const uint32_t (&v)[32], int c) {
    uint32_t a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = (c & 16) ? v[16 + i] : v[i];
#pragma unroll
    for (int i = 0; i < 8; ++i) a[i] = (c & 8) ? a[8 + i] : a[i];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = (c & 4) ? a[4 + i] : a[i];
#pragma unroll
    for (int i = 0; i < 2; ++i) a[i] = (c & 2) ? a[2 + i] : a[i];
    return (c & 1) ? a[1] : a[0];
}

// Survivors of one 32-column group (called only when some lane of the warp has one).  The 32 scores
// of the group are in registers with STATIC indices; a survivor's column is dynamic, so the scores
// are first spilled to a 128-byte per-thread scratch (local memory, L1-resident) and then indexed
// per lane — every lane walks its OWN set bits, the trip count is the largest number of survivors
// of a single row (1-2 after the first levels), not the number of distinct columns in the warp.
//   all pass (level 0, tau = -inf): slots are base + row, no ballots or dynamic indexing at all
//   sparse (normal) : every thread parks its few survivors in its Stash
//   dense (first levels, or a thread would overflow its Stash): the pass matrix is transposed so
//           that lane c knows which rows survive query column c; ONE atomic instruction bumps all
//           32 counters; each row then fetches (base, ballot) of its columns from the owner lanes
//           by shuffle and stores at base + (number of lower rows that also survive)
__device__ __forceinline__ void handle_survivors(const ScanArgs& a, const uint32_t (&v)[32], uint32_t pass,
                                                 int64_t q0g, int col_g, int32_t row, int lane, Stash& st) {
    if (__all_sync(0xffffffffu, pass == 0xffffffffu)) {
        // level 0 (tau = -inf): every row survives every column.  Lane c reserves 32 slots of query
        // column c; row r takes slot base_c + r.  Static register indices, no ballots.
        int mybase = a.cap;
        if (q0g + lane < a.nq) mybase = atomicAdd(a.cnt + q0g + lane, 32);
#pragma unroll
        for (int c = 0; c < 32; ++c) {
            const int slot = __shfl_sync(0xffffffffu, mybase, c) + lane;
            if (slot < a.cap) {
                Cand cd;
                cd.s = __uint_as_float(v[c]);
                cd.id = row;
                a.cand[(q0g + c) * (int64_t)a.cap + slot] = cd;
            }
        }
        return;
    }
    const bool dense = __any_sync(0xffffffffu, st.n + __popc(pass) > kStash);
    if (!dense) {
        // the common case after the first levels: a binary select tree over the 32 registers (31 SEL per survivor,
        // no memory).  The per-thread scratch below cost 4 KB of local stores per warp and call: 14 GB of L2 writes
        // per 2.6M-row level at 4096 queries, 10 % of the kernel's L2 sectors (ncu r2m), 2.9 GB of DRAM write-backs
        // per 21M-row step.  Same-process A/B (profiles/r02_ab/r2q, r2r): 21M rows B=4096 137.5 -> 135.4 ms, B=256
        // 10.9 -> 9.4 ms, 2.6M rows B=128 1.07 -> 1.02 ms, B <= 64 unchanged.
        for (uint32_t u = pass; u; u &= u - 1) {
            const int c = __ffs(u) - 1;
            const uint32_t val = select32(v, c);
#pragma unroll
            for (int j = 0; j < kStash; ++j)
                if (st.n == j) { st.sv[j] = val; st.sc[j] = col_g + c; }
            ++st.n;
        }
        return;
    }
    uint32_t loc[32];  // dense levels only: a 128-byte per-thread scratch (local memory, L1-resident) indexed per lane
#pragma unroll
    for (int c = 0; c < 32; ++c) loc[c] = v[c];
    uint32_t mybal = warp_transpose_bits(pass, lane);  // bit r: row (lane) r survives column `lane`
    if (q0g + lane >= a.nq) mybal = 0;
    int mybase = 0;
    if (mybal != 0) mybase = atomicAdd(a.cnt + q0g + lane, __popc(mybal));
    const unsigned lt = (1u << lane) - 1u;
    const int iters = __reduce_max_sync(0xffffffffu, __popc(pass));
    uint32_t u = pass;
    for (int i = 0; i < iters; ++i) {
        const bool has = u != 0;
        const int c = has ? (__ffs(u) - 1) : 0;
        u &= u - 1;
        const unsigned bal = __shfl_sync(0xffffffffu, mybal, c);
        const int base = __shfl_sync(0xffffffffu, mybase, c);
        if (has) {
            const int slot = base + __popc(bal & lt);
            if (slot < a.cap && ((bal >> lane) & 1u)) {
                Cand cd;
                cd.s = __uint_as_float(loc[c]);
                cd.id = row;
                a.cand[(q0g + c) * (int64_t)a.cap + slot] = cd;
            }
        }
    }
}

// taddr: TMEM address of this warp's first column (lane quadrant included); q0: first query of it.
// `release` is called exactly once, right after this warp's last read of the accumulator.
template <int NG, typename Release>
__device__ __forceinline__ void filter_item(const ScanArgs& a, uint32_t taddr, int64_t q0, int64_t row, bool row_ok,
                                            int lane, Stash& st, const float (&mytau)[NG], Release release) {
    stash_clear(st);
    st.q0 = q0;
    st.row = (int32_t)row;
#pragma unroll 1
    for (int g = 0; g < NG; ++g) {
        uint32_t v[32];
        tmem_ld32(taddr + g * 32, v);
        tmem_ld_wait();
        const uint32_t pass = pass_mask(a, v, q0 + g * 32, row, row_ok, mytau[g]);
        if (__any_sync(0xffffffffu, pass != 0))
            handle_survivors(a, v, pass, q0 + g * 32, g * 32, (int32_t)row, lane, st);
    }
    release();
}

// ---------------------------------------------------------------- kernel ----
// filter warps: 4 (one per TMEM lane quadrant), or 8 for wide query tiles (two warps per quadrant,
// each taking half of the columns)
template <int BQ> struct EpiCfg {
    static constexpr int kWarps = (BQ >= 128) ? 8 : 4;
    static constexpr int kThreads = 64 + 32 * kWarps;
    static constexpr int kGroups = BQ / 32 / (kWarps / 4);  // 32-column groups per warp
};

// ------------------------------------------------------------- pair kernel ----
// With one CTA per corpus tile the query operand made the L2 -> shared-memory traffic the limiter of
// large batches (48 KB per 128x256x64 MMA block); the pair stages 16 KB of corpus and 16 KB of queries
// per CTA for the same flops.
//   rank 0 (leader): producer, MMA issuer, filter warps
//   rank 1 (peer)  : producer, forwarder (tells the leader that the peer's stage is full),
//                    filter warps
// Barriers: full[s] lives in each CTA (leader: own expect_tx + the peer's forwarded arrive);
// empty[s] and tmem_full[a] are signalled in both CTAs by a multicast tcgen05.commit;
// tmem_empty[a] of the LEADER collects the filter warps of both CTAs.
// Instantiations:
//   PQ = 256, streamed  : large batches (tensor-bound); corpus block + half query block per stage
//   PQ = 128, resident  : 64 < batch <= 128 (HBM-bound); each CTA keeps ITS half of the single query
//                         tile (64 queries x d, 128 KB at d = 1024) resident in shared memory, so
//                         only corpus blocks are streamed: L2 -> SM traffic equals the HBM traffic
//   PQ = 64, resident   : batch <= 64 (HBM-bound, the default for KiRAG's 1-2 queries per retrieval):
//                         32 queries = 64 KB resident per CTA at d = 1024, 10-stage ring, four filter warps
//   PQ = 128 / 64, streamed : the same batches at a d where the resident half leaves too short a ring
template <int PQ, bool RES> struct PairCfg {
    static constexpr int kHalfQ = PQ / 2;                      // query rows staged per CTA
    static constexpr int kQHalfBytes = kHalfQ * 128;           // one [half x 64] bf16 block
    static constexpr int kStageBytes = kBlockBytes + (RES ? 0 : kQHalfBytes);
};

template <int PQ, bool RES>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(EpiCfg<PQ>::kThreads, 1)
scan_tc_pair_kernel(const ScanArgs a) {
    constexpr int kHalfQ = PairCfg<PQ, RES>::kHalfQ;
    constexpr int kQHalfBytes = PairCfg<PQ, RES>::kQHalfBytes;
    constexpr int kStageBytes = PairCfg<PQ, RES>::kStageBytes;
    constexpr uint16_t kPairMask = 0x3;  // both CTAs of the cluster
    extern __shared__ uint8_t smem_raw[];
    // 1024-byte alignment for the 128B swizzle atoms
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int KC = a.d >> 6;  // 64-wide k-blocks per row
    const int NS = a.n_stages;
    uint8_t* stage_base = smem;
    uint8_t* q_res = smem + (size_t)NS * kStageBytes;  // resident half query tile (RES only)
    uint8_t* tail = q_res + (RES ? (size_t)KC * kQHalfBytes : 0);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(tail);
    uint64_t* empty_bar = full_bar + kMaxStages;
    uint64_t* tmem_full = empty_bar + kMaxStages;
    uint64_t* tmem_empty = tmem_full + 2;
    uint64_t* q_bar = tmem_empty + 2;  // leader: own bytes + the peer's forward; peer: own bytes
    uint32_t* tmem_holder = reinterpret_cast<uint32_t*>(q_bar + 1);

    const int warp = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();  // 0: leader (issues the MMAs), 1: peer
    const int64_t pair = blockIdx.x / 2;
    const int64_t n_pairs = gridDim.x / 2;
    constexpr uint32_t kTmemCols = 2 * PQ;  // two accumulator stages of PQ columns
    const int n_qt = (int)((a.nq + PQ - 1) / PQ);
    // work item w = (pair of walk positions, query tile), query tile fastest so that a CTA re-reads its corpus tile
    // from L2; every pair takes one contiguous, equally sized range of w, so small levels still occupy all SM pairs
    const int64_t W = ((a.tile_hi - a.tile_lo + 1) / 2) * n_qt;
    const int64_t w_lo = W * pair / n_pairs;
    const int64_t w_hi = W * (pair + 1) / n_pairs;

    if (threadIdx.x == 0) {
        for (int s = 0; s < NS; ++s) { mbar_init(&full_bar[s], rank == 0 ? 2 : 1); mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { mbar_init(&tmem_full[s], 1); mbar_init(&tmem_empty[s], 2 * EpiCfg<PQ>::kWarps); }
        mbar_init(q_bar, rank == 0 ? 2 : 1);
        fence_barrier_init();
    }
    if (warp == 1) tmem_alloc2(tmem_holder, kTmemCols);
    tc_fence_before();
    cluster_sync_all();  // barriers of both CTAs are initialised before anyone signals across
    tc_fence_after();
    const uint32_t tmem_base = *tmem_holder;

    // tiles of this level are taken two at a time: walk position 2 p + rank
    if (warp == 0) {
        // =============================== producer ===============================
        // (all lanes run the warp-uniform loop, one elected lane issues: see elect_one)
        {
            // corpus blocks that are re-read once per query tile: evict_last, and evict_first on their LAST read (last
            // query tile) so that dead tiles, not live ones, make room for the next tiles.  DRAM reads of a 21M-row step
            // at batch 4096 (43.0 GB algorithmic; single-pass ncu, profiles/r02_ab/r2w, r2x): evict_normal 78.6 GB,
            // evict_last 61.8 GB, with the demotion 54.3 GB; time unchanged (DRAM is at 6 %).
            const uint64_t pol_x = (n_qt == 1) ? policy_evict_first() : policy_evict_last();
            const uint64_t pol_x_last = policy_evict_first();
            const uint64_t pol_q = policy_evict_last();
            if (a.q_dep) pdl_wait();  // level 0: the query shadow is being written by the previous kernel
            if (RES && elect_one()) {  // the batch is one query tile: this CTA's half stays in shared memory for the whole launch
                mbar_expect_tx(q_bar, (uint32_t)(KC * kQHalfBytes));
                bulk_g2s(q_res, a.qshadow + (size_t)rank * ((size_t)a.d * kHalfQ * 2), (uint32_t)(KC * kQHalfBytes),
                         q_bar, pol_q);
            }
            __syncwarp();
            int s = 0;
            uint32_t ph = 0;
            for (int64_t w = w_lo; w < w_hi; ++w) {
                const int64_t p = w / n_qt;
                const int qt = (int)(w - p * n_qt);
                int64_t ti = a.tile_lo + 2 * p + rank;
                if (ti >= a.tile_hi) ti = a.tile_hi - 1;  // ragged tail: stage a valid tile, rows are masked later
                const int64_t tile = (ti * a.tile_mult) % a.n_tiles;
                const uint8_t* xsrc = a.shadow + (size_t)tile * ((size_t)a.d * kTileRows * 2);
                // query shadow is stored in half tiles of PQ/2 rows: this CTA stages half tile 2*qt + rank
                const uint8_t* qsrc = a.qshadow + (size_t)(2 * qt + rank) * ((size_t)a.d * kHalfQ * 2);
                const uint64_t pol_xw = (n_qt > 1 && qt == n_qt - 1) ? pol_x_last : pol_x;
                for (int kc = 0; kc < KC; ++kc) {
                    mbar_wait_warp(&empty_bar[s], ph ^ 1u, 100 + s, lane);
                    uint8_t* dst = stage_base + (size_t)s * kStageBytes;
                    if (elect_one()) {
                        mbar_expect_tx(&full_bar[s], (uint32_t)kStageBytes);
                        bulk_g2s(dst, xsrc + (size_t)kc * kBlockBytes, kBlockBytes, &full_bar[s], pol_xw);
                        if (!RES)
                            bulk_g2s(dst + kBlockBytes, qsrc + (size_t)kc * kQHalfBytes, kQHalfBytes, &full_bar[s], pol_q);
                    }
                    __syncwarp();
                    if (++s == NS) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        {
            int s = 0;
            uint32_t ph = 0;
            if (rank == 1) {
                // ============================= forwarder =============================
                if (RES) {
                    mbar_wait_warp(q_bar, 0, 650, lane);                          // this CTA's half of the query tile has landed
                    if (elect_one()) mbar_arrive_cluster(map_to_rank(q_bar, 0));  // tell the leader
                    __syncwarp();
                }
                for (int64_t w = w_lo; w < w_hi; ++w) {
                    for (int kc = 0; kc < KC; ++kc) {
                        mbar_wait_warp(&full_bar[s], ph, 600 + s, lane);                    // this CTA's stage has landed
                        if (elect_one()) mbar_arrive_cluster(map_to_rank(&full_bar[s], 0));  // tell the leader
                        __syncwarp();
                        if (++s == NS) { s = 0; ph ^= 1u; }
                    }
                }
            } else {
                // ================================ MMA ================================
                constexpr uint32_t idesc = make_idesc_bf16(2 * kTileRows, PQ);
                if (RES) mbar_wait_warp(q_bar, 0, 200, lane);  // both halves of the query tile are resident
                uint32_t it = 0;
                for (int64_t w = w_lo; w < w_hi; ++w, ++it) {
                    const uint32_t as = it & 1u;
                    const uint32_t aph = (it >> 1) & 1u;
                    mbar_wait_warp(&tmem_empty[as], aph ^ 1u, 300 + as, lane);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + as * PQ;
                    for (int kc = 0; kc < KC; ++kc) {
                        mbar_wait_warp(&full_bar[s], ph, 400 + s, lane);  // own bytes + the peer's forward
                        tc_fence_after();
                        const uint32_t xa = smem_u32(stage_base + (size_t)s * kStageBytes);
                        const uint64_t da = make_sw128_desc(xa);
                        const uint64_t db = make_sw128_desc(RES ? smem_u32(q_res + (size_t)kc * kQHalfBytes) : xa + kBlockBytes);
                        if (elect_one()) {
#pragma unroll
                            for (int k4 = 0; k4 < 4; ++k4)
                                // +32 bytes (two 16-byte units) per K=16 step inside the 128-byte swizzle row
                                umma_bf16_2cta(d_tmem, da + (uint64_t)(k4 * 2), db + (uint64_t)(k4 * 2), idesc,
                                               (kc | k4) ? 1u : 0u);
                            umma_commit_2cta(&empty_bar[s], kPairMask);  // frees the stage in both CTAs once read
                            if (kc == KC - 1) umma_commit_2cta(&tmem_full[as], kPairMask);  // accumulator complete
                        }
                        __syncwarp();
                        if (++s == NS) { s = 0; ph ^= 1u; }
                    }
                }
            }
        }
    } else {
        // ================================ filter ================================
        const int quad = warp & 3;  // TMEM lane quadrant this warp may read
        const uint32_t lane_base = (uint32_t)(quad * 32) << 16;
        uint32_t leader_empty[2];
        leader_empty[0] = map_to_rank(&tmem_empty[0], 0);
        leader_empty[1] = map_to_rank(&tmem_empty[1], 0);
        constexpr int NG = EpiCfg<PQ>::kGroups;
        const int col0 = ((warp - 2) >> 2) * (NG * 32);  // this warp's first column inside the query tile
        uint32_t it = 0;
        Stash pend, cur;
        stash_clear(pend);
        pdl_wait();  // tau / cand / cnt come from the previous compaction; the corpus stream did not have to wait
        // Thresholds of this warp's columns: lane l holds tau of column g*32 + l.  They are fetched through L2 one
        // work item AHEAD (the streamed variant changes query tile with every item): ncu r2a at B = 256 had the
        // filter warps spend 52 % of their time on the in-loop tau loads — with the memory system saturated by the
        // corpus stream an L2 hit takes ~3000 cycles, four of them per item made the filter, not HBM or the tensor
        // pipe, the bound (22.6k cycles per item against 8.2k of MMA).
        float mytau[NG], nxtau[NG];
        {
            const int qt0 = RES ? 0 : (int)(w_lo % n_qt);
#pragma unroll
            for (int g = 0; g < NG; ++g)
                mytau[g] = (w_lo < w_hi) ? __ldcg(a.tau + (int64_t)qt0 * PQ + col0 + g * 32 + lane) : 0.f;
        }
        for (int64_t w = w_lo; w < w_hi; ++w, ++it) {
            const int64_t p = w / n_qt;
            const int qt = (int)(w - p * n_qt);
            const int64_t ti = a.tile_lo + 2 * p + rank;
            const bool tile_ok = ti < a.tile_hi;
            const int64_t tile = ((tile_ok ? ti : a.tile_hi - 1) * a.tile_mult) % a.n_tiles;
            const int64_t row = tile * kTileRows + quad * 32 + lane;
            const bool row_ok = tile_ok && row < a.n_rows;
            const uint32_t as = it & 1u;
            const uint32_t aph = (it >> 1) & 1u;
            const int qt_next = (qt + 1 == n_qt) ? 0 : qt + 1;
            const bool fetch = !RES && n_qt > 1 && w + 1 < w_hi;
#pragma unroll
            for (int g = 0; g < NG; ++g)
                nxtau[g] = fetch ? __ldcg(a.tau + (int64_t)qt_next * PQ + col0 + g * 32 + lane) : mytau[g];
            mbar_wait(&tmem_full[as], aph, 500 + as);
            tc_fence_after();
            const uint32_t ebar = leader_empty[as];
            filter_item<NG>(a, tmem_base + lane_base + as * PQ + col0, (int64_t)qt * PQ + col0, row, row_ok,
                            lane, cur, mytau, [=]() {
                                // all of this warp's reads of the accumulator are done
                                tc_fence_before();
                                __syncwarp();
                                if (lane == 0) mbar_arrive_cluster(ebar);
                            });
#pragma unroll
            for (int g = 0; g < NG; ++g) mytau[g] = nxtau[g];
            stash_store(a, pend);    // slots reserved one item ago
            stash_reserve(a, cur);   // atomics in flight until the next item has been read
            pend = cur;
        }
        stash_store(a, pend);
    }
    // Dependents are released only here: this kernel is tensor/epilogue-bound, and compaction CTAs that
    // sit resident (blocked in their pdl_wait) next to the filter warps for the whole level measurably
    // slowed it down; at the end the trigger still hides the next kernel's launch latency.
    pdl_launch_dependents();
    tc_fence_before();
    cluster_sync_all();  // nobody leaves (or frees TMEM) while the partner can still signal into this CTA
    if (warp == 1) {
        tc_fence_after();
        tmem_dealloc2(tmem_base, kTmemCols);
    }
}

// ------------------------------------------------------------------ host ----
int scan_tc_supported(int d) { return (d % 64 == 0 && d >= 64 && d <= 4096) ? 1 : 0; }

template <int PQ, bool RES>
static size_t pair_fixed_bytes(int d) {
    return 1024 + (2 * kMaxStages + 5) * 8 + 16 + (RES ? (size_t)(d / 64) * PairCfg<PQ, RES>::kQHalfBytes : 0);
}
template <int PQ, bool RES>
static int pair_stages(int d) {
    int ns = kMaxStages;
    while (ns > 0 && pair_fixed_bytes<PQ, RES>(d) + (size_t)ns * PairCfg<PQ, RES>::kStageBytes > (size_t)kSmemLimit) --ns;
    return ns;
}

int scan_tc_pick(int64_t nq, int d, ScanTcPlan* plan) {
    KIRAG_CHECK(scan_tc_supported(d), "scan_tc: dimension %d is not supported (need a multiple of 64, <= 4096)", d);
    // up to 64 queries: a resident 64-query tile (32 queries = 64 KB per CTA at d = 1024, 10 stages).  Same-box A/B
    // against the single-CTA resident kernels it replaced, 21M rows (profiles/r02_ab/r3j_ab.log, r3k_ab.log): 5.85 vs
    // 6.2 ms at 1-32 queries (7.3 TB/s whole-step), 6.1 vs 6.4 ms at 48, 6.2-6.6 vs 6.6-6.7 ms at 64.
    if (nq <= 64) { plan->bq = 64; plan->resident = pair_stages<64, true>(d) >= 6; }
    else if (nq <= 128) { plan->bq = 128; plan->resident = pair_stages<128, true>(d) >= 4; }
    else { plan->bq = 256; plan->resident = 0; }
    return 0;
}

size_t scan_tc_qshadow_bytes(int64_t nq, int d, const ScanTcPlan& plan) {
    const int64_t tiles = (nq + plan.bq - 1) / plan.bq;
    return (size_t)tiles * plan.bq * d * 2;
}

// one pair per SM pair with equal contiguous work ranges.  More, shorter ranges for the hardware block scheduler to
// balance (ncu r2a, B = 256: sm__cycles_active 0.99M-1.43M of 1.44M elapsed) gained nothing at 21M rows
// (profiles/r02_ab/r2c_knobs.log: B=256 13.3 vs 13.4 ms, B=512 20.5 vs 19.2 ms).
template <int PQ, bool RES>
static int launch_scan_pair(const ScanArgs& args_in, int num_sms, cudaStream_t st) {
    ScanArgs args = args_in;
    const int ns = pair_stages<PQ, RES>(args.d);
    KIRAG_CHECK(ns >= 2, "scan_tc pair: no room for a shared-memory pipeline");
    KIRAG_CHECK(!RES || args.nq <= PQ, "scan_tc pair: the resident variant takes a single query tile");
    args.n_stages = ns;
    const size_t smem = pair_fixed_bytes<PQ, RES>(args.d) + (size_t)ns * PairCfg<PQ, RES>::kStageBytes;
    if (ensure_dynamic_smem(scan_tc_pair_kernel<PQ, RES>, kSmemLimit)) return 1;
    int64_t pairs = ((args.tile_hi - args.tile_lo + 1) / 2) * ((args.nq + PQ - 1) / PQ);  // work items
    if (pairs > num_sms / 2) pairs = num_sms / 2;
    if (pairs <= 0) return 0;
    KIRAG_CUDA_OK(launch_chained(scan_tc_pair_kernel<PQ, RES>, dim3((unsigned)(2 * pairs)), dim3(EpiCfg<PQ>::kThreads), smem, st, args));
    KIRAG_LAUNCH_OK("scan_tc_pair_kernel");
    return 0;
}

static int launch_scan_args(const ScanArgs& args, const ScanTcPlan& plan, int num_sms, cudaStream_t st) {
    if (plan.bq == 64 && plan.resident) return launch_scan_pair<64, true>(args, num_sms, st);
    if (plan.bq == 64 && !plan.resident) return launch_scan_pair<64, false>(args, num_sms, st);
    if (plan.bq == 128 && plan.resident) return launch_scan_pair<128, true>(args, num_sms, st);
    if (plan.bq == 128 && !plan.resident) return launch_scan_pair<128, false>(args, num_sms, st);
    if (plan.bq == 256 && !plan.resident) return launch_scan_pair<256, false>(args, num_sms, st);
    set_error("scan_tc: no kernel for plan (bq=%d resident=%d)", plan.bq, plan.resident);
    return 1;
}

int launch_scan_tc(const void* shadow, int64_t n_rows, int d, const void* qshadow, int64_t nq,
                   const ScanTcPlan& plan, int64_t tile_lo, int64_t tile_hi, int64_t n_tiles,
                   int64_t tile_mult, const float* tau, Cand* cand, int* cnt, int cap, int num_sms,
                   int q_dep, cudaStream_t st) {
    ScanArgs args{};
    args.q_dep = q_dep;
    args.shadow = (const uint8_t*)shadow;
    args.qshadow = (const uint8_t*)qshadow;
    args.n_rows = n_rows;
    args.d = d;
    args.nq = nq;
    args.tile_lo = tile_lo;
    args.tile_hi = tile_hi;
    args.n_tiles = n_tiles;
    args.tile_mult = tile_mult;
    args.tau = tau;
    args.cand = cand;
    args.cnt = cnt;
    args.cap = cap;
    args.dump = nullptr;
    args.dump_ld = 0;
    return launch_scan_args(args, plan, num_sms, st);
}

int launch_scan_tc_dump(const void* shadow, int64_t n_rows, int d, const void* qshadow, int64_t nq,
                        const ScanTcPlan& plan, const float* tau_inf, int* cnt_scratch, float* dump,
                        int64_t dump_ld, int num_sms, cudaStream_t st) {
    ScanArgs args{};
    args.shadow = (const uint8_t*)shadow;
    args.qshadow = (const uint8_t*)qshadow;
    args.n_rows = n_rows;
    args.d = d;
    args.nq = nq;
    args.n_tiles = (n_rows + kTileRows - 1) / kTileRows;
    args.tile_lo = 0;
    args.tile_hi = args.n_tiles;
    args.tile_mult = 1;
    args.tau = tau_inf;  // +inf everywhere: nothing is appended
    args.cand = nullptr;
    args.cnt = cnt_scratch;
    args.cap = 0;
    args.dump = dump;
    args.dump_ld = dump_ld;
    args.q_dep = 1;
    return launch_scan_args(args, plan, num_sms, st);
}

}  // namespace kirag
