// select.cu — top-m selection by (score descending, id ascending).
//
// FAISS keeps a per-query heap (k < 100) or reservoir (k >= 100) while it
// scans (the code behind faiss.IndexFlatIP.search, reference call site
// /root/reference/retriever/index.py:47).  Here selection is a separate,
// small stage: every list that has to be reduced — a 8192-row segment of
// dense exact scores, a query's candidate buffer after a filter level, the
// rescored candidates, the all-gathered per-shard results — is sorted by one
// CTA in shared memory with a bitonic network over 64-bit items whose integer
// order IS the (score desc, id asc) total order (common.cuh: pack_item).
// Lists are at most 8192 items (64 KB of shared memory).
#include "common.cuh"

namespace kirag {

__device__ __forceinline__ int next_pow2(int v) {
    int p = 32;
    while (p < v) p <<= 1;
    return p;
}

// ---- dense exact scores -> per-segment top-m --------------------------------
// grid (n_seg, nq); scores[q*ld + row]; out[(q*n_seg + seg)*m + j]
__global__ void __launch_bounds__(1024)
select_dense_kernel(const float* __restrict__ scores, int64_t ld, int64_t n, int m,
                    Cand* __restrict__ out) {
    extern __shared__ uint64_t items[];
    const int seg = blockIdx.x, q = blockIdx.y, n_seg = gridDim.x;
    const int64_t lo = (int64_t)seg * kSelectSeg;
    const int len = (int)((n - lo < kSelectSeg) ? (n - lo) : kSelectSeg);
    const int P = next_pow2(len);
    const float* src = scores + (int64_t)q * ld + lo;
    for (int i = threadIdx.x; i < P; i += blockDim.x)
        items[i] = (i < len) ? pack_item(src[i], (int32_t)(lo + i)) : 0ull;
    __syncthreads();
    bitonic_sort_desc(items, P);
    Cand* dst = out + ((int64_t)q * n_seg + seg) * m;
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
        Cand c;
        if (j < P && item_key(items[j]) != 0u) {
            c.s = key_score(item_key(items[j]));
            c.id = item_id(items[j]);
        } else {
            c.s = __int_as_float(0x7fc00000);
            c.id = -1;
        }
        dst[j] = c;
    }
}

// ---- candidate lists -> per-segment top-m ------------------------------------
// grid (n_seg, nq).  When n_seg == 1 this is also the between-level compaction
// of the filter path: it tightens tau[q] to the m-th best approximate score,
// resets the append counter and records buffer overflow.
__global__ void __launch_bounds__(1024)
select_pairs_kernel(const Cand* __restrict__ in, int64_t in_stride, const int* __restrict__ cnt,
                    int fixed_count, int cap, int m, Cand* __restrict__ out, int64_t out_stride,
                    float* __restrict__ tau, int* __restrict__ cnt_out, int* __restrict__ overflow) {
    extern __shared__ uint64_t items[];
    const int seg = blockIdx.x, q = blockIdx.y, n_seg = gridDim.x;
    int raw = cnt ? cnt[q] : fixed_count;
    int count = raw > cap ? cap : raw;
    const int lo = seg * kSelectSeg;
    int len = count - lo;
    if (len > kSelectSeg) len = kSelectSeg;
    if (len < 0) len = 0;
    const int P = next_pow2(len > m ? len : m);
    const Cand* src = in + (int64_t)q * in_stride + lo;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        uint64_t it = 0ull;
        if (i < len) {
            const Cand c = src[i];
            if (c.id >= 0) it = pack_item(c.s, c.id);
        }
        items[i] = it;
    }
    __syncthreads();
    // a list that already fits needs no sort unless it is the last reduction
    bitonic_sort_desc(items, P);
    Cand* dst = out + (int64_t)q * out_stride + (int64_t)seg * m;
    for (int j = threadIdx.x; j < m; j += blockDim.x) {
        Cand c;
        if (item_key(items[j]) != 0u) {
            c.s = key_score(item_key(items[j]));
            c.id = item_id(items[j]);
        } else {
            c.s = __int_as_float(0x7fc00000);
            c.id = -1;
        }
        dst[j] = c;
    }
    if (threadIdx.x == 0 && n_seg == 1) {
        // number of valid items kept
        int kept = len < m ? len : m;
        // items with key 0 (NaN scores / empty) sort last; count the valid prefix
        // by binary search over the sorted keys
        int a = 0, b = kept;
        while (a < b) {
            const int mid = (a + b) >> 1;
            if (item_key(items[mid]) != 0u) a = mid + 1; else b = mid;
        }
        kept = a;
        if (cnt_out) cnt_out[q] = kept;
        if (tau && kept >= m) tau[q] = key_score(item_key(items[m - 1]));
        if (overflow && raw > cap) overflow[q] = 1;
    }
}

// ---- between-level compaction: exact top-m SET + m-th value, no sort -----------
// After a filter level a query's buffer holds the m kept candidates plus the new survivors
// (a few thousand at most).  The next level only needs (a) the set of the m best and (b) the
// m-th best score (the new tau) — not their order.  One 256-thread CTA per query (several CTAs
// per SM), items in registers:
//   1. bits on which all score keys agree are taken from the AND/OR of the keys (no counting);
//   2. the m-th largest SCORE key is found by an MSB-first radix selection over the remaining
//      bits, 8 bits per pass: a 256-bin shared-memory histogram of the still-undecided items,
//      a suffix scan over the bins, three barriers per pass (scores of one query share their
//      high bits, so this is 2-4 passes);
//   3. only if several items tie with that score is the same selection run on the row ids of the
//      tied items (lower row wins, like the final order);
//   4. the kept items are compacted back to the front of the list (unordered).
constexpr int kCompactThreads = 256;       // normal buffers (<= kSelectSeg items): several CTAs per SM
constexpr int kCompactThreadsWide = 1024;  // wide buffers of small query batches (<= kWideCap items)
constexpr int kCompactMaxWarps = kCompactThreadsWide / 32;

struct CompactSmem {
    int hist[2][256];
    int warp_tot[8];                       // the bin scan is always done by the first 256 threads
    int warp_off[kCompactMaxWarps + 1];
    unsigned s_and, s_or, s_min;
    int s_valid;
    int piv_digit, piv_kk, piv_count;
};

// Among the items selected by `active(e)`, with digits `digit(e)` in [0, 256): finds the largest
// digit D such that at least kk active items have a digit >= D.  Returns D; kk becomes the rank
// still to be resolved INSIDE bin D and n_in_bin the population of bin D.  `hist` must be zero on
// entry and is left dirty; the caller alternates between the two histograms and re-zeroes the
// other one meanwhile.
template <int NS, typename Active, typename Digit>
__device__ __forceinline__ int radix_pass(CompactSmem& sm, int which, int& kk, int& n_in_bin, Active active,
                                          Digit digit) {
    int* hist = sm.hist[which];
#pragma unroll
    for (int e = 0; e < NS; ++e)
        if (active(e)) atomicAdd(&hist[digit(e)], 1);
    const bool binner = threadIdx.x < 256;  // warp-uniform: whole warps 0..7
    if (binner) sm.hist[which ^ 1][threadIdx.x] = 0;  // ready for the next pass
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int h = 0, incl = 0;
    if (binner) {
        h = hist[255 - threadIdx.x];  // thread t looks at digit 255 - t: descending digits
        incl = h;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) sm.warp_tot[warp] = incl;
    }
    __syncthreads();
    if (binner) {
        int before = 0;
#pragma unroll
        for (int w = 0; w < 8; ++w)
            if (w < warp) before += sm.warp_tot[w];
        incl += before;
        if (incl >= kk && incl - h < kk) {  // exactly one thread: the bin that holds rank kk
            sm.piv_digit = 255 - threadIdx.x;
            sm.piv_kk = kk - (incl - h);
            sm.piv_count = h;
        }
    }
    __syncthreads();
    kk = sm.piv_kk;
    n_in_bin = sm.piv_count;
    return sm.piv_digit;
}

// NS = register slots per thread (compile-time so that the counting loops carry no dead iterations)
template <int NS, int THREADS>
__device__ __forceinline__ void compact_topm_body(Cand* __restrict__ list, int q, int raw, int count, int cap, int m,
                                                  int* __restrict__ cnt, float* __restrict__ tau,
                                                  int* __restrict__ overflow, float* __restrict__ tauk, int kth_k,
                                                  CompactSmem& sm) {
    uint32_t sk[NS];  // score key, 0 = absent (NaN score / empty slot)
    uint32_t ik[NS];  // 0xffffffff - row: larger = lower row = better
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) { sm.s_and = 0xffffffffu; sm.s_or = 0u; sm.s_valid = 0; sm.s_min = 0xffffffffu; }
    if (threadIdx.x < 256) sm.hist[0][threadIdx.x] = 0;
    int valid_local = 0;
    unsigned my_and = 0xffffffffu, my_or = 0u;
#pragma unroll
    for (int e = 0; e < NS; ++e) {
        sk[e] = 0u;
        ik[e] = 0u;
        const int i = e * THREADS + threadIdx.x;
        if (i < count) {
            const Cand c = list[i];
            if (c.id >= 0) {
                sk[e] = score_key(c.s);
                ik[e] = 0xffffffffu - (uint32_t)c.id;
            }
        }
        if (sk[e] != 0u) { ++valid_local; my_and &= sk[e]; my_or |= sk[e]; }
    }
    __syncthreads();
    my_and = __reduce_and_sync(0xffffffffu, my_and);
    my_or = __reduce_or_sync(0xffffffffu, my_or);
    valid_local = __reduce_add_sync(0xffffffffu, valid_local);
    if (lane == 0) { atomicAnd(&sm.s_and, my_and); atomicOr(&sm.s_or, my_or); atomicAdd(&sm.s_valid, valid_local); }
    __syncthreads();
    const int valid = sm.s_valid;
    const int keep = valid < m ? valid : m;
    uint32_t spiv = 0u, ipiv = 0u;  // keep rule: sk > spiv || (sk == spiv && ik >= ipiv); (0,0) keeps every valid item
    int which = 0;
    const unsigned all_and = sm.s_and, differ = sm.s_and ^ sm.s_or;
    // MSB-first radix selection of the kk-th largest SCORE key among the items selected by `in_set`; n_eq = number
    // of set members tied at that key, kk = rank still to be resolved among them.  Bits above the highest bit in
    // which the valid keys differ are shared by every key (all_and) and need no pass.
    auto select_key = [&](auto in_set, int& kk, int& n_eq) -> uint32_t {
        int pos = 32 - __clz(differ);   // undecided low bits (0 if every key is the same)
        uint32_t prefix = (pos >= 32) ? 0u : (all_and >> pos) << pos;
        while (pos > 0) {
            const int w = pos < 8 ? pos : 8;
            const int shift = pos - w;
            const uint32_t hi = (pos >= 32) ? 0u : (prefix >> pos);
            const int ppos = pos;
            const int d = radix_pass<NS>(
                sm, which, kk, n_eq,
                [&](int e) { return in_set(e) && ((ppos >= 32) ? 0u : (sk[e] >> ppos)) == hi; },
                [&](int e) { return (int)((sk[e] >> shift) & ((1u << w) - 1u)); });
            which ^= 1;
            prefix |= (uint32_t)d << shift;
            pos = shift;
        }
        return prefix;
    };
    if (valid > m) {
        int kk = m;
        int n_eq = valid;               // items tied with the pivot prefix decided so far
        spiv = select_key([&](int e) { return sk[e] != 0u; }, kk, n_eq);
        // score key of the m-th best; kk of the n_eq items tied at spiv are kept
        if (n_eq > kk) {  // ties straddle rank m: the kk lowest rows among them win
            uint32_t ipre = 0u;
            int n_in = n_eq;
            for (int p2 = 32; p2 > 0; p2 -= 8) {
                const int shift = p2 - 8;
                const uint32_t hi = (p2 >= 32) ? 0u : (ipre >> p2);
                const int d = radix_pass<NS>(
                    sm, which, kk, n_in,
                    [&](int e) { return sk[e] == spiv && ((p2 >= 32) ? 0u : (ik[e] >> p2)) == hi; },
                    [&](int e) { return (int)((ik[e] >> shift) & 0xffu); });
                which ^= 1;
                ipre |= (uint32_t)d << shift;
            }
            ipiv = ipre;
        }
    }
    // Last level only (tauk != nullptr): the kth_k-th best APPROXIMATE score among the kept candidates.  Rescoring
    // then skips every candidate whose approximate score is below tauk - 2 eps: at least kth_k candidates have a
    // canonical score >= tauk - eps, the skipped ones have one < tauk - eps, so none of them can be in the top-k.
    if (tauk) {
        float tk = -INFINITY;
        if (keep >= kth_k) {  // block-uniform
            int kk = kth_k, n_eq = keep;
            const uint32_t key = select_key(
                [&](int e) { return sk[e] != 0u && (sk[e] > spiv || (sk[e] == spiv && ik[e] >= ipiv)); }, kk, n_eq);
            tk = key_score(key);
        }
        if (threadIdx.x == 0) tauk[q] = tk;
    }
    // compaction of the kept items back to the front of the list
    int mine = 0;
#pragma unroll
    for (int e = 0; e < NS; ++e) mine += (sk[e] != 0u && (sk[e] > spiv || (sk[e] == spiv && ik[e] >= ipiv)));
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) sm.warp_off[warp + 1] = incl;
    // the m-th best of exactly m items is their minimum
    if (valid == m) {
        uint32_t mn = 0xffffffffu;
#pragma unroll
        for (int e = 0; e < NS; ++e)
            if (sk[e] != 0u && sk[e] < mn) mn = sk[e];
        mn = __reduce_min_sync(0xffffffffu, mn);
        if (lane == 0) atomicMin(&sm.s_min, mn);
    }
    __syncthreads();  // every read of list[] happened before the loads above: safe to overwrite
    int pos = incl - mine;
#pragma unroll
    for (int w = 0; w < THREADS / 32; ++w)
        if (w < warp) pos += sm.warp_off[w + 1];
#pragma unroll
    for (int e = 0; e < NS; ++e) {
        if (sk[e] != 0u && (sk[e] > spiv || (sk[e] == spiv && ik[e] >= ipiv))) {
            Cand c;
            c.s = key_score(sk[e]);
            c.id = (int32_t)(0xffffffffu - ik[e]);
            list[pos++] = c;
        }
    }
    if (threadIdx.x == 0) {
        // new threshold: the m-th best score, once m items exist
        if (valid > m) tau[q] = key_score(spiv);
        else if (valid == m) tau[q] = key_score(sm.s_min);
        cnt[q] = keep;
        if (raw > cap) overflow[q] = 1;
    }
}

template <int THREADS, int MIN_CTAS>
__global__ void __launch_bounds__(THREADS, MIN_CTAS)
compact_topm_kernel(Cand* __restrict__ buf, int64_t stride, int* __restrict__ cnt, int cap, int m,
                    float* __restrict__ tau, int* __restrict__ overflow, float* __restrict__ tauk, int kth_k) {
    __shared__ CompactSmem sm;
    pdl_wait();
    pdl_launch_dependents();
    const int q = blockIdx.x;
    const int raw = cnt[q];
    const int count = raw > cap ? cap : raw;
    const int n_slots = (count + THREADS - 1) / THREADS;  // block-uniform
    Cand* list = buf + (int64_t)q * stride;
#define KIRAG_COMPACT_CASE(NS) compact_topm_body<NS, THREADS>(list, q, raw, count, cap, m, cnt, tau, overflow, tauk, kth_k, sm)
    if (n_slots <= 2) KIRAG_COMPACT_CASE(2);
    else if (n_slots <= 4) KIRAG_COMPACT_CASE(4);
    else if (n_slots <= 8) KIRAG_COMPACT_CASE(8);
    else if (n_slots <= 12) KIRAG_COMPACT_CASE(12);
    else if (n_slots <= 16) KIRAG_COMPACT_CASE(16);
    else if (n_slots <= 24) KIRAG_COMPACT_CASE(24);
    else KIRAG_COMPACT_CASE(32);
#undef KIRAG_COMPACT_CASE
}

// ---- rescored candidates -> D, I (+ certificate) -----------------------------
// grid nq.  Sorts the (canonical fp32 score, row) pairs, writes the first k as
// the result row and checks the exactness certificate:
//   every row that is NOT a candidate has approximate score <= tau[q]; its
//   canonical score is therefore <= tau[q] + eps with eps = eps_a * ||q|| +
//   eps_b * ||q - bf16(q)|| (api.cu::CertEps: the corpus-side maxima are folded
//   into eps_a / eps_b).  If the k-th canonical
//   score exceeds tau[q] + eps, no dropped row can enter the top-k.
// items[0..P) hold the packed (canonical score, row) pairs of query q (0 = absent); sorts them, writes row qo of
// D / I and evaluates the certificate.  Called by all threads of a CTA.
__device__ __forceinline__ void final_body(uint64_t* items, int P, int q, int64_t qo, int k, float* __restrict__ D,
                                           int64_t* __restrict__ I, int64_t id_offset, const float* __restrict__ tau,
                                           const float* __restrict__ qnorm, const float* __restrict__ qerr,
                                           const float* __restrict__ qcdot, float eps_a,
                                           float eps_b, int check_cert, const int* __restrict__ overflow,
                                           int* __restrict__ flags) {
    bitonic_sort_desc(items, P);
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        float s = -FLT_MAX;
        int64_t id = -1;
        if (j < P && item_key(items[j]) != 0u) {
            s = key_score(item_key(items[j]));
            id = (int64_t)item_id(items[j]) + id_offset;
        }
        D[qo * k + j] = s;
        I[qo * k + j] = id;
    }
    if (threadIdx.x == 0 && flags) {
        int fail = 0;  // 0 ok, 1 certificate failed, 2 candidate buffer overflowed
        const bool ovf = overflow && __ldcg(overflow + q);
        if (check_cert && tau) {
            const float t = __ldcg(tau + q);
            if (t > -INFINITY) {
                // something may have been dropped: need k valid results whose
                // k-th score clears the dropped bound
                if (k > P || item_key(items[k - 1]) == 0u) {
                    fail = 1;
                } else {
                    // tau lives in the domain of the (possibly centred) shadow: a dropped row's true score is at
                    // most tau + <q, c> + eps
                    const float kth = key_score(item_key(items[k - 1]));
                    const float eps = eps_a * qnorm[q] + eps_b * qerr[q];
                    const float shift = qcdot ? qcdot[q] : 0.0f;
                    if (!(kth - eps > t + shift)) fail = 1;
                }
            }
        }
        flags[q] = ovf ? 2 : fail;
    }
}

__global__ void __launch_bounds__(1024)
final_kernel(const Cand* __restrict__ cand, int64_t cand_stride, const float* __restrict__ rescored,
             const int* __restrict__ cnt, int fixed_count, int m_in, int k, float* __restrict__ D,
             int64_t* __restrict__ I, int64_t id_offset, const float* __restrict__ tau,
             const float* __restrict__ qnorm, const float* __restrict__ qerr, const float* __restrict__ qcdot,
             float eps_a, float eps_b, int check_cert,
             const int* __restrict__ overflow, int* __restrict__ flags,
             const int* __restrict__ qmap) {
    extern __shared__ uint64_t items[];
    pdl_wait();
    pdl_launch_dependents();
    const int q = blockIdx.x;
    int count = cnt ? cnt[q] : fixed_count;
    if (count > m_in) count = m_in;
    const int P = next_pow2(count > 0 ? count : 1);
    const Cand* src = cand + (int64_t)q * cand_stride;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        uint64_t it = 0ull;
        if (i < count) {
            const int32_t id = src[i].id;
            const float s = rescored ? rescored[(int64_t)q * m_in + i] : src[i].s;
            if (id >= 0) it = pack_item(s, id);
        }
        items[i] = it;
    }
    __syncthreads();
    const int64_t qo = qmap ? qmap[q] : q;
    final_body(items, P, q, qo, k, D, I, id_offset, tau, qnorm, qerr, qcdot, eps_a, eps_b, check_cert, overflow, flags);
}

// ---- fused tail of a small-batch search --------------------------------------------------
// Small query batches are latency-bound: last compaction, rescoring and the final sort are three dependent launches
// of a few microseconds each.  Here ONE kernel does all three, a thread-block cluster of C CTAs per query:
//   phase 1 (CTA 0)   exact top-k' selection of the candidate buffer (compact_topm_body)
//   phase 2 (all C)   fp32 rescoring of the k' survivors from the master, one warp per candidate, spread over the
//                     C SMs of the cluster (a single SM cannot pull 400 rows x 4 KB quickly)
//   phase 3 (CTA 0)   sort by (canonical score desc, row asc), write D / I, certificate
// The phases are separated by cluster barriers with release / acquire semantics; what crosses CTAs (the compacted
// list, the rescored scores) goes through global memory and is read with L2 loads.
__device__ __forceinline__ void cluster_barrier() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}

constexpr int kTailMaxM = 2048;

__global__ void __launch_bounds__(kCompactThreadsWide, 1)
tail_fused_kernel(Cand* __restrict__ buf, int64_t stride, int* __restrict__ cnt, int cap, int m,
                  float* __restrict__ tau, int* __restrict__ overflow, const float* __restrict__ master, int d,
                  const float* __restrict__ qmat, int vec4, float* __restrict__ rescored, int k,
                  float* __restrict__ D, int64_t* __restrict__ I, int64_t id_offset, const float* __restrict__ qnorm,
                  const float* __restrict__ qerr, const float* __restrict__ qcdot, float eps_a, float eps_b,
                  int* __restrict__ flags) {
    __shared__ CompactSmem sm;
    __shared__ uint64_t items[kTailMaxM];
    uint32_t crank, csize;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(crank));
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(csize));
    pdl_wait();
    pdl_launch_dependents();
    const int q = blockIdx.x / csize;
    Cand* list = buf + (int64_t)q * stride;
    if (crank == 0) {
        const int raw = cnt[q];
        const int count = raw > cap ? cap : raw;
        const int n_slots = (count + kCompactThreadsWide - 1) / kCompactThreadsWide;  // block-uniform
#define KIRAG_TAIL_CASE(NS) \
    compact_topm_body<NS, kCompactThreadsWide>(list, q, raw, count, cap, m, cnt, tau, overflow, nullptr, 0, sm)
        if (n_slots <= 2) KIRAG_TAIL_CASE(2);
        else if (n_slots <= 4) KIRAG_TAIL_CASE(4);
        else if (n_slots <= 8) KIRAG_TAIL_CASE(8);
        else if (n_slots <= 12) KIRAG_TAIL_CASE(12);
        else if (n_slots <= 16) KIRAG_TAIL_CASE(16);
        else if (n_slots <= 24) KIRAG_TAIL_CASE(24);
        else KIRAG_TAIL_CASE(32);
#undef KIRAG_TAIL_CASE
        __threadfence();
    }
    cluster_barrier();
    int keep = __ldcg(cnt + q);
    if (keep > m) keep = m;
    {
        const int lane = threadIdx.x & 31;
        const int gw = (int)crank * (kCompactThreadsWide / 32) + (threadIdx.x >> 5);
        const int n_gw = (int)csize * (kCompactThreadsWide / 32);
        const float* qrow = qmat + (int64_t)q * d;
        for (int j = gw; j < keep; j += n_gw) {
            const int32_t row = __ldcg(&list[j].id);
            float result = __int_as_float(0x7fc00000);
            if (row >= 0) result = warp_butterfly_sum(canonical_partial(master + (int64_t)row * d, qrow, d, lane, vec4 != 0));
            if (lane == 0) __stcg(rescored + (int64_t)q * m + j, result);
        }
        __threadfence();
    }
    cluster_barrier();
    if (crank != 0) return;
    const int P = next_pow2(keep > 0 ? keep : 1);
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        uint64_t it = 0ull;
        if (i < keep) {
            const int32_t id = __ldcg(&list[i].id);
            if (id >= 0) it = pack_item(__ldcg(rescored + (int64_t)q * m + i), id);
        }
        items[i] = it;
    }
    __syncthreads();
    final_body(items, P, q, q, k, D, I, id_offset, tau, qnorm, qerr, qcdot, eps_a, eps_b, 1, overflow, flags);
}

// ---- multi-GPU merge ---------------------------------------------------------
// grid nq.  G*k (score, int64 id) pairs -> top-k by (score desc, id asc).
__device__ __forceinline__ bool kv_before(uint32_t ka, int64_t ia, uint32_t kb, int64_t ib) {
    return (ka > kb) || (ka == kb && ia < ib);
}

__global__ void __launch_bounds__(1024)
merge_kernel(const float* __restrict__ D_all, const int64_t* __restrict__ I_all, int G, int64_t nq,
             int k, float* __restrict__ D_out, int64_t* __restrict__ I_out, int P) {
    extern __shared__ uint64_t smem_raw[];
    int64_t* ids = reinterpret_cast<int64_t*>(smem_raw);
    uint32_t* keys = reinterpret_cast<uint32_t*>(ids + P);
    const int64_t q = blockIdx.x;
    const int L = G * k;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        uint32_t key = 0u;
        int64_t id = INT64_MAX;
        if (i < L) {
            const int g = i / k, j = i - g * k;
            const int64_t src = ((int64_t)g * nq + q) * k + j;
            const int64_t v = I_all[src];
            if (v >= 0) { key = score_key(D_all[src]); id = v; }
            if (key == 0u) id = INT64_MAX;
        }
        keys[i] = key;
        ids[i] = id;
    }
    __syncthreads();
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < (P >> 1); t += blockDim.x) {
                const int pos = 2 * t - (t & (stride - 1));
                const int par = pos + stride;
                const bool desc = ((pos & size) == 0);
                const uint32_t ka = keys[pos], kb = keys[par];
                const int64_t ia = ids[pos], ib = ids[par];
                // in a descending run the element that comes "before" goes first
                const bool b_first = kv_before(kb, ib, ka, ia);
                if (b_first == desc && !(ka == kb && ia == ib)) {
                    keys[pos] = kb; keys[par] = ka;
                    ids[pos] = ib; ids[par] = ia;
                }
            }
            __syncthreads();
        }
    }
    for (int j = threadIdx.x; j < k; j += blockDim.x) {
        float s = -FLT_MAX;
        int64_t id = -1;
        if (j < P && keys[j] != 0u) { s = key_score(keys[j]); id = ids[j]; }
        D_out[q * k + j] = s;
        I_out[q * k + j] = id;
    }
}

__global__ void fill_pad_kernel(float* __restrict__ D, int64_t* __restrict__ I, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) { D[i] = -FLT_MAX; I[i] = -1; }
}

// ------------------------------------------------------------------ hosts ----
static int host_pow2(int v) {
    int p = 32;
    while (p < v) p <<= 1;
    return p;
}
static int sort_threads(int P) {
    int t = P / 2;
    if (t > 1024) t = 1024;
    if (t < 32) t = 32;
    return t;
}

template <typename K>
static int ensure_smem(K kernel, size_t bytes) {
    if (bytes > 48 * 1024) return ensure_dynamic_smem(kernel, bytes);
    return 0;
}

int launch_select_dense(const float* scores, int64_t ld, int64_t n, int nq, int m, Cand* out,
                        int* n_seg_out, cudaStream_t st) {
    const int64_t n_seg = (n + kSelectSeg - 1) / kSelectSeg;
    KIRAG_CHECK(n_seg > 0 && n_seg < 0x7fffffffLL && nq > 0 && nq <= 65535,
                "select_dense: bad grid (n_seg=%lld nq=%d)", (long long)n_seg, nq);
    KIRAG_CHECK(m <= kSelectSeg, "select_dense: m=%d > %d", m, kSelectSeg);
    const int P = host_pow2((int)((n < kSelectSeg) ? n : kSelectSeg));
    const size_t smem = (size_t)P * 8;
    if (ensure_smem(select_dense_kernel, (size_t)kSelectSeg * 8)) return 1;
    dim3 grid((unsigned)n_seg, (unsigned)nq);
    select_dense_kernel<<<grid, sort_threads(P), smem, st>>>(scores, ld, n, m, out);
    KIRAG_LAUNCH_OK("select_dense_kernel");
    if (n_seg_out) *n_seg_out = (int)n_seg;
    return 0;
}

int launch_select_pairs(const Cand* in, int64_t in_stride, const int* cnt, int fixed_count, int cap,
                        int nq, int m, Cand* out, int64_t out_stride, int n_seg, float* tau,
                        int* cnt_out, int* overflow, cudaStream_t st) {
    KIRAG_CHECK(nq > 0 && nq <= 65535 && n_seg > 0, "select_pairs: bad grid (n_seg=%d nq=%d)", n_seg, nq);
    KIRAG_CHECK(m <= kSelectSeg, "select_pairs: m=%d > %d", m, kSelectSeg);
    int longest = cap < kSelectSeg ? cap : kSelectSeg;
    if (longest < m) longest = m;
    const int P = host_pow2(longest);
    const size_t smem = (size_t)P * 8;
    if (ensure_smem(select_pairs_kernel, (size_t)kSelectSeg * 8)) return 1;
    dim3 grid((unsigned)n_seg, (unsigned)nq);
    select_pairs_kernel<<<grid, sort_threads(P), smem, st>>>(in, in_stride, cnt, fixed_count, cap, m,
                                                            out, out_stride, tau, cnt_out, overflow);
    KIRAG_LAUNCH_OK("select_pairs_kernel");
    return 0;
}

int launch_compact_topm(Cand* buf, int64_t stride, int* cnt, int cap, int nq, int m, float* tau, int* overflow,
                        float* tauk, int kth_k, cudaStream_t st) {
    KIRAG_CHECK(cap <= kWideCap && m <= cap, "compact_topm: cap=%d m=%d out of range", cap, m);
    if (nq <= 0) return 0;
    if (cap <= kSelectSeg) {
        KIRAG_CUDA_OK(launch_chained(compact_topm_kernel<kCompactThreads, 4>, dim3((unsigned)nq), dim3(kCompactThreads), 0,
                                     st, buf, stride, cnt, cap, m, tau, overflow, tauk, kth_k));
    } else {
        KIRAG_CUDA_OK(launch_chained(compact_topm_kernel<kCompactThreadsWide, 1>, dim3((unsigned)nq),
                                     dim3(kCompactThreadsWide), 0, st, buf, stride, cnt, cap, m, tau, overflow, tauk, kth_k));
    }
    KIRAG_LAUNCH_OK("compact_topm_kernel");
    return 0;
}

int launch_final(const Cand* cand, int64_t cand_stride, const float* rescored, const int* cnt,
                 int fixed_count, int m_in, int nq, int k, float* D, int64_t* I, int64_t id_offset,
                 const float* tau, const float* qnorm, const float* qerr, const float* qcdot, float eps_a, float eps_b,
                 int check_cert, const int* overflow, int* flags, const int* qmap, cudaStream_t st) {
    KIRAG_CHECK(m_in <= kSelectSeg, "final: m_in=%d > %d", m_in, kSelectSeg);
    const int P = host_pow2(m_in);
    const size_t smem = (size_t)P * 8;
    if (ensure_smem(final_kernel, (size_t)kSelectSeg * 8)) return 1;
    KIRAG_CUDA_OK(launch_chained(final_kernel, dim3((unsigned)nq), dim3(sort_threads(P)), smem, st, cand, cand_stride,
                                 rescored, cnt, fixed_count, m_in, k, D, I, id_offset, tau, qnorm, qerr, qcdot, eps_a, eps_b,
                                 check_cert, overflow, flags, qmap));
    KIRAG_LAUNCH_OK("final_kernel");
    return 0;
}

int launch_tail_fused(Cand* buf, int64_t stride, int* cnt, int cap, int nq, int m, float* tau, int* overflow,
                      const float* master, int d, const float* q, float* rescored, int k, float* D, int64_t* I,
                      int64_t id_offset, const float* qnorm, const float* qerr, const float* qcdot, float eps_a, float eps_b,
                      int* flags, int num_sms, cudaStream_t st) {
    KIRAG_CHECK(cap <= kWideCap && m <= cap && m <= kTailMaxM, "tail_fused: cap=%d m=%d out of range", cap, m);
    if (nq <= 0) return 0;
    // cluster size: as many SMs per query as the GPU has to spare, at most 8 (the portable limit)
    int C = 8;
    while (C > 1 && (int64_t)nq * C > num_sms) C >>= 1;
    const int vec4 = (d % 4 == 0) && ((reinterpret_cast<uintptr_t>(master) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(q) & 15) == 0);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(nq * C));
    cfg.blockDim = dim3(kCompactThreadsWide);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = st;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)C;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 2 : 1;
    KIRAG_CUDA_OK(cudaLaunchKernelEx(&cfg, tail_fused_kernel, buf, stride, cnt, cap, m, tau, overflow, master, d, q, vec4,
                                     rescored, k, D, I, id_offset, qnorm, qerr, qcdot, eps_a, eps_b, flags));
    KIRAG_LAUNCH_OK("tail_fused_kernel");
    return 0;
}

int launch_merge(const float* D_all, const int64_t* I_all, int G, int64_t nq, int k, float* D_out,
                 int64_t* I_out, cudaStream_t st) {
    if (nq <= 0) return 0;
    const int64_t L = (int64_t)G * k;
    KIRAG_CHECK(L <= kSelectSeg, "merge: G*k=%lld exceeds %d", (long long)L, kSelectSeg);
    const int P = host_pow2((int)L);
    const size_t smem = (size_t)P * 12;
    if (ensure_smem(merge_kernel, (size_t)kSelectSeg * 12)) return 1;
    merge_kernel<<<(unsigned)nq, sort_threads(P), smem, st>>>(D_all, I_all, G, nq, k, D_out, I_out, P);
    KIRAG_LAUNCH_OK("merge_kernel");
    return 0;
}

int launch_fill_pad(float* D, int64_t* I, int64_t n, cudaStream_t st) {
    if (n <= 0) return 0;
    fill_pad_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(D, I, n);
    KIRAG_LAUNCH_OK("fill_pad_kernel");
    return 0;
}

}  // namespace kirag
