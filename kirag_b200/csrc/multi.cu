// multi.cu — the merges of a single-process multi-device index (kirag_index_create_multi; the shards, their worker
// threads and the stripe copies are in api.cu).  Both kernels run on the home device and read every shard's results in
// place through peer pointers; no [G, nq, k] gather comes first.
//   top-k   the G sorted [nq, k] lists are read, local ids are remapped to global ones by the stripe arithmetic
//           (common.cuh::stripe_global) and the lists are merged by the rank-based pairwise tree
//           (common.cuh::merge_tree, shared with the exchange of the row-sharded search); the merged global rows are
//           written through common.cuh::out_id (offset or id table);
//   range   one thread per shard entry computes its global position: global lims[q] + own position + for every other
//           shard the number of its entries of query q that precede it (one binary search each, on global ids).
#include "common.cuh"
#include "../../include/kirag_b200.h"

namespace kirag {

// ----------------------------------------------------------------------------------------------- top-k merge ----
constexpr int kMultiMergeThreads = 512;
constexpr int kMultiMergeSmem = 96 * 1024;
constexpr int kMultiMergeWsBlocks = 148;  // CTAs of a merge whose lists do not fit shared memory (global workspace)

struct MultiMergeArgs {
    const float* D[kMaxShards];
    const int64_t* I[kMaxShards];
    int G, k, n_groups;
    int64_t nq;
    IdOut ids;
    float* D_out;
    int64_t* I_out;
    uint8_t* ws;  // null: the lists live in shared memory
};

__global__ void __launch_bounds__(kMultiMergeThreads) multi_merge_kernel(const MultiMergeArgs a) {
    extern __shared__ uint64_t msmem[];
    __shared__ int nv_all[4][2 * kMaxShards];
    const int G = a.G, k = a.k;
    const size_t L = (size_t)G * k;
    const int n_groups = a.n_groups;
    const int gthreads = kMultiMergeThreads / n_groups;
    const int grp = threadIdx.x / gthreads;
    const int gt = threadIdx.x - grp * gthreads;
    uint8_t* base = a.ws ? a.ws + ((size_t)blockIdx.x * n_groups + grp) * 2 * L * 12
                         : reinterpret_cast<uint8_t*>(msmem) + (size_t)grp * 2 * L * 12;
    int64_t* ids_buf = reinterpret_cast<int64_t*>(base);                 // [2][L]
    uint32_t* keys_buf = reinterpret_cast<uint32_t*>(base + 2 * L * 8);  // [2][L]
    int* const nv[2] = {nv_all[grp], nv_all[grp] + kMaxShards};
    for (int64_t q = (int64_t)blockIdx.x * n_groups + grp; q < a.nq; q += (int64_t)gridDim.x * n_groups) {
        if (gt < G) nv[0][gt] = 0;
        group_barrier(1 + grp, gthreads);
        for (int i = gt; i < (int)L; i += gthreads) {
            const int s = i / k, j = i - s * k;
            int64_t id = a.I[s][q * k + j];
            uint32_t key = 0u;
            if (id >= 0) key = score_key(a.D[s][q * k + j]);
            if (key != 0u) {
                id = stripe_global(id, s, G);
                atomicAdd(&nv[0][s], 1);  // valid items form a prefix of each list
            }
            keys_buf[i] = key;
            ids_buf[i] = id;
        }
        group_barrier(1 + grp, gthreads);
        const int cur = merge_tree(keys_buf, ids_buf, nv, G, k, gt, gthreads, 1 + grp);
        const int total = nv[cur][0];
        for (int j = gt; j < k; j += gthreads) {
            const bool ok = j < total;
            a.D_out[q * k + j] = ok ? key_score(keys_buf[(size_t)cur * L + j]) : -FLT_MAX;
            a.I_out[q * k + j] = ok ? ids_buf[(size_t)cur * L + j] : -1;
        }
        group_barrier(1 + grp, gthreads);
    }
    // global rows -> ids, each thread over the entries it wrote above.  A separate pass: mapping in the loop above made
    // ptxas spill a pointer across the merge.
    if (!a.ids.map && !a.ids.offset) return;
    for (int64_t q = (int64_t)blockIdx.x * n_groups + grp; q < a.nq; q += (int64_t)gridDim.x * n_groups)
        for (int j = gt; j < k; j += gthreads) {
            const int64_t row = a.I_out[q * k + j];
            if (row >= 0) a.I_out[q * k + j] = out_id(a.ids, row);
        }
}

// thread groups per CTA when the two list buffers of a group fit shared memory; 0 when they do not
static int multi_merge_groups(int G, int k) {
    const size_t per_query = (size_t)2 * G * k * 12;
    for (int g = 4; g >= 1; g >>= 1)
        if (per_query * g <= (size_t)kMultiMergeSmem) return g;
    return 0;
}

size_t multi_merge_ws_bytes(int G, int k, int64_t nq) {
    if (multi_merge_groups(G, k) > 0) return 0;
    const int64_t blocks = nq < kMultiMergeWsBlocks ? nq : kMultiMergeWsBlocks;
    return (size_t)blocks * 2 * G * k * 12;
}

int launch_multi_merge(const float* const* D_sh, const int64_t* const* I_sh, int G, int64_t nq, int k, IdOut ids,
                       float* D_out, int64_t* I_out, void* ws, cudaStream_t st) {
    KIRAG_CHECK(G >= 1 && G <= kMaxShards && k >= 1 && nq >= 0, "multi_merge: bad shape G=%d k=%d", G, k);
    if (nq == 0) return 0;
    MultiMergeArgs a{};
    for (int s = 0; s < G; ++s) { a.D[s] = D_sh[s]; a.I[s] = I_sh[s]; }
    a.G = G; a.k = k; a.nq = nq; a.ids = ids; a.D_out = D_out; a.I_out = I_out;
    const int groups = multi_merge_groups(G, k);
    size_t smem = 0;
    int64_t blocks;
    if (groups > 0) {
        a.n_groups = groups;
        smem = (size_t)groups * 2 * G * k * 12;
        blocks = (nq + groups - 1) / groups;
        if (blocks > 2 * 148) blocks = 2 * 148;
        // unconditionally (the call is cached): the kernel's static shared memory counts against the default 48 KB too
        if (ensure_dynamic_smem(multi_merge_kernel, kMultiMergeSmem)) return 1;
    } else {
        KIRAG_CHECK(ws != nullptr, "multi_merge: G*k=%lld needs a workspace", (long long)G * k);
        a.n_groups = 1;
        a.ws = static_cast<uint8_t*>(ws);
        blocks = nq < kMultiMergeWsBlocks ? nq : kMultiMergeWsBlocks;
    }
    multi_merge_kernel<<<(unsigned)blocks, kMultiMergeThreads, smem, st>>>(a);
    KIRAG_LAUNCH_OK("multi_merge_kernel");
    return 0;
}

// ----------------------------------------------------------------------------------------------- range merge ----
struct MultiRangeArgs {
    const float* D[kMaxShards];
    const int64_t* I[kMaxShards];
    const int64_t* lims;   // [G, nq + 1]
    const int64_t* glims;  // [nq + 1]
    int G;
    int64_t nq;
    IdOut ids;
    float* D_out;
    int64_t* I_out;
};

// entries of shard s's segment [lo, hi) (local ids, remapped on the fly) that precede (key, gid)
__device__ __forceinline__ int64_t count_before_shard(const MultiRangeArgs& a, int s, int64_t lo, int64_t hi,
                                                      uint32_t key, int64_t gid) {
    int64_t l = lo, h = hi;
    while (l < h) {
        const int64_t mid = (l + h) >> 1;
        if (item_before(score_key(a.D[s][mid]), stripe_global(a.I[s][mid], s, a.G), key, gid)) l = mid + 1; else h = mid;
    }
    return l - lo;
}

// grid (entries of the largest shard / 256, G): thread e of row s places entry e of shard s
__global__ void multi_range_merge_kernel(const MultiRangeArgs a) {
    const int s = blockIdx.y;
    const int64_t* lims = a.lims + (size_t)s * (a.nq + 1);
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= lims[a.nq]) return;
    int64_t lo = 0, hi = a.nq;  // query q with lims[q] <= e < lims[q + 1]
    while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (lims[mid] <= e) lo = mid; else hi = mid;
    }
    const int64_t q = lo;
    const float score = a.D[s][e];
    const uint32_t key = score_key(score);
    const int64_t gid = stripe_global(a.I[s][e], s, a.G);
    int64_t pos = a.glims[q] + (e - lims[q]);
    for (int t = 0; t < a.G; ++t) {
        if (t == s) continue;
        const int64_t* lt = a.lims + (size_t)t * (a.nq + 1);
        pos += count_before_shard(a, t, lt[q], lt[q + 1], key, gid);
    }
    a.D_out[pos] = score;
    a.I_out[pos] = out_id(a.ids, gid);
}

int launch_multi_range_merge(const float* const* D_sh, const int64_t* const* I_sh, const int64_t* lims_sh,
                             const int64_t* glims, int G, int64_t nq, int64_t max_n, IdOut ids, float* D_out,
                             int64_t* I_out, cudaStream_t st) {
    KIRAG_CHECK(G >= 1 && G <= kMaxShards && nq >= 0 && max_n >= 0, "multi_range_merge: bad shape G=%d", G);
    if (nq == 0 || max_n == 0) return 0;
    MultiRangeArgs a{};
    for (int s = 0; s < G; ++s) { a.D[s] = D_sh[s]; a.I[s] = I_sh[s]; }
    a.lims = lims_sh; a.glims = glims; a.G = G; a.nq = nq; a.ids = ids; a.D_out = D_out; a.I_out = I_out;
    multi_range_merge_kernel<<<dim3((unsigned)((max_n + 255) / 256), (unsigned)G), 256, 0, st>>>(a);
    KIRAG_LAUNCH_OK("multi_range_merge_kernel");
    return 0;
}

}  // namespace kirag
