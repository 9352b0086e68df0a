// common.cuh — shared declarations for the kirag_b200 sm_100a library.
//
// Vocabulary (follows the reference's domain, /root/reference/retriever/index.py):
//   corpus row   one passage embedding, fp32 [d], implicit id = row number
//   master       the fp32 row-major corpus matrix [ntotal, d] (what faiss.IndexFlatIP stores)
//   shadow       a bf16 copy of the master in 128-row x 64-column blocks laid out
//                exactly as the 128B-swizzled shared-memory image tcgen05.mma reads
//   candidate    (approximate score, row) pair that survived the bf16 filter scan
//   level        one launch of the filter scan over a geometric slice of the tiles
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>
#include <float.h>

namespace kirag {

// ---------------------------------------------------------------- errors ---
void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define KIRAG_CUDA_OK(expr)                                                              \
    do {                                                                                  \
        cudaError_t _e = (expr);                                                          \
        if (_e != cudaSuccess) {                                                          \
            kirag::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),      \
                             __FILE__, __LINE__);                                         \
            return 1;                                                                     \
        }                                                                                 \
    } while (0)

#define KIRAG_CHECK(cond, ...)                                                            \
    do {                                                                                  \
        if (!(cond)) {                                                                    \
            kirag::set_error(__VA_ARGS__);                                                \
            return 1;                                                                     \
        }                                                                                 \
    } while (0)

#define KIRAG_LAUNCH_OK(name)                                                             \
    do {                                                                                  \
        cudaError_t _e = cudaGetLastError();                                              \
        if (_e != cudaSuccess) {                                                          \
            kirag::set_error("launch of %s failed: %s (%s:%d)", name,                     \
                             cudaGetErrorString(_e), __FILE__, __LINE__);                 \
            return 1;                                                                     \
        }                                                                                 \
        kirag::count_launch();                                                            \
    } while (0)

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) is a driver round trip; do it once per
// (kernel, device) instead of before every launch.  Keyed by the kernel's address (different
// template instantiations share one function-pointer TYPE).
int ensure_dynamic_smem_impl(const void* kernel, size_t bytes);
template <typename K>
inline int ensure_dynamic_smem(K kernel, size_t bytes) {
    return ensure_dynamic_smem_impl(reinterpret_cast<const void*>(kernel), bytes);
}

// ------------------------------------------- programmatic dependent launch ---
// The kernels of one search form a chain on one stream (init, convert, {scan, compact} per level,
// rescore, final), many of them a few microseconds long.  They are launched with the
// programmatic-stream-serialization attribute: a kernel's CTAs may become resident and run their
// independent prologue (barrier init, TMEM allocation, streaming the first corpus blocks, which no
// kernel of the chain modifies) while the previous kernel drains; everything that reads data produced
// earlier in the chain sits behind pdl_wait(), which returns once the previous grid has completed
// and its memory is visible.  Every kernel triggers its dependents at the very top: the trigger only
// allows the next grid to be SCHEDULED, ordering comes from pdl_wait() alone.
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#endif
bool pdl_enabled();  // KIRAG_PDL=0 turns the launch attribute off (the device-side instructions are then no-ops)

template <typename... KArgs, typename... Args>
inline cudaError_t launch_chained(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                                  Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

// ------------------------------------------------------- shadow geometry ---
constexpr int kTileRows = 128;   // corpus rows per shadow tile (= UMMA M)
constexpr int kKChunk = 64;      // bf16 elements per 128-byte swizzle row (= one k-block)
constexpr int kChunkBytes = 16;  // swizzle granule

// Byte offset of element (r, c) inside a [rows_per_tile x d] bf16 matrix stored
// as tiles of `rows_per_tile` rows; each tile is d/64 blocks of
// [rows_per_tile x 64] bf16, each block the SWIZZLE_128B K-major image:
// row rr at rr*128 bytes, 16-byte granule g stored at position g ^ (rr & 7).
__host__ __device__ __forceinline__ size_t shadow_offset(int64_t r, int c, int d, int rows_per_tile) {
    const int64_t tile = r / rows_per_tile;
    const int rr = (int)(r - tile * rows_per_tile);
    const int kc = c >> 6;
    const int cc = c & 63;
    const int g = cc >> 3;
    const size_t tile_bytes = (size_t)rows_per_tile * d * 2;
    const size_t block_bytes = (size_t)rows_per_tile * 128;
    return (size_t)tile * tile_bytes + (size_t)kc * block_bytes + (size_t)rr * 128 +
           (size_t)((g ^ (rr & 7)) << 4) + (size_t)(cc & 7) * 2;
}

// ------------------------------------------------------------- ordering ---
// Monotone map float -> uint32 (larger float => larger key).  NaN maps to 0,
// below -inf, so a NaN score never displaces a real one (FAISS's heap admits
// an element only if `thresh < score`, which is false for NaN).  -0.0f is
// folded onto +0.0f so that float equality and key equality coincide.
__host__ __device__ __forceinline__ uint32_t score_key(float f) {
    if (!(f == f)) return 0u;
    f += 0.0f;
#ifdef __CUDA_ARCH__
    uint32_t u = __float_as_uint(f);
#else
    union { float f; uint32_t u; } cv; cv.f = f; uint32_t u = cv.u;
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__host__ __device__ __forceinline__ float key_score(uint32_t k) {
    uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#ifdef __CUDA_ARCH__
    return __uint_as_float(u);
#else
    union { float f; uint32_t u; } cv; cv.u = u; return cv.f;
#endif
}
// 64-bit sort item: descending order on this value == (score desc, id asc).
__host__ __device__ __forceinline__ uint64_t pack_item(float score, int32_t id) {
    return ((uint64_t)score_key(score) << 32) | (uint64_t)(0xffffffffu - (uint32_t)id);
}
__host__ __device__ __forceinline__ int32_t item_id(uint64_t it) {
    return (int32_t)(0xffffffffu - (uint32_t)(it & 0xffffffffu));
}
__host__ __device__ __forceinline__ uint32_t item_key(uint64_t it) { return (uint32_t)(it >> 32); }

struct __align__(8) Cand {
    float s;
    int32_t id;
};

// ---------------------------------------------------- canonical fp32 dot ---
// THE definition of a returned score: lane l of a warp accumulates, in
// ascending order, the products of elements e = c*128 + l*4 + j (j = 0..3,
// c = 0, 1, ...) with round-to-nearest FMAs, then the 32 partials are summed by
// an xor-butterfly (16, 8, 4, 2, 1).  Both the rescoring kernel and the exact
// scan use this function, so a score does not depend on the path, the query
// batch size or the number of GPUs.
#ifdef __CUDACC__
__device__ __forceinline__ float canonical_partial(const float* __restrict__ x,
                                                   const float* __restrict__ q, int d, int lane,
                                                   bool vec4) {
    float acc = 0.0f;
    if (vec4) {
        // unrolled so that the independent loads of a row are in flight together; the FMA chain (and with
        // it the summation order) is the same sequential one
#pragma unroll 8
        for (int c = lane * 4; c < d; c += 128) {
            const float4 xv = *reinterpret_cast<const float4*>(x + c);
            const float4 qv = *reinterpret_cast<const float4*>(q + c);
            acc = __fmaf_rn(xv.x, qv.x, acc);
            acc = __fmaf_rn(xv.y, qv.y, acc);
            acc = __fmaf_rn(xv.z, qv.z, acc);
            acc = __fmaf_rn(xv.w, qv.w, acc);
        }
    } else {
        for (int c = lane * 4; c < d; c += 128) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (c + j < d) acc = __fmaf_rn(x[c + j], q[c + j], acc);
        }
    }
    return acc;
}
__device__ __forceinline__ float warp_butterfly_sum(float v) {
    v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, 16));
    v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, 8));
    v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, 4));
    v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, 2));
    v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, 1));
    return v;
}

// In-place descending bitonic sort of P (a power of two) 64-bit items in shared memory by the whole CTA.
__device__ __forceinline__ void bitonic_sort_desc(uint64_t* s, int P) {
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < (P >> 1); t += blockDim.x) {
                const int pos = 2 * t - (t & (stride - 1));
                const int par = pos + stride;
                const bool desc = ((pos & size) == 0);
                const uint64_t a = s[pos], b = s[par];
                if ((a < b) == desc) { s[pos] = b; s[par] = a; }
            }
            __syncthreads();
        }
    }
}

// (key, id) total order of the result lists: larger key first, then lower id
__device__ __forceinline__ bool item_before(uint32_t ka, int64_t ia, uint32_t kb, int64_t ib) {
    return (ka > kb) || (ka == kb && ia < ib);
}

// number of items of the sorted list (keys[0..n), ids[0..n)) that come before (key, id)
__device__ __forceinline__ int count_before(const uint32_t* keys, const int64_t* ids, int n, uint32_t key, int64_t id) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (item_before(keys[mid], ids[mid], key, id)) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__device__ __forceinline__ void group_barrier(int id, int n_threads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n_threads) : "memory");
}

// Pairwise merge tree of G lists sorted by (key desc, id asc), with distinct ids, run by one thread group (thread gt of
// gthreads, named barrier bar_id).  Buffer b of keys_buf / ids_buf is [G*k] (list l at [l*k, l*k + nv[b][l])); the
// lists start in buffer 0.  Two lists are merged by giving every element the rank "own position + number of elements
// of the sibling list that precede it" (one binary search) and keeping ranks < k: the top-k of a union is in the union
// of the top-k's, so truncating after every round is exact.  log2 G rounds, O(G k log k) steps, no sort.  Returns the
// buffer that holds the merged list (nv[result][0] items).  The buffers may be shared or global memory.
__device__ __forceinline__ int merge_tree(uint32_t* keys_buf, int64_t* ids_buf, int* const nv[2], int G, int k, int gt,
                                          int gthreads, int bar_id) {
    const size_t L = (size_t)G * k;
    int cur = 0;
    for (int n_lists = G; n_lists > 1; n_lists = (n_lists + 1) >> 1) {
        const uint32_t* kin = keys_buf + (size_t)cur * L;
        const int64_t* iin = ids_buf + (size_t)cur * L;
        uint32_t* kout = keys_buf + (size_t)(cur ^ 1) * L;
        int64_t* iout = ids_buf + (size_t)(cur ^ 1) * L;
        const int* nin = nv[cur];
        int* nout = nv[cur ^ 1];
        for (int i = gt; i < n_lists * k; i += gthreads) {
            const int l = i / k, j = i - l * k;
            const int mate = l ^ 1;
            const int n_own = nin[l];
            const int n_mate = (mate < n_lists) ? nin[mate] : 0;
            if (j == 0 && (l & 1) == 0) nout[l >> 1] = (n_own + n_mate < k) ? (n_own + n_mate) : k;
            if (j >= n_own) continue;
            const uint32_t key = kin[i];
            const int64_t id = iin[i];
            const int r = j + (n_mate ? count_before(kin + (size_t)mate * k, iin + (size_t)mate * k, n_mate, key, id) : 0);
            if (r < k) {
                kout[(size_t)(l >> 1) * k + r] = key;
                iout[(size_t)(l >> 1) * k + r] = id;
            }
        }
        group_barrier(bar_id, gthreads);
        cur ^= 1;
    }
    return cur;
}
#endif

// --------------------------------------------------- multi-device stripes ---
// A multi-device index (kirag_index_create_multi) with G shards keeps global row r in shard (r / 128) mod G at local
// row (r / (128 G)) * 128 + r mod 128.  Pure arithmetic: no id tables, shards within 128 rows of each other whatever
// the add sizes, and local order within a shard is monotone in the global id.
constexpr int kStripeRows = 128;
__host__ __device__ __forceinline__ int stripe_shard(int64_t r, int G) { return (int)((r / kStripeRows) % G); }
__host__ __device__ __forceinline__ int64_t stripe_local(int64_t r, int G) {
    return r / ((int64_t)kStripeRows * G) * kStripeRows + r % kStripeRows;
}
__host__ __device__ __forceinline__ int64_t stripe_global(int64_t local, int s, int G) {
    return (local / kStripeRows * G + s) * kStripeRows + local % kStripeRows;
}
// rows of shard s among the global rows [0, n)
__host__ __device__ __forceinline__ int64_t stripe_rows(int64_t n, int s, int G) {
    const int64_t span = (int64_t)kStripeRows * G;
    const int64_t rem = n % span - (int64_t)s * kStripeRows;
    return n / span * kStripeRows + (rem < 0 ? 0 : rem > kStripeRows ? kStripeRows : rem);
}

// ------------------------------------------------------------ result ids ---
// Every writer of a result id I takes it through this descriptor: map[row] for an index with an id table
// (KIRAG_INDEX_ID_MAP: the caller's external ids, FAISS's IndexIDMap), else row + offset (the row-sharded search's
// global id).  The table is indexed by the global row; a multi-device merge maps after the stripe -> global remap.
struct IdOut {
    int64_t offset;
    const int64_t* map;  // null: no id table
};
__device__ __forceinline__ int64_t out_id(const IdOut& o, int64_t row) { return o.map ? __ldg(o.map + row) : row + o.offset; }

// ------------------------------------------------------ kernel launchers ---
// convert.cu
// center: corpus rows are stored as bf16(x - center) (row_cdot == nullptr); for query rows pass row_cdot to get
// <q, center> per row instead (the rows themselves are converted unshifted)
int launch_convert_rows(const float* src, int64_t n_rows, int d, int64_t dst_row0, void* shadow,
                        int rows_per_tile, unsigned* maxnorm2_bits, float* row_norms, float* row_errs,
                        const float* center, float* row_cdot, cudaStream_t st);
// sums[0..d) += column sums of rows [0, n_rows), sums[d] += sum of squared elements
int launch_column_sums(const float* src, int64_t n_rows, int d, float* sums, cudaStream_t st);
// scan_exact.cu
constexpr int kExactNQ = 8;
int launch_scan_exact(const float* master, int64_t n, int d, const float* q, int nq_valid,
                      float* scores, int64_t ld, int num_sms, cudaStream_t st);
// rescore.cu
// tauk / qnorm / qerr (optional): candidates whose approximate score is below tauk[q] - 2 (eps_a |q| + eps_b |q - q~|)
// are not rescored (their slot gets NaN = absent)
int launch_rescore(const float* master, int d, const float* q, const Cand* cand, const int* cnt,
                   int cand_stride, int m, float* out_scores, int64_t nq, const float* tauk, const float* qnorm,
                   const float* qerr, float eps_a, float eps_b, cudaStream_t st);
// Same scores from a host-resident master (pinned, mapped at the same address): a row's loads are all issued before
// they are consumed.  The skip's qnorm / qerr are indexed by qmap[q] when qmap is given (else by q).
int launch_rescore_host(const float* master, int d, const float* q, const Cand* cand, const int* cnt,
                        int cand_stride, int m, float* out_scores, int64_t nq, const float* tauk, const int* qmap,
                        const float* qnorm, const float* qerr, float eps_a, float eps_b, cudaStream_t st);
// select.cu
constexpr int kSelectSeg = 8192;
constexpr int kWideCap = 32768;  // candidate buffer of small query batches (fewer, longer levels)
int launch_select_dense(const float* scores, int64_t ld, int64_t n, int nq, int m, Cand* out,
                        int* n_seg_out, cudaStream_t st);
int launch_select_pairs(const Cand* in, int64_t in_stride, const int* cnt, int fixed_count, int cap,
                        int nq, int m, Cand* out, int64_t out_stride, int n_seg, float* tau,
                        int* cnt_out, int* overflow, cudaStream_t st);
// tauk (optional, last level): receives the kth_k-th best approximate score among the kept candidates (-inf if fewer)
int launch_compact_topm(Cand* buf, int64_t stride, int* cnt, int cap, int nq, int m, float* tau, int* overflow,
                        float* tauk, int kth_k, cudaStream_t st);
// last compaction + fp32 rescoring + final sort + certificate in ONE cluster kernel (small query batches)
int launch_tail_fused(Cand* buf, int64_t stride, int* cnt, int cap, int nq, int m, float* tau, int* overflow,
                      const float* master, int d, const float* q, float* rescored, int k, float* D, int64_t* I,
                      IdOut ids, const float* qnorm, const float* qerr, const float* qcdot, float eps_a, float eps_b,
                      int* flags, int num_sms, cudaStream_t st);
int launch_final(const Cand* cand, int64_t cand_stride, const float* rescored, const int* cnt,
                 int fixed_count, int m_in, int nq, int k, float* D, int64_t* I, IdOut ids,
                 const float* tau, const float* qnorm, const float* qerr, const float* qcdot, float eps_a, float eps_b,
                 int check_cert, const int* overflow, int* flags, const int* qmap, cudaStream_t st);
int launch_merge(const float* D_all, const int64_t* I_all, int G, int64_t nq, int k, float* D_out,
                 int64_t* I_out, cudaStream_t st);
int launch_fill_pad(float* D, int64_t* I, int64_t n, cudaStream_t st);
// scan_tc.cu
// The scan runs on CTA pairs (cta_group::2, M = 256 corpus rows per MMA); each CTA stages half of a query tile,
// so the query shadow is laid out in half tiles of bq / 2 rows.
struct ScanTcPlan {
    int bq;        // query-tile width (UMMA N): 64, 128 or 256
    int resident;  // 1: query tile stays in shared memory for the whole launch (64 and 128 only)
};
int scan_tc_supported(int d);
int scan_tc_pick(int64_t nq, int d, ScanTcPlan* plan);
size_t scan_tc_qshadow_bytes(int64_t nq, int d, const ScanTcPlan& plan);
int launch_scan_tc(const void* shadow, int64_t n_rows, int d, const void* qshadow, int64_t nq,
                   const ScanTcPlan& plan, int64_t tile_lo, int64_t tile_hi, int64_t n_tiles,
                   int64_t tile_mult, const float* tau, Cand* cand, int* cnt, int cap, int num_sms,
                   int q_dep, cudaStream_t st);
int launch_scan_tc_dump(const void* shadow, int64_t n_rows, int d, const void* qshadow, int64_t nq,
                        const ScanTcPlan& plan, const float* tau_inf, int* cnt_scratch, float* dump,
                        int64_t dump_ld, int num_sms, cudaStream_t st);
// range.cu — range search: collect every entry with score > radius, then sort each query's segment
constexpr int kRangeRun = 8192;  // segments up to this length are sorted by one CTA; longer ones in runs of it + merges
// tau[i] = radius - eps(q) - <q, c> with q = qmap[i] (qmap == nullptr: q = i); +inf on the pad up to nb_pad; cnt zeroed
int launch_range_threshold(const int* qmap, const float* qnorm, const float* qerr, const float* qcdot, float radius,
                           float eps_a, float eps_b, int64_t nb, int64_t nb_pad, float* tau, int* cnt, cudaStream_t st);
// candidate buffer [nq, cap] of a filter scan, rescored [nq, m] its canonical scores (m >= every count <= cap; a query
// with cnt > cap overflowed and counts as empty): counts[q] = entries with score > radius; collect appends them at
// cursor[q] (advanced)
int launch_range_count_cand(const Cand* cand, int cap, const float* rescored, int m, const int* cnt, int64_t nq,
                            float radius, int* counts, cudaStream_t st);
int launch_range_collect_cand(const Cand* cand, int cap, const float* rescored, int m, const int* cnt, int64_t nq,
                              float radius, unsigned long long* cursor, uint64_t* items, cudaStream_t st);
// dense exact scores scores[q * ld + row], rows [0, n)
int launch_range_count_dense(const float* scores, int64_t ld, int64_t n, int nq, float radius, int* counts,
                             cudaStream_t st);
int launch_range_collect_dense(const float* scores, int64_t ld, int64_t n, int nq, float radius,
                               unsigned long long* cursor, uint64_t* items, cudaStream_t st);
// Query q's items[src_off[q] .. + lims[q+1] - lims[q]) -> D / I [lims[q], lims[q+1]) by (score desc, row asc), ids
// out_id(ids, row).  Segments of at most kRangeRun items: one CTA each.  The n_seg longer ones are listed in the device table
// tab = seg_src [n_seg] (item offset), seg_dst [n_seg] (result offset), seg_len [n_seg], seg_e0 [n_seg + 1] (prefix of
// the lengths, total_long in all); they are sorted in items / items2 (same offsets).  Stream-ordered.
int launch_range_emit(uint64_t* items, uint64_t* items2, int64_t nq, const int64_t* src_off, const int64_t* lims,
                      int n_seg, int64_t longest, int64_t total_long, const int64_t* tab, IdOut ids, float* D,
                      int64_t* I, cudaStream_t st);
// multi.cu — merges of a multi-device index's shard results on the home device (shard buffers read in place, through
// peer pointers)
constexpr int kMaxShards = 16;
// D_sh[s] / I_sh[s]: shard s's top-k [nq, k] (local ids, padding id -1).  Out: the global top-k [nq, k] by (score
// desc, global row asc), ids out_id(ids, global row), padding (-FLT_MAX, -1).  ws: workspace of multi_merge_ws_bytes(G, k, nq) bytes (may be null if 0).
size_t multi_merge_ws_bytes(int G, int k, int64_t nq);
int launch_multi_merge(const float* const* D_sh, const int64_t* const* I_sh, int G, int64_t nq, int k, IdOut ids,
                       float* D_out, int64_t* I_out, void* ws, cudaStream_t st);
// D_sh[s] / I_sh[s]: shard s's range result (local ids) with lims lims_sh [G, nq + 1] (device); glims [nq + 1] (device)
// the global lims; max_n the largest shard total.  Out: the global result, (score desc, global row asc) per query,
// ids out_id(ids, global row).
int launch_multi_range_merge(const float* const* D_sh, const int64_t* const* I_sh, const int64_t* lims_sh,
                             const int64_t* glims, int G, int64_t nq, int64_t max_n, IdOut ids, float* D_out,
                             int64_t* I_out, cudaStream_t st);

// compact.cu — row removal.  bits: (n_rows + 127) / 128 * 16 bytes, zeroed here, then bit r set for every removed old
// row r: the ids in ids[0..n_ids) that lie in [0, n_rows), or with ids == null the rows [lo, hi) (0 <= lo <= hi <=
// n_rows).  kept [(n_rows + 127) / 128]: rows of each 128-row group that stay.
int launch_removal_counts(const int64_t* ids, int64_t n_ids, int64_t lo, int64_t hi, int64_t n_rows, uint32_t* bits,
                          int* kept, cudaStream_t st);
// The same bitmap and counts for an index with an id table: old row r is removed when its id table[r] is selected —
// with sel == null the ids lo <= id < hi, else the ids of sel[0..n_sel), sorted ascending (launch_sort_ids).
int launch_removal_counts_by_id(const int64_t* table, int64_t n_rows, const int64_t* sel, int64_t n_sel, int64_t lo,
                                int64_t hi, uint32_t* bits, int* kept, cudaStream_t st);
// out[0..n) = in[0..n) sorted ascending (CUB radix sort).  temp: sort_ids_temp_bytes(n) bytes.
size_t sort_ids_temp_bytes(int64_t n);
int launch_sort_ids(const int64_t* in, int64_t* out, int64_t n, void* temp, size_t temp_bytes, cudaStream_t st);
// The id table follows the rows: the id of every kept old row of [i0, n_rows) goes to out[new - j0] (new row number as
// for launch_gather_kept).
int launch_compact_ids(const int64_t* table, const uint32_t* bits, const int64_t* group_base, int64_t i0, int64_t n_rows,
                       int64_t j0, int64_t* out, cudaStream_t st);
// the fp32 master of every shard, readable from the launching device (peer access, or a mapped host master)
struct ShardMasters { const float* p[kMaxShards]; };
// Kept old rows of [i0, i1) whose new row number lies in [j0, j1) -> out[(new - j0) * d ...], new = group_base[i / 128]
// (kept rows of the groups before) + kept rows before i in its group.  Old row i is read from shard stripe_shard(i, G)
// at local row stripe_local(i, G).
int launch_gather_kept(const ShardMasters& masters, int G, int d, const uint32_t* bits, const int64_t* group_base,
                       int64_t i0, int64_t i1, int64_t j0, int64_t j1, float* out, int num_sms, cudaStream_t st);

// pool.cu
int launch_pool_normalize(const void* hidden, const void* mask, float* out, void* out_lp, float* pooled_norm,
                          int64_t B, int64_t S, int64_t H, int64_t sb, int64_t ss, int64_t mb,
                          int hidden_dtype, int mask_dtype, int mode, int normalize,
                          cudaStream_t st);
int launch_pool_normalize_backward(const float* grad_out, const float* out, const float* pooled_norm,
                                   const void* mask, void* grad_hidden, int64_t B, int64_t S,
                                   int64_t H, int64_t mb, int hidden_dtype, int mask_dtype, int mode,
                                   int normalize, cudaStream_t st);

}  // namespace kirag
