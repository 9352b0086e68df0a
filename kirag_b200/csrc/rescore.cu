// rescore.cu — fp32 rescoring of the candidates that survived the bf16 filter.
//
// The bf16 tcgen05 scan only decides WHICH rows can be in the top-k; the
// score that is returned (and that orders the result) is recomputed here from
// the fp32 master with the canonical summation order, so it is what
// faiss.IndexFlatIP.search would return up to fp32 summation order (reference
// call site /root/reference/retriever/index.py:47).
//
// One warp per (query, candidate): a gather of 4*d-byte rows.  Implementation
// traffic (not algorithmic): nq * m * d * 4 bytes.
#include "common.cuh"

namespace kirag {

__global__ void __launch_bounds__(256)
rescore_kernel(const float* __restrict__ master, int d, const float* __restrict__ q,
               const Cand* __restrict__ cand, const int* __restrict__ cnt, int cand_stride, int m,
               float* __restrict__ out, int64_t nq, bool vec4, const float* __restrict__ tauk,
               const float* __restrict__ qnorm, const float* __restrict__ qerr, float eps_a, float eps_b) {
    pdl_wait();
    pdl_launch_dependents();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (warp >= nq * m) return;
    const int64_t qi = warp / m;
    const int j = (int)(warp - qi * m);
    int count = cnt ? cnt[qi] : m;
    if (count > m) count = m;
    float result = __int_as_float(0x7fc00000);  // NaN marks an empty slot
    if (j < count) {
        const Cand cd = cand[qi * (int64_t)cand_stride + j];
        const int32_t row = cd.id;
        // a candidate this far below the k-th best approximate score cannot reach the top-k (select.cu, tauk)
        bool needed = true;
        if (tauk) needed = cd.s >= __ldcg(tauk + qi) - 2.0f * (eps_a * __ldcg(qnorm + qi) + eps_b * __ldcg(qerr + qi));
        if (row >= 0 && needed) {
            const float* x = master + (int64_t)row * d;
            const float part = canonical_partial(x, q + qi * (int64_t)d, d, lane, vec4);
            result = warp_butterfly_sum(part);
        }
    }
    if (lane == 0) out[qi * (int64_t)m + j] = result;
}

int launch_rescore(const float* master, int d, const float* q, const Cand* cand, const int* cnt,
                   int cand_stride, int m, float* out_scores, int64_t nq, const float* tauk, const float* qnorm,
                   const float* qerr, float eps_a, float eps_b, cudaStream_t st) {
    if (nq <= 0 || m <= 0) return 0;
    const int threads = 256;
    const int64_t warps = nq * m;
    const int64_t blocks = (warps + (threads / 32) - 1) / (threads / 32);
    KIRAG_CHECK(blocks < 0x7fffffffLL, "rescore: too many candidates (%lld warps)", (long long)warps);
    const bool vec4 = (d % 4 == 0) && ((reinterpret_cast<uintptr_t>(master) & 15) == 0) &&
                      ((reinterpret_cast<uintptr_t>(q) & 15) == 0);
    KIRAG_CUDA_OK(launch_chained(rescore_kernel, dim3((unsigned)blocks), dim3(threads), 0, st, master, d, q, cand, cnt,
                                 cand_stride, m, out_scores, nq, vec4, tauk, qnorm, qerr, eps_a, eps_b));
    KIRAG_LAUNCH_OK("rescore_kernel");
    return 0;
}

// ---- rescoring from a host-resident master --------------------------------------------------------------------
// With KIRAG_INDEX_HOST_MASTER the master is pinned host memory mapped at the same address on the device, and every
// row a rescoring reads crosses PCIe (~50 GB/s, microseconds of latency).  Same warp-per-(query, candidate) layout and
// skip as rescore_kernel, so each needed pair is read once and an unneeded one not at all; the difference is that a
// lane issues ALL its loads of a row (kHostBatch float4 per batch: d <= 2048 in one batch) before the first FMA, so a
// warp keeps a whole 4-KB row in flight instead of two 512-byte slices.  The FMA chain of a lane runs over
// c = lane*4 + 128*i in ascending order and the partials go through the same butterfly: bit-identical to
// canonical_partial.  The skip's norms are looked up through qmap (the second bf16 pass rescores a gathered subset of
// a chunk's queries whose norms stay in the chunk's arrays).
constexpr int kHostBatch = 16;

template <bool QVEC4>
__global__ void __launch_bounds__(256)
rescore_host_kernel(const float* __restrict__ master, int d, const float* __restrict__ q,
                    const Cand* __restrict__ cand, const int* __restrict__ cnt, int cand_stride, int m,
                    float* __restrict__ out, int64_t nq, const float* __restrict__ tauk, const int* __restrict__ qmap,
                    const float* __restrict__ qnorm, const float* __restrict__ qerr, float eps_a, float eps_b) {
    pdl_wait();
    pdl_launch_dependents();
    const int lane = threadIdx.x & 31;
    const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (warp >= nq * m) return;
    const int64_t qi = warp / m;
    const int j = (int)(warp - qi * m);
    int count = cnt ? cnt[qi] : m;
    if (count > m) count = m;
    float result = __int_as_float(0x7fc00000);  // NaN marks an empty (or skipped) slot
    if (j < count) {
        const Cand cd = cand[qi * (int64_t)cand_stride + j];
        const int32_t row = cd.id;
        bool needed = true;
        if (tauk) {
            const int64_t qn = qmap ? (int64_t)qmap[qi] : qi;
            needed = cd.s >= __ldcg(tauk + qi) - 2.0f * (eps_a * __ldcg(qnorm + qn) + eps_b * __ldcg(qerr + qn));
        }
        if (row >= 0 && needed) {
            const float* x = master + (int64_t)row * d;
            const float* qr = q + qi * (int64_t)d;
            float acc = 0.0f;
            for (int c0 = lane * 4; c0 < d; c0 += kHostBatch * 128) {
                float4 v[kHostBatch];
#pragma unroll
                for (int u = 0; u < kHostBatch; ++u)
                    if (c0 + u * 128 < d) v[u] = __ldcs(reinterpret_cast<const float4*>(x + c0 + u * 128));
#pragma unroll
                for (int u = 0; u < kHostBatch; ++u) {
                    const int c = c0 + u * 128;
                    if (c < d) {
                        float4 qv;
                        if (QVEC4) qv = *reinterpret_cast<const float4*>(qr + c);
                        else qv = make_float4(qr[c], qr[c + 1], qr[c + 2], qr[c + 3]);
                        acc = __fmaf_rn(v[u].x, qv.x, acc);
                        acc = __fmaf_rn(v[u].y, qv.y, acc);
                        acc = __fmaf_rn(v[u].z, qv.z, acc);
                        acc = __fmaf_rn(v[u].w, qv.w, acc);
                    }
                }
            }
            result = warp_butterfly_sum(acc);
        }
    }
    if (lane == 0) out[qi * (int64_t)m + j] = result;
}

int launch_rescore_host(const float* master, int d, const float* q, const Cand* cand, const int* cnt,
                        int cand_stride, int m, float* out_scores, int64_t nq, const float* tauk, const int* qmap,
                        const float* qnorm, const float* qerr, float eps_a, float eps_b, cudaStream_t st) {
    if (nq <= 0 || m <= 0) return 0;
    // rows are read as float4: d % 4 == 0 and a 16-byte aligned master (a host master always has d % 64 == 0 and a
    // page-aligned base)
    KIRAG_CHECK(d % 4 == 0 && (reinterpret_cast<uintptr_t>(master) & 15) == 0,
                "rescore_host: the master must hold 16-byte aligned rows (d=%d)", d);
    const int threads = 256;
    const int64_t warps = nq * m;
    const int64_t blocks = (warps + (threads / 32) - 1) / (threads / 32);
    KIRAG_CHECK(blocks < 0x7fffffffLL, "rescore_host: too many candidates (%lld warps)", (long long)warps);
    const bool qvec4 = (reinterpret_cast<uintptr_t>(q) & 15) == 0;
    if (qvec4)
        KIRAG_CUDA_OK(launch_chained(rescore_host_kernel<true>, dim3((unsigned)blocks), dim3(threads), 0, st, master, d, q,
                                     cand, cnt, cand_stride, m, out_scores, nq, tauk, qmap, qnorm, qerr, eps_a, eps_b));
    else
        KIRAG_CUDA_OK(launch_chained(rescore_host_kernel<false>, dim3((unsigned)blocks), dim3(threads), 0, st, master, d,
                                     q, cand, cnt, cand_stride, m, out_scores, nq, tauk, qmap, qnorm, qerr, eps_a, eps_b));
    KIRAG_LAUNCH_OK("rescore_host_kernel");
    return 0;
}

}  // namespace kirag
