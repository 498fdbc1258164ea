// ranks.cu — exact target ranks of query batches against dense float32 rows (vbq_score_ranks, vbq_pair_scores).
//
// A rank counts the rows that beat a query's target under the score and order contract of include/vbq_b200.h (the
// numerics of vbq_rans_shared_row_scores, the order of CompressedEmbedding.topk).  vbq_score_ranks is an FP32 SIMT
// contraction whose epilogue compares every score with the query's threshold and adds integer counts: it never writes
// a score, and integer atomics make the counts independent of tiling and launch order.
//
// Tiling.  A CTA of 256 threads owns 64 queries x 64 rows and streams d in chunks of 32.  The thread quad q (lanes
// 4q .. 4q+3) owns an 8 x 8 micro-tile of outputs, and lane c of the quad owns accumulator class d = c (mod 4) of all
// 64: it steps d = c, c + 4, c + 8, ... in increasing order, which is exactly the sequential chain a[d % 4] of the
// contract.  The quad then forms (a0 + a1) + (a2 + a3) with two xor shuffles, which gives every lane of the quad the
// same bits as one thread holding four accumulators.  Padding (d >= D, rows or queries past the end) is 0: an FMA with
// 0 x 0 changes at most the sign of a zero sum, and the order maps -0 and +0 to the same key.
//
// Shared memory holds the chunk transposed, [d][m] with a row stride of 72 floats (72 = 8 mod 32): a quad's four
// lanes read rows d .. d+3, so the 8 distinct float4 of a warp's query load fall in 8 different bank quads (one
// wavefront) and the 16 of its row load in two wavefronts; the loader's stores (lanes over 4 d x 8 rows) hit 32
// different banks.
#include <climits>

#include "common.h"

namespace {

constexpr int kRankTile = 64;                   // queries and rows per CTA
constexpr int kRankChunk = 32;                  // d per shared-memory chunk
constexpr int kRankStride = 72;                 // floats per shared row; 72 = 8 (mod 32)
constexpr int kRankThreads = 256;
constexpr int kPairThreads = 256;

// The order of CompressedEmbedding.topk on float32 scores: the order-preserving map of the bits, -0.0 as +0.0, NaN
// lowest.
__device__ __forceinline__ int rank_key(float s) {
    if (s != s) return INT_MIN;
    if (s == 0.f) return 0;
    const int b = __float_as_int(s);
    return b < 0 ? (b ^ 0x7FFFFFFF) : b;
}

__device__ __forceinline__ float quad_sum(float a) {           // (a0 + a1) + (a2 + a3) over the quad, on every lane
    a = __fadd_rn(a, __shfl_xor_sync(0xffffffffu, a, 1));
    return __fadd_rn(a, __shfl_xor_sync(0xffffffffu, a, 2));
}

template <bool COS>
__global__ void __launch_bounds__(kRankThreads, 2) vbq_score_ranks_kernel(
        const float *__restrict__ Z, long long n_rows, long long D, long long row0, const float *__restrict__ Qm,
        int B, long long n_qt, const float *__restrict__ thr, const long long *__restrict__ tgt,
        unsigned long long *__restrict__ counts) {
    __shared__ __align__(16) float sq[kRankChunk][kRankStride];
    __shared__ __align__(16) float sz[kRankChunk][kRankStride];
    __shared__ float s_qn[kRankTile], s_zn[kRankTile];
    __shared__ int s_kt[kRankTile], s_cnt[kRankTile];
    __shared__ long long s_t[kRankTile];

    const long long tile = blockIdx.x;
    const int q0 = (int)(tile % n_qt) * kRankTile;
    const long long r0 = (tile / n_qt) * kRankTile;              // first row of the tile, relative to Z
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, c = lane & 3, qiw = lane >> 2;
    const int qm = (warp >> 1) * 2 + (qiw >> 2);                   // the quad's micro-tile: queries 4 qm + {0..3},
    const int qn = (warp & 1) * 4 + (qiw & 3);                     // 32 + 4 qm + {0..3}; rows likewise with qn

    // loader: thread t stages row lm = t / 4 of both tiles at d = 4 i + c, i.e. exactly class c of that row in order
    const int lm = tid >> 2;
    const bool q_ok = q0 + lm < B, z_ok = r0 + lm < n_rows;
    const float *qsrc = Qm + (long long)(q_ok ? q0 + lm : 0) * D;
    const float *zsrc = Z + (z_ok ? r0 + lm : 0) * D;
    if (tid < kRankTile) {
        const int b = min(q0 + tid, B - 1);
        s_kt[tid] = rank_key(__ldg(thr + b));
        s_t[tid] = __ldg(tgt + b);
        s_cnt[tid] = 0;
    }
    float pq[kRankChunk / 4], pz[kRankChunk / 4];
#pragma unroll
    for (int i = 0; i < kRankChunk / 4; ++i) {
        const long long d = 4 * i + c;
        pq[i] = q_ok && d < D ? __ldg(qsrc + d) : 0.f;
        pz[i] = z_ok && d < D ? __ldg(zsrc + d) : 0.f;
    }
    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    float qq = 0.f, zz = 0.f;

    for (long long k0 = 0; k0 < D; k0 += kRankChunk) {
        __syncthreads();                                           // the previous chunk's reads are done
#pragma unroll
        for (int i = 0; i < kRankChunk / 4; ++i) {
            sq[4 * i + c][lm] = pq[i];
            sz[4 * i + c][lm] = pz[i];
            if (COS) {
                qq = __fmaf_rn(pq[i], pq[i], qq);
                zz = __fmaf_rn(pz[i], pz[i], zz);
            }
        }
        __syncthreads();
        if (k0 + kRankChunk < D) {                                  // the next chunk is in flight during this one
#pragma unroll
            for (int i = 0; i < kRankChunk / 4; ++i) {
                const long long d = k0 + kRankChunk + 4 * i + c;
                pq[i] = q_ok && d < D ? __ldg(qsrc + d) : 0.f;
                pz[i] = z_ok && d < D ? __ldg(zsrc + d) : 0.f;
            }
        }
#pragma unroll
        for (int s = 0; s < kRankChunk / 4; ++s) {
            const int d = 4 * s + c;
            const float4 a0 = *(const float4 *)&sq[d][4 * qm], a1 = *(const float4 *)&sq[d][32 + 4 * qm];
            const float4 b0 = *(const float4 *)&sz[d][4 * qn], b1 = *(const float4 *)&sz[d][32 + 4 * qn];
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = __fmaf_rn(b[j], a[i], acc[i][j]);
        }
    }

    if (COS) {
        const float qs = quad_sum(qq), zs = quad_sum(zz);
        if (c == 0) {
            s_qn[lm] = __fsqrt_rn(qs);
            s_zn[lm] = __fsqrt_rn(zs);
        }
    }
    __syncthreads();

    // epilogue: every lane of the quad holds the 64 sums; lane c compares the outputs of columns j = c and c + 4
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = i < 4 ? 4 * qm + i : 32 + 4 * qm + i - 4;
        const int kt = s_kt[m];
        const long long t = s_t[m];
        int cnt = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float v = quad_sum(acc[i][j]);
            if ((j & 3) == c) {
                const int n = j < 4 ? 4 * qn + j : 32 + 4 * qn + j - 4;
                if (COS) {
                    const float den = __fmul_rn(s_zn[n], s_qn[m]);
                    v = den > 0.f ? __fdiv_rn(v, den) : 0.f;
                }
                const int k = rank_key(v);
                const long long gid = row0 + r0 + n;
                cnt += (r0 + n < n_rows) && (k > kt || (k == kt && gid < t));
            }
        }
        cnt += __shfl_xor_sync(0xffffffffu, cnt, 1);
        cnt += __shfl_xor_sync(0xffffffffu, cnt, 2);
        if (c == 0 && cnt) atomicAdd(&s_cnt[m], cnt);
    }
    __syncthreads();
    if (tid < kRankTile && q0 + tid < B && s_cnt[tid])
        atomicAdd(counts + q0 + tid, (unsigned long long)s_cnt[tid]);
}

template <bool COS>
__global__ void __launch_bounds__(kPairThreads) vbq_pair_scores_kernel(
        const float *__restrict__ Z, long long n_rows, long long D, const float *__restrict__ Qm, long long B,
        const long long *__restrict__ prow, const long long *__restrict__ pqry, long long P, float *__restrict__ out) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const long long r = __ldg(prow + p), b = __ldg(pqry + p);
    if (r < 0 || r >= n_rows || b < 0 || b >= B) {
        out[p] = __int_as_float(0x7fffffff);
        return;
    }
    const float *z = Z + r * D, *q = Qm + b * D;
    float a[4] = {0.f, 0.f, 0.f, 0.f}, zz[4] = {0.f, 0.f, 0.f, 0.f}, qq[4] = {0.f, 0.f, 0.f, 0.f};
    for (long long d0 = 0; d0 < D; d0 += 4) {
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (d0 + u < D) {
                const float zv = __ldg(z + d0 + u), qv = __ldg(q + d0 + u);
                a[u] = __fmaf_rn(zv, qv, a[u]);
                if (COS) {
                    zz[u] = __fmaf_rn(zv, zv, zz[u]);
                    qq[u] = __fmaf_rn(qv, qv, qq[u]);
                }
            }
        }
    }
    float v = __fadd_rn(__fadd_rn(a[0], a[1]), __fadd_rn(a[2], a[3]));
    if (COS) {
        const float den = __fmul_rn(__fsqrt_rn(__fadd_rn(__fadd_rn(zz[0], zz[1]), __fadd_rn(zz[2], zz[3]))),
                                    __fsqrt_rn(__fadd_rn(__fadd_rn(qq[0], qq[1]), __fadd_rn(qq[2], qq[3]))));
        v = den > 0.f ? __fdiv_rn(v, den) : 0.f;
    }
    out[p] = v;
}

}  // namespace

extern "C" int vbq_score_ranks(const float *d_rows, long long n_rows, long long row_size, long long row_offset,
                               const float *d_queries, long long n_queries, int metric, const float *d_thresholds,
                               const long long *d_targets, long long *d_counts, void *stream) {
    if (n_rows < 0 || row_size < 1 || row_offset < 0 || row_offset > LLONG_MAX - n_rows || n_queries < 0 ||
        n_queries > INT_MAX - kRankTile || (metric != VBQ_SCORE_DOT && metric != VBQ_SCORE_COSINE) ||
        (n_rows > 0 && row_size > LLONG_MAX / n_rows))
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_score_ranks: n_rows=%lld row_size=%lld row_offset=%lld n_queries=%lld "
                        "metric=%d", n_rows, row_size, row_offset, n_queries, metric);
    const bool work = n_rows > 0 && n_queries > 0;
    if (work && (!d_rows || !d_queries || !d_thresholds || !d_targets || !d_counts))
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_score_ranks: null pointer");
    if (((uintptr_t)d_rows & 3) || ((uintptr_t)d_queries & 3) || ((uintptr_t)d_thresholds & 3) ||
        ((uintptr_t)d_targets & 7) || ((uintptr_t)d_counts & 7))
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_score_ranks: misaligned pointer");
    if (!work) return VBQ_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const long long n_qt = (n_queries + kRankTile - 1) / kRankTile;
    // one launch takes at most INT_MAX tiles (query tiles vary fastest, so consecutive CTAs share a row tile)
    const long long rows_per_launch = (INT_MAX / n_qt) * kRankTile;
    for (long long a = 0; a < n_rows; a += rows_per_launch) {
        const long long nr = min(rows_per_launch, n_rows - a);
        const unsigned grid = (unsigned)(n_qt * ((nr + kRankTile - 1) / kRankTile));
        if (metric == VBQ_SCORE_COSINE)
            vbq_score_ranks_kernel<true><<<grid, kRankThreads, 0, st>>>(
                d_rows + a * row_size, nr, row_size, row_offset + a, d_queries, (int)n_queries, n_qt, d_thresholds,
                d_targets, (unsigned long long *)d_counts);
        else
            vbq_score_ranks_kernel<false><<<grid, kRankThreads, 0, st>>>(
                d_rows + a * row_size, nr, row_size, row_offset + a, d_queries, (int)n_queries, n_qt, d_thresholds,
                d_targets, (unsigned long long *)d_counts);
        CUDA_TRY(cudaGetLastError());
    }
    return VBQ_OK;
}

extern "C" int vbq_pair_scores(const float *d_rows, long long n_rows, long long row_size, const float *d_queries,
                               long long n_queries, const long long *d_pair_rows, const long long *d_pair_queries,
                               long long n_pairs, int metric, float *d_scores, void *stream) {
    if (n_rows < 0 || row_size < 1 || n_queries < 0 || n_pairs < 0 ||
        n_pairs > (long long)INT_MAX * kPairThreads || (metric != VBQ_SCORE_DOT && metric != VBQ_SCORE_COSINE))
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_pair_scores: n_rows=%lld row_size=%lld n_queries=%lld n_pairs=%lld "
                        "metric=%d", n_rows, row_size, n_queries, n_pairs, metric);
    if (n_pairs > 0 && (!d_pair_rows || !d_pair_queries || !d_scores || (n_rows > 0 && !d_rows) ||
                        (n_queries > 0 && !d_queries)))
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_pair_scores: null pointer");
    if (((uintptr_t)d_rows & 3) || ((uintptr_t)d_queries & 3) || ((uintptr_t)d_pair_rows & 7) ||
        ((uintptr_t)d_pair_queries & 7) || ((uintptr_t)d_scores & 3))
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_pair_scores: misaligned pointer");
    if (n_pairs == 0) return VBQ_OK;
    cudaStream_t st = (cudaStream_t)stream;
    const unsigned grid = (unsigned)((n_pairs + kPairThreads - 1) / kPairThreads);
    if (metric == VBQ_SCORE_COSINE)
        vbq_pair_scores_kernel<true><<<grid, kPairThreads, 0, st>>>(d_rows, n_rows, row_size, d_queries, n_queries,
                                                                     d_pair_rows, d_pair_queries, n_pairs, d_scores);
    else
        vbq_pair_scores_kernel<false><<<grid, kPairThreads, 0, st>>>(d_rows, n_rows, row_size, d_queries, n_queries,
                                                                      d_pair_rows, d_pair_queries, n_pairs, d_scores);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}
