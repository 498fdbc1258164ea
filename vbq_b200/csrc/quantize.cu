// quantize.cu — the rate-distortion search kernel (sm_100a) and its C ABI.
//
// Reference behaviour reproduced (paths relative to mandt-lab/vbq):
//   img-compression/quantizer.py:65-80     per-depth bracket of mu (searchsorted in edge-padded grids)
//   img-compression/quantizer.py:156-188   candidates left_0..left_N, right_1..right_N and their code lengths
//   img-compression/utils.py:318-320       score -0.5*((z-mu)/sigma)^2, float32
//   img-compression/utils.py:392-415       per lambda: score - lambda*len, first argmax, gather
//   img-compression/quantizer.py:223-228   sorted index of z_hat and entropy-model bits
//
// Design.  The prior's quantile function tabulated on the dyadic grid is, in the reference's own heap order, an
// implicit binary search tree (node (n,i) has children (n+1,2i), (n+1,2i+1)).  Walking it with one compare per bit
// depth yields at every depth exactly the searchsorted bracket of the reference.  A CTA owns 16 channels: their
// trees (depths 0..10, each level padded by one entry on both sides so that bracket ends never need clamping) sit
// interleaved in shared memory (bank = channel + 16*(entry&1)); a warp covers 16 channels x 2 rows, so global
// accesses are full 64-byte segments of the channel-last latents.  Each thread keeps its channel's penalties in
// registers and processes U rows at a time for instruction-level parallelism, prefetching the next rows.  Only the
// winning depth is tracked; the winning index is rebuilt from the final tree path.  No tensor cores: nothing here
// is a dense contraction.
#include <stdlib.h>

#include "tree.cuh"

// ------------------------------------------------------------------------------------------------------------
// packed table: [group][entry][16 channels]; unused depths (> N) repeat the parent so the walk stays defined
// ------------------------------------------------------------------------------------------------------------
__global__ void pack_table_kernel(const float *__restrict__ table, int C, int N, int Q, int n_groups,
                                  float *__restrict__ packed) {
    const long long total = (long long)n_groups * kPadEntries * VBQ_GROUP;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
        const int j = (int)(t % VBQ_GROUP);
        const long long r = t / VBQ_GROUP;
        const int e = (int)(r % kPadEntries);
        const int g = (int)(r / kPadEntries);
        const int c = min(g * VBQ_GROUP + j, C - 1);
        // level of padded entry e: largest n with entry_of(n, -1) <= e
        int n = 0;
        while (n + 1 < VBQ_SMEM_LEVELS && entry_of(n + 1, -1) <= e) ++n;
        const int k = e - entry_of(n, -1);          // 0 = left pad, 1..2^n = points, 2^n+1 = right pad
        const int last = (1 << n) - 1;
        int i = min(max(k - 1, 0), last);
        // depth N has no edge padding in the reference (quantizer.py:57): above the highest point the bracket is
        // (second highest, highest), so the right pad of depth N holds the second-highest point
        if (n == N && k == last + 2) i = max(last - 1, 0);
        int nn = n;
        while (nn > N) {  // unused depth: repeat the ancestor at depth N
            --nn;
            i >>= 1;
        }
        packed[t] = table[(size_t)c * Q + ((1 << nn) - 1 + i)];
    }
}


// ------------------------------------------------------------------------------------------------------------
// walk tree of vbq_bisect_tma_kernel (quantize_tma.cu): per group [2048][16] floats in heap order (row K = node K,
// children 2K and 2K+1, row 0 unused) followed by [257][2][16]: rows K <= 256 again, twice (one copy per half-warp);
// every value scaled by 2^24; unused depths (> N) repeat the ancestor at depth N
// ------------------------------------------------------------------------------------------------------------
__global__ void pack_walk_tree_kernel(const float *__restrict__ table, int C, int N, int Q, int n_groups,
                                      float *__restrict__ walk) {
    const int per_group = (int)(vbq_walk_tree_floats(1));
    const int single = (1 << VBQ_SMEM_LEVELS) * VBQ_GROUP;
    const long long total = (long long)n_groups * per_group;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
        const int g = (int)(t / per_group);
        const int o = (int)(t - (long long)g * per_group);
        const int j = o % VBQ_GROUP;
        int K = o < single ? o / VBQ_GROUP : (o - single) / (2 * VBQ_GROUP);
        float v = 0.0f;
        if (K >= 1) {
            int n = 31 - __clz(K);
            while (n > N) {
                --n;
                K >>= 1;
            }
            const int c = min(g * VBQ_GROUP + j, C - 1);
            v = table[(size_t)c * Q + (K - 1)] * 16777216.0f;
        }
        walk[t] = v;
    }
}

__global__ void selftest_divide_kernel(const float *__restrict__ x, const float *__restrict__ y, long long n,
                                       float *__restrict__ out) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride)
        out[t] = div_rn(x[t], y[t], rcp_rn(y[t]));
}

__global__ void selftest_sigma_kernel(const float *__restrict__ lv, long long n, float *__restrict__ out) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += stride) out[t] = sigma_of_logvar(lv[t]);
}

// ------------------------------------------------------------------------------------------------------------
// C ABI
// ------------------------------------------------------------------------------------------------------------
extern "C" long long vbq_packed_table_floats(int C, int N) {
    if (C < 1 || N < 0 || N > VBQ_MAX_DEPTH) return -1;
    const long long groups = (C + VBQ_GROUP - 1) / VBQ_GROUP;
    return groups * kPadEntries * VBQ_GROUP + vbq_walk_tree_floats((int)groups);
}

extern "C" int vbq_pack_code_points(const float *d_table, int C, int N, float *d_packed, void *stream) {
    if (!d_table || !d_packed) return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_pack_code_points: null pointer");
    if (C < 1) return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_pack_code_points: C=%d", C);
    RETURN_IF(vbq_check_depth(N));
    if (((uintptr_t)d_packed & 15) != 0)
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_pack_code_points: d_packed not 16-byte aligned");
    const int Q = (1 << (N + 1)) - 1;
    const int groups = (C + VBQ_GROUP - 1) / VBQ_GROUP;
    int grid;
    RETURN_IF(vbq_grid_for((long long)groups * kPadEntries * VBQ_GROUP, 256, &grid));
    pack_table_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_table, C, N, Q, groups, d_packed);
    CUDA_TRY(cudaGetLastError());
    RETURN_IF(vbq_grid_for(vbq_walk_tree_floats(groups), 256, &grid));
    pack_walk_tree_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_table, C, N, Q, groups,
                                                                 d_packed + (size_t)groups * kPadEntries * VBQ_GROUP);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

extern "C" long long vbq_quantize_workspace_bytes(int n_lambda) {
    if (n_lambda < 1) return -1;
    return (long long)ticket_bytes(n_lambda) + (long long)n_lambda * kMaxGrid * VBQ_TOTALS * (long long)sizeof(double);
}

extern "C" int vbq_quantize(const float *d_mu, const float *d_sigma, long long rows, int C, const float *d_table,
                            const float *d_packed, int N, const float *d_penalty, const float *d_length, int n_lambda,
                            int pen_channels, const float *d_entropy_model, float *d_zhat, int *d_qidx, int *d_level,
                            float *d_bits, float *d_em_bits, double *d_totals, void *d_workspace,
                            long long workspace_bytes, unsigned flags, void *stream) {
    return vbq_quantize_hp(d_mu, d_sigma, rows, C, d_table, d_packed, N, d_penalty, nullptr, d_length, n_lambda,
                           pen_channels, d_entropy_model, d_zhat, d_qidx, d_level, d_bits, d_em_bits, d_totals,
                           d_workspace, workspace_bytes, flags, stream);
}

extern "C" int vbq_quantize_hp(const float *d_mu, const float *d_sigma, long long rows, int C, const float *d_table,
                               const float *d_packed, int N, const float *d_penalty, const float *h_penalty,
                               const float *d_length, int n_lambda, int pen_channels, const float *d_entropy_model,
                               float *d_zhat, int *d_qidx, int *d_level, float *d_bits, float *d_em_bits,
                               double *d_totals, void *d_workspace, long long workspace_bytes, unsigned flags,
                               void *stream) {
    return vbq_quantize_impl(d_mu, d_sigma, rows, C, d_table, d_packed, N, d_penalty, h_penalty, d_length, n_lambda,
                             pen_channels, d_entropy_model, d_zhat, d_qidx, d_level, d_bits, d_em_bits, d_totals,
                             d_workspace, workspace_bytes, flags, stream, nullptr);
}

// `push` (optional): where the last CTA of the search kernel also delivers this call's totals (peer.cu).  *push_fused
// tells the caller whether a kernel did; otherwise the caller sends them with a kernel of its own.
int vbq_quantize_impl(const float *d_mu, const float *d_sigma, long long rows, int C, const float *d_table,
                      const float *d_packed, int N, const float *d_penalty, const float *h_penalty,
                      const float *d_length, int n_lambda, int pen_channels, const float *d_entropy_model,
                      float *d_zhat, int *d_qidx, int *d_level, float *d_bits, float *d_em_bits,
                      double *d_totals, void *d_workspace, long long workspace_bytes, unsigned flags,
                      void *stream, PeerPush *push) {
    if (rows < 0 || C < 1 || n_lambda < 1 || n_lambda > 65535 || (pen_channels != 1 && pen_channels != C))
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_quantize: rows=%lld C=%d n_lambda=%d pen_channels=%d", rows, C,
                        n_lambda, pen_channels);
    RETURN_IF(vbq_check_depth(N));
    if (flags & ~(VBQ_FLAG_LOGVAR | VBQ_FLAG_NO_PRUNE | VBQ_FLAG_FAST | VBQ_FLAG_ACCUMULATE_TOTALS | VBQ_FLAG_NO_SWEEP |
                  VBQ_FLAG_REFERENCE_WALK | VBQ_FLAG_RESERVE_SM | VBQ_FLAG_BRACKET_WALK | VBQ_FLAG_WORKSPACE_ZEROED |
                  VBQ_FLAG_NO_TMA | VBQ_FLAG_TABLE_STABLE | VBQ_FLAG_NEIGHBOUR_EVERY_DEPTH))
        return vbq_fail(VBQ_ERR_BAD_FLAGS, "vbq_quantize: unknown flag bits 0x%x", flags);
    if (!d_table || !d_packed || !d_penalty || (rows > 0 && (!d_mu || !d_sigma)))
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_quantize: null input pointer");
    if (d_em_bits && !d_entropy_model)
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_quantize: d_em_bits requested without d_entropy_model");
    if (((uintptr_t)d_packed & 15) != 0)
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_quantize: d_packed not 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;

    QArgs a;
    a.mu = d_mu; a.sigma = d_sigma; a.rows = rows; a.C = C;
    a.table = d_table; a.packed = d_packed;
    a.N = N; a.Q = (1 << (N + 1)) - 1;
    a.pen = d_penalty; a.h_pen = h_penalty; a.len = d_length; a.n_lambda = n_lambda; a.pen_channels = pen_channels;
    a.em = d_entropy_model;
    a.zhat = d_zhat; a.qidx = d_qidx; a.level = d_level; a.bits = d_bits; a.em_bits = d_em_bits;
    a.totals = d_totals; a.partials = nullptr; a.ticket = nullptr; a.queue = nullptr;
    a.peer_inbox = nullptr; a.peer_src = nullptr; a.peer_world = 0; a.peer_off = 0; a.peer_flag = 0; a.peer_seq = 0;
    a.peer_own = nullptr; a.peer_coff = 0; a.peer_entry = 0; a.peer_cseq = 0; a.peer_cout = nullptr;
    if (push) push->fused = false;
    a.flags = flags;
    a.kout = 0;
    a.one = 1;
    a.two = 2;
    a.keymask = 0xfffffff0u;
    a.outm = (d_zhat ? 1u : 0u) | (d_qidx ? 2u : 0u) | (d_level ? 4u : 0u) | (d_bits ? 8u : 0u) |
             (d_em_bits ? 16u : 0u) | (d_entropy_model ? 32u : 0u) | (d_length ? 64u : 0u);
    a.n_groups = (C + VBQ_GROUP - 1) / VBQ_GROUP;

    if (d_totals) {
        const long long need = vbq_quantize_workspace_bytes(n_lambda);
        if (!d_workspace || workspace_bytes < need)
            return vbq_fail(VBQ_ERR_WORKSPACE, "vbq_quantize: totals need a %lld-byte workspace (got %lld)", need,
                            workspace_bytes);
        if (((uintptr_t)d_workspace & 255) != 0)
            return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_quantize: workspace not 256-byte aligned");
        a.ticket = (unsigned *)d_workspace;
        a.partials = (double *)((char *)d_workspace + ticket_bytes(n_lambda));
        // one lambda: the rest of the first 256-byte block holds the tile queues of vbq_bisect_tma_kernel (zero between calls)
        if (n_lambda == 1 && a.n_groups <= 62) a.queue = a.ticket + 1;
        if (!(flags & VBQ_FLAG_WORKSPACE_ZEROED)) CUDA_TRY(cudaMemsetAsync(a.ticket, 0, ticket_bytes(n_lambda), st));
    }
    if (rows == 0) {
        if (d_totals) CUDA_TRY(cudaMemsetAsync(d_totals, 0, (size_t)n_lambda * VBQ_TOTALS * sizeof(double), st));
        return VBQ_OK;
    }

    int dev = 0, sms = 0;
    RETURN_IF(vbq_current_device(&dev, &sms));
    if ((flags & VBQ_FLAG_RESERVE_SM) && sms > 1) --sms;
    // the kernel addresses a channel-last array with 32-bit BYTE offsets: split calls beyond 2^29 elements into row chunks
    const long long max_chunk_rows = ((1ll << 29) - 1) / C > 1024 ? (((1ll << 29) - 1) / C) & ~1023ll : ((1ll << 29) - 1) / C;
    a.lam_stride = rows * (long long)C;
    for (long long r0 = 0; r0 < rows; r0 += max_chunk_rows) {
        const long long nr = rows - r0 < max_chunk_rows ? rows - r0 : max_chunk_rows;
        const size_t eo = (size_t)r0 * C;
        QArgs b = a;
        b.rows = nr;
        b.mu = d_mu + eo;
        b.sigma = d_sigma + eo;
        if (d_zhat) b.zhat = d_zhat + eo;
        if (d_qidx) b.qidx = d_qidx + eo;
        if (d_level) b.level = d_level + eo;
        if (d_bits) b.bits = d_bits + eo;
        if (d_em_bits) b.em_bits = d_em_bits + eo;
        b.accumulate = r0 > 0 || (flags & VBQ_FLAG_ACCUMULATE_TOTALS);
        // one lambda, one chunk: the last CTA of the TMA kernels can deliver the totals to the peers itself
        const bool can_fuse = push && n_lambda == 1 && rows <= max_chunk_rows && !b.accumulate;
        if (can_fuse) {
            b.peer_inbox = push->inbox; b.peer_world = push->world; b.peer_off = push->off; b.peer_flag = push->flag;
            b.peer_seq = push->seq; b.peer_src = push->src;
            b.peer_own = push->own; b.peer_coff = push->coff; b.peer_entry = push->entry; b.peer_cseq = push->cseq;
            b.peer_cout = push->cout;
        }
        int st_;
        if (!(flags & VBQ_FLAG_NO_SWEEP)) {   // several lambdas: one walk per coordinate serves all of them
            st_ = vbq_launch_sweep_bisect(b, dev, sms, st);
            // where the both-ends sweep does not apply (C % 4, unaligned arrays, no host copy of the penalties): with
            // per-coordinate outputs one launch of the both-ends TMA kernel per lambda is faster than the bracket-walk sweep
            // (measured, 16 lambdas on the Kodak batch: 1.40 vs 1.97 ms with the entropy-model bits, 0.91 vs 1.16 ms
            // without); totals-only sweeps go to the bracket-walk sweep (0.77 vs 0.87 ms)
            // arbitrary penalties, several lambdas: the both-ends sweep (one walk for all lambdas)
            if (st_ < 0 && !getenv("VBQ_NO_SWEEP_BOTH")) st_ = vbq_launch_sweep_both(b, dev, sms, st);
            if (st_ < 0 && n_lambda > 1 && (b.outm & 15u) &&
                !(flags & (VBQ_FLAG_BRACKET_WALK | VBQ_FLAG_NO_TMA | VBQ_FLAG_FAST | VBQ_FLAG_REFERENCE_WALK)))
                st_ = vbq_launch_quantize_tma_both(b, dev, sms, st);
            if (st_ < 0) st_ = vbq_launch_sweep(b, dev, sms, st);
            if (st_ >= 0) {
                RETURN_IF(st_);
                continue;
            }
        }
        if (flags & VBQ_FLAG_FAST) st_ = vbq_launch_quantize_fast(b, dev, sms, st);
        else if (flags & VBQ_FLAG_REFERENCE_WALK) st_ = vbq_launch_quantize_reference(b, dev, sms, st);
        else {
            // default: certified bisection (raw code lengths, N <= 10); otherwise the bracket walk in strict mode
            st_ = (flags & (VBQ_FLAG_BRACKET_WALK | VBQ_FLAG_NO_TMA)) ? -1 : vbq_launch_quantize_tma(b, dev, sms, st);
            if (st_ >= 0 && can_fuse) push->fused = true;
            if (st_ < 0) st_ = (flags & VBQ_FLAG_BRACKET_WALK) ? -1 : vbq_launch_quantize_bisect(b, dev, sms, st);
            if (st_ < 0) {
                st_ = (flags & (VBQ_FLAG_BRACKET_WALK | VBQ_FLAG_NO_TMA)) ? -1 : vbq_launch_quantize_tma_both(b, dev, sms, st);
                if (st_ >= 0 && can_fuse) push->fused = true;
            }
            if (st_ < 0) st_ = vbq_launch_quantize_strict(b, dev, sms, st);
        }
        RETURN_IF(st_);
    }
    return VBQ_OK;
}

extern "C" int vbq_selftest_divide(const float *d_a, const float *d_b, long long n, float *d_out, void *stream) {
    if (n > 0 && (!d_a || !d_b || !d_out)) return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_selftest_divide: null pointer");
    if (n < 0) return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_selftest_divide: n=%lld", n);
    if (n == 0) return VBQ_OK;
    int grid;
    RETURN_IF(vbq_grid_for(n, 256, &grid));
    selftest_divide_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_a, d_b, n, d_out);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

extern "C" int vbq_selftest_sigma_from_logvar(const float *d_lv, long long n, float *d_out, void *stream) {
    if (n > 0 && (!d_lv || !d_out)) return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_selftest_sigma_from_logvar: null pointer");
    if (n < 0) return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_selftest_sigma_from_logvar: n=%lld", n);
    if (n == 0) return VBQ_OK;
    int grid;
    RETURN_IF(vbq_grid_for(n, 256, &grid));
    selftest_sigma_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_lv, n, d_out);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}
