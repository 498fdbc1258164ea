// quantize_kernel.cuh — the single-lambda rate-distortion search kernel template and its launch dispatch.
// Included by one translation unit per scoring mode (quantize_strict.cu, quantize_reference.cu, quantize_fast.cu) so
// that nvcc can compile the modes in parallel.  See quantize.cu for the design notes.
#pragma once
#include <stdlib.h>

#include "tree.cuh"

// Scoring modes.  All three produce the reference's result; they differ in how much work proves it.
//   kModeReference: both bracket ends of every depth are scored with the reference's float32 roundings and two
//                   running maxima (left / right candidates) reproduce argmax's first-maximum order directly.
//   kModeStrict   : (default) only the NEARER end of every depth is scored (same roundings; the farther end can never
//                   score higher), one running maximum; the left/right decision is made exactly for the winning depth
//                   in the epilogue, and whenever two depths reach exactly the same float32 score (the only situation
//                   in which the candidate order matters) the coordinate is re-done by `reference_walk`.
//                   Bit-identical to kModeReference by construction and by test.
//   kModeFast     : nearer end, d*d*(0.5/sigma^2) instead of the division; may differ inside float32 rounding ties.
constexpr int kModeReference = 0, kModeStrict = 1, kModeFast = 2;

// Fully faithful scalar walk of one coordinate (the slow path of kModeStrict): returns the winning depth and side.
static __device__ __noinline__ int reference_walk(const char *pb, const float *sPenc, float z0, float mu, float sg, int NS) {
    const float rs = rcp_rn(sg);
    float bestL = score_exact(z0, mu, sg, rs, sPenc[0]), bestR = -CUDART_INF_F;
    int nL = 0, nR = 0;
    int V = mu > z0 ? 96 : 32;
    for (int n = 1; n <= NS; ++n) {
        const int imm = entry_of(n, 0) * kRowStrideBytes;
        const char *pa = pb + V;
        const float zp = lds_f32(pa, imm);
        const int s = mu > zp ? 32 : -32;
        const float zn = lds_f32(pa + 2 * s, imm);
        V = 2 * V + s;
        const float npn = sPenc[n * VBQ_GROUP];
        const float sl = score_exact(fminf(zp, zn), mu, sg, rs, npn);
        const float sr = score_exact(fmaxf(zp, zn), mu, sg, rs, npn);
        if (sl > bestL) { bestL = sl; nL = n; }
        if (sr > bestR) { bestR = sr; nR = n; }
    }
    return bestR > bestL ? (nR | 0x100) : nL;
}

// NT > 0: max_bits_per_coord == NT is known at compile time (no per-depth bound checks); NT == 0: runtime depth.
// EXTRAS: a code-length table (corrected lengths) and/or an entropy model is present; without them the code length
// of depth n is n itself and the epilogue has neither table lookups nor their totals.
template <int MODE, bool PRUNE, bool TOTALS, bool DEEP, bool EXTRAS, int NT, int U, int kThreads>
__global__ void __launch_bounds__(kThreads, 1) vbq_quantize_kernel(const QArgs a) {
    constexpr bool FAST = MODE == kModeFast;
    constexpr bool STRICT = MODE == kModeStrict;
    static_assert(!(STRICT && DEEP), "depths beyond shared memory use the reference walk");
    static_assert(U % 2 == 0, "coordinates are processed in f32x2 pairs");
    constexpr int RP = kThreads / VBQ_GROUP;              // rows covered by one pass of the CTA
    constexpr int P = U / 2;                              // coordinate pairs per thread
    extern __shared__ __align__(16) float smem[];
    float *sT = smem;                                   // [kPadEntries][16] code points of depths 0..10
    float *sPen = sT + kPadEntries * VBQ_GROUP;         // [N+1][16] negated penalties
    float *sSuf = sPen + (a.N + 1) * VBQ_GROUP;         // [N+1][16] max over deeper levels of the negated penalty
    float *sLen = sSuf + (a.N + 1) * VBQ_GROUP;         // [N+1][16] code lengths
    float *sStage = sLen + (a.N + 1) * VBQ_GROUP;       // [kStages][2][U][kThreads] thread-private staging ring
    float *myStage = sStage + threadIdx.x;
    __shared__ double sRed[VBQ_TOTALS][kMaxThreads / 32];
    __shared__ bool sLast;

    const int N = NT > 0 ? NT : a.N;
    const int NS = min(N, kSmemDepth);                  // depths walked in shared memory
    const int lam = blockIdx.y;
    // bit k set: zhat, qidx, level, bits, em_bits requested; 32: entropy model; 64: length table
    const unsigned outm = EXTRAS ? a.outm : (a.outm & 15u);
    const int col = threadIdx.x & (VBQ_GROUP - 1);
    const int rsub = threadIdx.x >> 4;
    const bool logvar = (a.flags & VBQ_FLAG_LOGVAR) != 0;
    const long long u0 = a.total_units * blockIdx.x / gridDim.x;
    const long long u1 = a.total_units * (blockIdx.x + 1) / gridDim.x;
    const int C = a.C;
    const int rows = (int)a.rows;                       // the host splits calls so that rows*C < 2^31
    const size_t lam_off = (size_t)lam * (size_t)a.lam_stride;
    // byte address of tree entry (n, i) of this thread's channel = pb + V + entry_of(n,0)*64, V = 64*i + 32
    const char *pb = reinterpret_cast<const char *>(sT) + col * 4 - 32;
    const int pbi = (int)__cvta_generic_to_shared(pb);   // the same base as a 32-bit shared-memory address
    const int one = a.one, two = a.two;
    const float *sTc = sT + col;
    const float *sLenc = sLen + col;

    double acc_len = 0.0, acc_em = 0.0, acc_dist = 0.0;
    int acc_level = 0;   // < 2^31: at most 2^31/C rows per launch, depth <= 20

    long long unit = u0;
    while (unit < u1) {
        // ---- segment: a run of row passes inside one 16-channel group --------------------------------------
        const int g = (int)(unit / a.passes);
        const int p0 = (int)(unit - (long long)g * a.passes);
        const int p1 = (int)min(a.passes, (long long)p0 + (u1 - unit));
        unit += p1 - p0;

        __syncthreads();
        {
            const float4 *src = reinterpret_cast<const float4 *>(a.packed + (size_t)g * kPadEntries * VBQ_GROUP);
            float4 *dst = reinterpret_cast<float4 *>(sT);
            for (int k = threadIdx.x; k < kPadEntries * (VBQ_GROUP / 4); k += kThreads) dst[k] = __ldg(src + k);
            if (threadIdx.x < VBQ_GROUP) {
                const int j = threadIdx.x;
                const int cj = min(g * VBQ_GROUP + j, C - 1);
                const size_t po = ((size_t)lam * a.pen_channels + (a.pen_channels == 1 ? 0 : cj)) * (N + 1);
                float suf = -CUDART_INF_F;
                for (int n = N; n >= 0; --n) {
                    const float np_ = -a.pen[po + n];
                    sPen[n * VBQ_GROUP + j] = np_;
                    sSuf[n * VBQ_GROUP + j] = suf;
                    suf = fmaxf(suf, np_);
                    sLen[n * VBQ_GROUP + j] = a.len ? a.len[po + n] : (float)n;
                }
            }
        }
        __syncthreads();

        const int c = g * VBQ_GROUP + col;
        const bool c_ok = c < C;
        const int cc = min(c, C - 1);
        const float *gT = a.table + (size_t)cc * a.Q;
        const float *gEm = a.em ? a.em + ((size_t)lam * C + cc) * a.Q : nullptr;
        // the channel-last arrays are addressed as (uniform base pointer) + (32-bit byte offset): the host splits
        // calls so that rows*C < 2^29 elements
        const char *mu_b = reinterpret_cast<const char *>(a.mu);
        const char *sg_b = reinterpret_cast<const char *>(a.sigma);
        float *zhat_c = a.zhat ? a.zhat + lam_off : nullptr;     // `off` below already contains the channel
        int *qidx_c = a.qidx ? a.qidx + lam_off : nullptr;
        int *level_c = a.level ? a.level + lam_off : nullptr;
        float *bits_c = a.bits ? a.bits + lam_off : nullptr;
        float *emb_c = a.em_bits ? a.em_bits + lam_off : nullptr;
        // this thread's channel is fixed for the segment: the penalties of the shared-memory depths live in
        // registers (duplicated into f32x2 pairs); depths beyond N get -inf and can never be selected
        float2 npen2[kSmemDepth + 1];
        float thr[kSmemDepth + 1];
#pragma unroll
        for (int n = 0; n <= kSmemDepth; ++n) {
            const float v = n <= N ? sPen[n * VBQ_GROUP + col] : -CUDART_INF_F;
            npen2[n] = make_float2(v, v);
            thr[n] = n <= N ? sSuf[n * VBQ_GROUP + col] : -CUDART_INF_F;
        }
        const float z0 = sTc[entry_of(0, 0) * VBQ_GROUP];

        const int row_end = c_ok ? min(p1 * RP, rows) : 0;   // threads of channels >= C never pass the row test
        int row = p0 * RP + rsub;
        unsigned off = (unsigned)row * (unsigned)C + (unsigned)cc;     // element offset of (row, channel)
        const unsigned off_step = (unsigned)(RP * C);

        // stage kStages-1 iterations ahead; every iteration commits exactly one group (possibly empty)
        auto stage_rows = [&](int it_row, unsigned it_off, int slot) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (it_row + u * RP < row_end) {
                    const unsigned bo = (it_off + u * off_step) * 4u;
                    cp_async_f32(myStage + ((slot * 2 + 0) * U + u) * kThreads,
                                 reinterpret_cast<const float *>(mu_b + bo));
                    cp_async_f32(myStage + ((slot * 2 + 1) * U + u) * kThreads,
                                 reinterpret_cast<const float *>(sg_b + bo));
                }
            }
            cp_async_commit();
        };
#pragma unroll
        for (int k = 0; k < kStages - 1; ++k) stage_rows(row + k * U * RP, off + k * U * off_step, k);
        int slot = 0;

        for (; row - rsub < p1 * RP; row += U * RP, off += U * off_step) {
            float mu[U], sg[U];
            float2 nmu2[P], nsg2[P], rs2[P];   // rs2 = 1/sigma (exact mode) or -0.5/sigma^2 (fast mode)
            cp_async_wait<kStages - 2>();        // this iteration's rows have landed
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const bool ok = row + u * RP < row_end;
                mu[u] = ok ? myStage[((slot * 2 + 0) * U + u) * kThreads] : 0.0f;
                float s = ok ? myStage[((slot * 2 + 1) * U + u) * kThreads] : 1.0f;
                if (logvar) s = sigma_of_logvar(s);
                sg[u] = s;
            }
            {   // refill the slot consumed in the previous iteration
                const int ps = slot == 0 ? kStages - 1 : slot - 1;
                stage_rows(row + (kStages - 1) * U * RP, off + (kStages - 1) * U * off_step, ps);
                slot = slot == kStages - 1 ? 0 : slot + 1;
            }
#pragma unroll
            for (int k = 0; k < P; ++k) {
                const float r0 = rcp_rn(sg[2 * k]), r1 = rcp_rn(sg[2 * k + 1]);
                nmu2[k] = make_float2(-mu[2 * k], -mu[2 * k + 1]);
                nsg2[k] = make_float2(-sg[2 * k], -sg[2 * k + 1]);
                rs2[k] = FAST ? make_float2(-0.5f * r0 * r0, -0.5f * r1 * r1) : make_float2(r0, r1);
            }

            // ---- depth 0: the median is the only candidate (left_0; quantizer.py:182-183) ---------------
            float bestL[U], bestR[U];
            int nL[U], nR[U], V[U];   // V = 64*path_index + 32 (byte offset of the path node inside its level)
#pragma unroll
            for (int k = 0; k < P; ++k) {
                const float2 z02 = make_float2(z0, z0);
                const float2 s0 = FAST ? score_fast2(z02, z02, nmu2[k], rs2[k], npen2[0])
                                       : score_exact2(z02, nmu2[k], nsg2[k], rs2[k], npen2[0]);
                bestL[2 * k] = s0.x;
                bestL[2 * k + 1] = s0.y;
            }
#pragma unroll
            for (int u = 0; u < U; ++u) {
                bestR[u] = -CUDART_INF_F;
                nL[u] = 0;
                nR[u] = 0;
                V[u] = mu[u] > z0 ? 96 : 32;
            }
            bool tie[U];   // kModeStrict: two depths reached exactly the same score
#pragma unroll
            for (int u = 0; u < U; ++u) tie[u] = false;
            int m_done = 0;   // deepest level processed (warp-uniform)

            // ---- depths 1..10 in shared memory, fully unrolled ------------------------------------------
#pragma unroll
            for (int n = 1; n <= kSmemDepth; ++n) {
                if (NT == 0 && n > NS) break;
                if (NT > 0 && n > NT) break;
                if (PRUNE && n % 3 == 0) {   // sound early exit: every deeper score is <= -penalty < best
                    bool done = true;
#pragma unroll
                    for (int u = 0; u < U; ++u) done = done && (fmaxf(bestL[u], bestR[u]) > thr[n - 1]);
                    if (__all_sync(0xffffffffu, done)) break;
                }
                const int imm = entry_of(n, 0) * kRowStrideBytes;
                float zp[U], zn[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    // integer multiply-adds with runtime factors 1 and 2: IMAD on the FMA pipe, not IADD3 on the ALU pipe
                    const int pa = imad(V[u], one, pbi);
                    zp[u] = lds_u32((unsigned)(pa + imm));
                    const int s = mu[u] > zp[u] ? 32 : -32;
                    zn[u] = lds_u32((unsigned)(imad(s, two, pa) + imm));   // the other bracket end (pads at the edges)
                    V[u] = imad(V[u], two, s);
                }
#pragma unroll
                for (int k = 0; k < P; ++k) {
                    const int u = 2 * k, v = 2 * k + 1;
                    if (FAST) {
                        const float2 s = score_fast2(make_float2(zp[u], zp[v]), make_float2(zn[u], zn[v]), nmu2[k],
                                                     rs2[k], npen2[n]);
                        if (s.x > bestL[u]) { bestL[u] = s.x; nL[u] = n; }
                        if (s.y > bestL[v]) { bestL[v] = s.y; nL[v] = n; }
                    } else if (STRICT) {
                        // |fl(z-mu)| of the nearer end, then the reference's roundings on it (sign-symmetric)
                        const float2 dp = __fadd2_rn(make_float2(zp[u], zp[v]), nmu2[k]);
                        const float2 dn = __fadd2_rn(make_float2(zn[u], zn[v]), nmu2[k]);
                        const float2 d = make_float2(fminf(fabsf(dp.x), fabsf(dn.x)), fminf(fabsf(dp.y), fabsf(dn.y)));
                        const float2 q0 = __fmul2_rn(d, rs2[k]);
                        const float2 e = __ffma2_rn(q0, nsg2[k], d);
                        const float2 q = __ffma2_rn(e, rs2[k], q0);
                        const float2 s = __ffma2_rn(__fmul2_rn(q, q), make_float2(-0.5f, -0.5f), npen2[n]);
                        tie[u] = tie[u] || (s.x == bestL[u]);
                        tie[v] = tie[v] || (s.y == bestL[v]);
                        if (s.x > bestL[u]) { bestL[u] = s.x; nL[u] = n; }
                        if (s.y > bestL[v]) { bestL[v] = s.y; nL[v] = n; }
                    } else {
                        // roles by value: the lower of (path, neighbour) is the left bracket end
                        const float2 zl = make_float2(fminf(zp[u], zn[u]), fminf(zp[v], zn[v]));
                        const float2 zr = make_float2(fmaxf(zp[u], zn[u]), fmaxf(zp[v], zn[v]));
                        const float2 sl = score_exact2(zl, nmu2[k], nsg2[k], rs2[k], npen2[n]);
                        const float2 sr = score_exact2(zr, nmu2[k], nsg2[k], rs2[k], npen2[n]);
                        if (sl.x > bestL[u]) { bestL[u] = sl.x; nL[u] = n; }
                        if (sl.y > bestL[v]) { bestL[v] = sl.y; nL[v] = n; }
                        if (sr.x > bestR[u]) { bestR[u] = sr.x; nR[u] = n; }
                        if (sr.y > bestR[v]) { bestR[v] = sr.y; nR[v] = n; }
                    }
                }
                m_done = n;
            }

            // ---- depths 11..N from the heap-order table in global memory (max_bits_per_coord > 10) --------
            int idx[U];
#pragma unroll
            for (int u = 0; u < U; ++u) idx[u] = V[u] >> 6;   // path index at depth m_done + 1
            if (DEEP && m_done == kSmemDepth) {
                for (int n = kSmemDepth + 1; n <= N; ++n) {
                    if (PRUNE) {
                        bool done = true;
                        const float th = sSuf[(n - 1) * VBQ_GROUP + col];
#pragma unroll
                        for (int u = 0; u < U; ++u) done = done && (fmaxf(bestL[u], bestR[u]) > th);
                        if (__all_sync(0xffffffffu, done)) break;
                    }
                    const int base = (1 << n) - 1;
                    const float npn = sPen[n * VBQ_GROUP + col];
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int ip = idx[u];
                        const float zp = __ldg(gT + base + ip);
                        const bool b = mu[u] > zp;
                        const int fg = ip + (b ? 1 : 0);
                        const int il = clamp_index(fg, n, N, false), ir = clamp_index(fg, n, N, true);
                        const float zl = il == ip ? zp : __ldg(gT + base + il);
                        const float zr = ir == ip ? zp : __ldg(gT + base + ir);
                        if (FAST) {
                            const float d = fminf(fabsf(zl - mu[u]), fabsf(zr - mu[u]));
                            const float w = u & 1 ? rs2[u / 2].y : rs2[u / 2].x;
                            const float s = __fmaf_rn(d * d, w, npn);
                            if (s > bestL[u]) { bestL[u] = s; nL[u] = n; }
                        } else {
                            const float r = u & 1 ? rs2[u / 2].y : rs2[u / 2].x;
                            const float sl = score_exact(zl, mu[u], sg[u], r, npn);
                            const float sr = score_exact(zr, mu[u], sg[u], r, npn);
                            if (sl > bestL[u]) { bestL[u] = sl; nL[u] = n; }
                            if (sr > bestR[u]) { bestR[u] = sr; nR[u] = n; }
                        }
                        idx[u] = 2 * ip + (b ? 1 : 0);
                    }
                    m_done = n;
                }
            }

            // ---- winner: first maximum in candidate order left_0..left_N, right_1..right_N (utils.py:401) ---
            // Only the winning depth was tracked; its bracket is rebuilt from the final tree path (idx is the path
            // index at depth m_done + 1), branch-free.
#pragma unroll
            for (int u = 0; u < U; ++u) {
                bool use_r = MODE == kModeReference && (bestR[u] > bestL[u]);
                int n = use_r ? nR[u] : nL[u];
                if (STRICT && tie[u]) {   // rare: the candidate order matters; redo this coordinate faithfully
                    const int r = reference_walk(pb, sPen + col, z0, mu[u], sg[u], NS);
                    n = r & 0xff;
                    use_r = (r & 0x100) != 0;
                }
                const int sh = m_done + 1 - n;
                const int ipn = idx[u] >> sh;                       // path node at depth n
                const int d = ((idx[u] >> (sh - 1)) & 1) ? 1 : -1;  // side of the other bracket end
                float zp, zn;
                if (!DEEP || n <= kSmemDepth) {
                    const float *e = sTc + (entry_of(n, 0) + ipn) * VBQ_GROUP;
                    zp = e[0];
                    zn = e[d * VBQ_GROUP];                          // pads make this valid at the edges
                } else {
                    const int last = (1 << n) - 1;
                    int inb = min(max(ipn + d, 0), last);
                    if (n == N && ipn + d > last) inb = max(last - 1, 0);
                    zp = __ldg(gT + last + ipn);
                    zn = __ldg(gT + last + inb);
                }
                bool path_wins;
                if (FAST) {   // nearer end; the left (lower) one when equidistant
                    const float dp = fabsf(zp - mu[u]), dn = fabsf(zn - mu[u]);
                    path_wins = dp < dn || (dp == dn && zp <= zn);
                } else {
                    if (STRICT && !tie[u]) {
                        // The winning depth is unique and bestL is the exact score of its nearer end.  The right end
                        // wins only with a strictly higher score than the left end (argmax order), so only the score
                        // of the FARTHER end is still needed: right wins iff the nearer end is the right one and the
                        // left (farther) end scores strictly less.
                        const float rs1 = u & 1 ? rs2[u / 2].y : rs2[u / 2].x;
                        const float zlo = fminf(zp, zn), zhi = fmaxf(zp, zn);
                        const bool near_is_right = fabsf(zhi - mu[u]) < fabsf(zlo - mu[u]);
                        const float s_far = score_exact(near_is_right ? zlo : zhi, mu[u], sg[u], rs1,
                                                        sPen[n * VBQ_GROUP + col]);
                        use_r = near_is_right && bestL[u] > s_far;
                    }
                    path_wins = use_r ? zp >= zn : zp <= zn;
                }
                // the neighbour's index is ipn + d except in the one padded case that holds a different point: above
                // the highest point of depth N the right pad is the second-highest point (no edge padding there)
                int i = path_wins ? ipn : ipn + d;
                if (!path_wins && n == N && ((ipn + d) >> n) != 0) i = ipn - 1;
                i = max(i, 0);   // left pad (d = -1 at ipn = 0) duplicates point 0; it never wins against the path
                const float zh = path_wins ? zp : zn;
                const int q = ((2 * i + 1) << (N - n)) - 1;
                if (row + u * RP < row_end) {
                    const unsigned o = off + u * off_step;
                    const float ln = (outm & 64u) ? sLenc[n * VBQ_GROUP] : (float)n;
                    float eb = 0.0f;
                    if (outm & 32u) eb = __ldg(gEm + q);
                    if (outm & 1u) zhat_c[o] = zh;
                    if (outm & 2u) qidx_c[o] = q;
                    if (outm & 4u) level_c[o] = n;
                    if (outm & 8u) bits_c[o] = ln;
                    if (outm & 16u) emb_c[o] = eb;
                    if (TOTALS) {
                        // distortion of the winner 0.5*t^2 = pen - (-score), up to one float32 rounding of the score
                        const float best = (MODE == kModeReference && use_r) ? bestR[u] : bestL[u];
                        acc_level += n;
                        if (outm & 64u) acc_len += (double)ln;
                        if (outm & 32u) acc_em += (double)eb;
                        acc_dist += (double)sPen[n * VBQ_GROUP + col] - (double)best;
                    }
                }
            }
        }
        cp_async_wait<0>();
    }

    if (TOTALS) {
        // raw-length mode: the code length of depth n is n itself
        double v[VBQ_TOTALS] = {(double)acc_level, (outm & 64u) ? acc_len : (double)acc_level, acc_em, acc_dist};
#pragma unroll
        for (int k = 0; k < VBQ_TOTALS; ++k) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
            if ((threadIdx.x & 31) == 0) sRed[k][threadIdx.x >> 5] = v[k];
        }
        __syncthreads();
        double *part = a.partials + ((size_t)lam * kMaxGrid + blockIdx.x) * VBQ_TOTALS;
        if (threadIdx.x < VBQ_TOTALS) {
            double s = 0.0;
            for (int w = 0; w < kThreads / 32; ++w) s += sRed[threadIdx.x][w];
            part[threadIdx.x] = s;
            __threadfence();
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned t = atomicAdd(a.ticket + lam, 1u);
            sLast = (t == gridDim.x - 1);
        }
        __syncthreads();
        if (sLast && threadIdx.x < VBQ_TOTALS) {   // the last CTA of this lambda adds the partials in a fixed order
            __threadfence();
            const volatile double *p = a.partials + (size_t)lam * kMaxGrid * VBQ_TOTALS;
            double s = a.accumulate ? a.totals[lam * VBQ_TOTALS + threadIdx.x] : 0.0;
            for (unsigned b = 0; b < gridDim.x; ++b) s += p[b * VBQ_TOTALS + threadIdx.x];
            a.totals[lam * VBQ_TOTALS + threadIdx.x] = s;
            if (threadIdx.x == 0) a.ticket[lam] = 0u;
        }
    }
}

template <int MODE, bool PRUNE, bool TOTALS, bool DEEP, bool EXTRAS, int NT, int U, int T>
static int launch_quantize(QArgs a, int dev, int sms, cudaStream_t st) {
    constexpr int rows_per_pass = T / VBQ_GROUP;
    a.passes = (a.rows + rows_per_pass - 1) / rows_per_pass;
    a.total_units = a.passes * a.n_groups;
    // one persistent CTA per SM, each taking a contiguous span of (group, row-pass) units
    long long gx = (a.total_units + U - 1) / U;
    if (gx > sms) gx = sms;
    if (gx > kMaxGrid) gx = kMaxGrid;
    const size_t smem = ((size_t)kPadEntries * VBQ_GROUP + 3 * (size_t)(a.N + 1) * VBQ_GROUP +
                         (size_t)kStages * 2 * U * T) * sizeof(float);
    auto kern = vbq_quantize_kernel<MODE, PRUNE, TOTALS, DEEP, EXTRAS, NT, U, T>;
    VBQ_ENSURE_MAX_SMEM(kern, dev);
    kern<<<dim3((int)gx, a.n_lambda), T, smem, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

template <int MODE, bool PRUNE, bool TOTALS, bool EXTRAS, int U, int T>
static int launch_mode3(const QArgs &a, int dev, int sms, cudaStream_t st) {
    if (a.N > kSmemDepth) {   // deep tables: depths 11..N come from global memory, reference walk (or fast)
        constexpr int M = MODE == kModeStrict ? kModeReference : MODE;
        return launch_quantize<M, PRUNE, TOTALS, true, EXTRAS, 0, U, T>(a, dev, sms, st);
    }
    if (a.N == kSmemDepth) return launch_quantize<MODE, PRUNE, TOTALS, false, EXTRAS, kSmemDepth, U, T>(a, dev, sms, st);
    return launch_quantize<MODE, PRUNE, TOTALS, false, EXTRAS, 0, U, T>(a, dev, sms, st);
}

template <int MODE, bool PRUNE, int U, int T>
static int launch_mode2(const QArgs &a, int dev, int sms, cudaStream_t st) {
    const bool tot = a.totals != nullptr, extras = a.len != nullptr || a.em != nullptr;
    if (tot) return extras ? launch_mode3<MODE, PRUNE, true, true, U, T>(a, dev, sms, st)
                           : launch_mode3<MODE, PRUNE, true, false, U, T>(a, dev, sms, st);
    return extras ? launch_mode3<MODE, PRUNE, false, true, U, T>(a, dev, sms, st)
                  : launch_mode3<MODE, PRUNE, false, false, U, T>(a, dev, sms, st);
}

// entry point of one scoring mode (defined by the translation unit that includes this header)
template <int MODE>
static int launch_quantize_mode(const QArgs &a, int dev, int sms, cudaStream_t st) {
    // 640 threads (20 warps, <= 102 registers): measured best of 512 / 640 / 768 for the strict kernel
    const bool prune = !(a.flags & VBQ_FLAG_NO_PRUNE);
    return prune ? launch_mode2<MODE, true, 2, 640>(a, dev, sms, st) : launch_mode2<MODE, false, 2, 640>(a, dev, sms, st);
}
