// sweep.cu — rate-distortion SWEEP: all lambdas of a call in one tree walk.
//
// The distortion term -0.5*((z-mu)/sigma)^2 of a candidate does not depend on lambda (the reference computes
// `fun_P` once, utils.py:387, then loops over lambs, utils.py:392-421).  This kernel walks the tree once per
// coordinate, keeps the 2N+1 distortion terms in registers, and evaluates every lambda from them:
// score = fl(h + (-pen[lambda][c][n])) is bit-identical to the reference's fl(fl(-0.5 t^2) - fl(lambda*len)).
// Used by vbq_quantize when n_lambda > 1 and max_bits_per_coord <= 10; the per-lambda results are identical to the
// single-lambda kernel (tests/test_gpu_parity.py::test_sweep_equals_per_lambda_walks).
#include <stdlib.h>

#include "tree.cuh"

// h = fl(-0.5 * fl(t^2)), t = fl(fl(z - mu) / sigma): the lambda-independent part of utils.py:318-320
__device__ __forceinline__ float2 distortion_exact2(float2 z, float2 nmu, float2 nsg, float2 rs) {
    const float2 d = __fadd2_rn(z, nmu);
    const float2 q0 = __fmul2_rn(d, rs);
    const float2 e = __ffma2_rn(q0, nsg, d);
    const float2 q = __ffma2_rn(e, rs, q0);
    return __fmul2_rn(__fmul2_rn(q, q), make_float2(-0.5f, -0.5f));
}

__device__ __forceinline__ float2 distortion_fast2(float2 zp, float2 zn, float2 nmu, float2 nw) {
    const float2 dp = __fadd2_rn(zp, nmu), dn = __fadd2_rn(zn, nmu);
    const float2 d = make_float2(fminf(fabsf(dp.x), fabsf(dn.x)), fminf(fabsf(dp.y), fabsf(dn.y)));
    return __fmul2_rn(__fmul2_rn(d, d), nw);
}

template <bool FAST, bool TOTALS, int kThreads, int LP>
__global__ void __launch_bounds__(kThreads, 1) vbq_sweep_kernel(const QArgs a) {
    constexpr int U = 2;                                  // one f32x2 pair of coordinates per thread
    constexpr int RP = kThreads / VBQ_GROUP;
    extern __shared__ __align__(16) float smem[];
    const int N = a.N;                                    // <= kSmemDepth
    const int L = a.n_lambda;
    float *sT = smem;                                     // [kPadEntries][16]
    float *sPen = sT + kPadEntries * VBQ_GROUP;           // [L][N+1][16] negated penalties
    float *sLen = sPen + (size_t)L * (N + 1) * VBQ_GROUP; // [L][N+1][16] code lengths (only if a.len is given)
    float *sStage = sLen + (a.len ? (size_t)L * (N + 1) * VBQ_GROUP : 0);   // [kStages][2][U][kThreads]
    double *sAcc = reinterpret_cast<double *>(sStage + kStages * 2 * U * kThreads);   // [warps][L][4]
    float *myStage = sStage + threadIdx.x;
    __shared__ bool sLast;

    const int col = threadIdx.x & (VBQ_GROUP - 1);
    const int rsub = threadIdx.x >> 4;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool logvar = (a.flags & VBQ_FLAG_LOGVAR) != 0;
    const long long u0 = a.total_units * blockIdx.x / gridDim.x;
    const long long u1 = a.total_units * (blockIdx.x + 1) / gridDim.x;
    const int C = a.C;
    const int rows = (int)a.rows;
    const char *pb = reinterpret_cast<const char *>(sT) + col * 4 - 32;
    const float *sTc = sT + col;
    const bool any_out = a.zhat || a.qidx || a.level || a.bits || a.em_bits;

    if (TOTALS) {
        for (int k = threadIdx.x; k < (kThreads / 32) * L * VBQ_TOTALS; k += kThreads) sAcc[k] = 0.0;
    }

    long long unit = u0;
    while (unit < u1) {
        const int g = (int)(unit / a.passes);
        const int p0 = (int)(unit - (long long)g * a.passes);
        const int p1 = (int)min(a.passes, (long long)p0 + (u1 - unit));
        unit += p1 - p0;

        __syncthreads();
        {
            const float4 *src = reinterpret_cast<const float4 *>(a.packed + (size_t)g * kPadEntries * VBQ_GROUP);
            float4 *dst = reinterpret_cast<float4 *>(sT);
            for (int k = threadIdx.x; k < kPadEntries * (VBQ_GROUP / 4); k += kThreads) dst[k] = __ldg(src + k);
            for (int k = threadIdx.x; k < L * (N + 1) * VBQ_GROUP; k += kThreads) {
                const int j = k & (VBQ_GROUP - 1);
                const int n = (k >> 4) % (N + 1);
                const int lam = (k >> 4) / (N + 1);
                const int cj = min(g * VBQ_GROUP + j, C - 1);
                const size_t po = ((size_t)lam * a.pen_channels + (a.pen_channels == 1 ? 0 : cj)) * (N + 1) + n;
                sPen[k] = -a.pen[po];
                if (a.len) sLen[k] = a.len[po];
            }
        }
        __syncthreads();

        const int c = g * VBQ_GROUP + col;
        const bool c_ok = c < C;
        const int cc = min(c, C - 1);
        const float *mu_c = a.mu + cc;
        const float *sg_c = a.sigma + cc;
        const float z0 = sTc[entry_of(0, 0) * VBQ_GROUP];

        const int row_end = c_ok ? min(p1 * RP, rows) : 0;
        int row = p0 * RP + rsub;
        unsigned off = (unsigned)row * (unsigned)C;
        const unsigned off_step = (unsigned)(RP * C);

        auto stage_rows = [&](int it_row, unsigned it_off, int slot) {
#pragma unroll
            for (int u = 0; u < U; ++u) {
                if (it_row + u * RP < row_end) {
                    cp_async_f32(myStage + ((slot * 2 + 0) * U + u) * kThreads, mu_c + it_off + u * off_step);
                    cp_async_f32(myStage + ((slot * 2 + 1) * U + u) * kThreads, sg_c + it_off + u * off_step);
                }
            }
            cp_async_commit();
        };
#pragma unroll
        for (int k = 0; k < kStages - 1; ++k) stage_rows(row + k * U * RP, off + k * U * off_step, k);
        int slot = 0;

        for (; row - rsub < p1 * RP; row += U * RP, off += U * off_step) {
            float mu[U], sg[U];
            cp_async_wait<kStages - 2>();
            bool ok[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                ok[u] = row + u * RP < row_end;
                mu[u] = ok[u] ? myStage[((slot * 2 + 0) * U + u) * kThreads] : 0.0f;
                float s = ok[u] ? myStage[((slot * 2 + 1) * U + u) * kThreads] : 1.0f;
                if (logvar) s = sigma_of_logvar(s);
                sg[u] = s;
            }
            {
                const int ps = slot == 0 ? kStages - 1 : slot - 1;
                stage_rows(row + (kStages - 1) * U * RP, off + (kStages - 1) * U * off_step, ps);
                slot = slot == kStages - 1 ? 0 : slot + 1;
            }
            const float r0 = rcp_rn(sg[0]), r1 = rcp_rn(sg[1]);
            const float2 nmu2 = make_float2(-mu[0], -mu[1]);
            const float2 nsg2 = make_float2(-sg[0], -sg[1]);
            const float2 rs2 = FAST ? make_float2(-0.5f * r0 * r0, -0.5f * r1 * r1) : make_float2(r0, r1);

            // ---- one walk: lambda-independent distortion terms of all candidates ---------------------------
            float2 hL[kSmemDepth + 1], hR[kSmemDepth + 1];   // hR unused in FAST mode
            int V[U];
            {
                const float2 z02 = make_float2(z0, z0);
                hL[0] = FAST ? distortion_fast2(z02, z02, nmu2, rs2) : distortion_exact2(z02, nmu2, nsg2, rs2);
                hR[0] = make_float2(-CUDART_INF_F, -CUDART_INF_F);
                V[0] = mu[0] > z0 ? 96 : 32;
                V[1] = mu[1] > z0 ? 96 : 32;
            }
#pragma unroll
            for (int n = 1; n <= kSmemDepth; ++n) {
                if (n > N) break;
                const int imm = entry_of(n, 0) * kRowStrideBytes;
                float zp[U], zn[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const char *pa = pb + V[u];
                    zp[u] = lds_f32(pa, imm);
                    const int s = mu[u] > zp[u] ? 32 : -32;
                    zn[u] = lds_f32(pa + 2 * s, imm);
                    V[u] = 2 * V[u] + s;
                }
                if (FAST) {
                    hL[n] = distortion_fast2(make_float2(zp[0], zp[1]), make_float2(zn[0], zn[1]), nmu2, rs2);
                } else {
                    hL[n] = distortion_exact2(make_float2(fminf(zp[0], zn[0]), fminf(zp[1], zn[1])), nmu2, nsg2, rs2);
                    hR[n] = distortion_exact2(make_float2(fmaxf(zp[0], zn[0]), fmaxf(zp[1], zn[1])), nmu2, nsg2, rs2);
                }
            }
            const int idx[U] = {V[0] >> 6, V[1] >> 6};   // path index at depth N + 1

            // ---- every lambda from the registers, LP lambdas at a time (independent running maxima => ILP) ------
            for (int lam0 = 0; lam0 < L; lam0 += LP) {
                float bL[LP][U], bR[LP][U];
                int nL[LP][U], nR[LP][U];
                const float *pl[LP];
#pragma unroll
                for (int j = 0; j < LP; ++j) {
                    const int lam = min(lam0 + j, L - 1);   // a ragged last group recomputes the last lambda
                    pl[j] = sPen + (size_t)lam * (N + 1) * VBQ_GROUP + col;
                    const float np0 = pl[j][0];
                    bL[j][0] = hL[0].x + np0;
                    bL[j][1] = hL[0].y + np0;
                    bR[j][0] = bR[j][1] = -CUDART_INF_F;
                    nL[j][0] = nL[j][1] = nR[j][0] = nR[j][1] = 0;
                }
#pragma unroll
                for (int n = 1; n <= kSmemDepth; ++n) {
                    if (n > N) break;
#pragma unroll
                    for (int j = 0; j < LP; ++j) {
                        const float npn = pl[j][n * VBQ_GROUP];
                        const float2 sl = __fadd2_rn(hL[n], make_float2(npn, npn));
                        if (sl.x > bL[j][0]) { bL[j][0] = sl.x; nL[j][0] = n; }
                        if (sl.y > bL[j][1]) { bL[j][1] = sl.y; nL[j][1] = n; }
                        if (!FAST) {
                            const float2 sr = __fadd2_rn(hR[n], make_float2(npn, npn));
                            if (sr.x > bR[j][0]) { bR[j][0] = sr.x; nR[j][0] = n; }
                            if (sr.y > bR[j][1]) { bR[j][1] = sr.y; nR[j][1] = n; }
                        }
                    }
                }
#pragma unroll
                for (int j = 0; j < LP; ++j) {
                    const int lam = lam0 + j;
                    if (lam >= L) break;
                    double t_len = 0.0, t_em = 0.0, t_dist = 0.0;
                    int t_level = 0;
                    const size_t lam_off = (size_t)lam * (size_t)a.lam_stride;
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const bool use_r = !FAST && (bR[j][u] > bL[j][u]);
                        const int n = use_r ? nR[j][u] : nL[j][u];
                        const float best = use_r ? bR[j][u] : bL[j][u];
                        const float ln = a.len ? sLen[((size_t)lam * (N + 1) + n) * VBQ_GROUP + col] : (float)n;
                        float eb = 0.0f;
                        if (any_out || a.em) {
                            // rebuild the bracket of depth n from the final path (see quantize.cu)
                            const int sh = N + 1 - n;
                            const int ipn = idx[u] >> sh;
                            const int d = ((idx[u] >> (sh - 1)) & 1) ? 1 : -1;
                            const int last = (1 << n) - 1;
                            int inb = min(max(ipn + d, 0), last);
                            if (n == N && ipn + d > last) inb = max(last - 1, 0);
                            const float *e = sTc + (entry_of(n, 0) + ipn) * VBQ_GROUP;
                            const float zp = e[0], zn = e[d * VBQ_GROUP];
                            bool path_wins;
                            if (FAST) {
                                const float dp = fabsf(zp - mu[u]), dn = fabsf(zn - mu[u]);
                                path_wins = dp < dn || (dp == dn && zp <= zn);
                            } else {
                                path_wins = use_r ? zp >= zn : zp <= zn;
                            }
                            const int i = path_wins ? ipn : inb;
                            const float zh = path_wins ? zp : zn;
                            const int q = ((2 * i + 1) << (N - n)) - 1;
                            if (ok[u]) {
                                const size_t o = lam_off + off + u * off_step + cc;
                                if (a.em) eb = __ldg(a.em + ((size_t)lam * C + cc) * a.Q + q);
                                if (a.zhat) a.zhat[o] = zh;
                                if (a.qidx) a.qidx[o] = q;
                                if (a.level) a.level[o] = n;
                                if (a.bits) a.bits[o] = ln;
                                if (a.em_bits) a.em_bits[o] = eb;
                            }
                        }
                        if (TOTALS && ok[u]) {
                            // distortion of the winner = -h = pen - (-score), up to one float32 rounding of the score
                            const float npw = pl[j][n * VBQ_GROUP];
                            t_level += n;
                            t_len += (double)ln;
                            t_em += (double)eb;
                            t_dist += (double)npw - (double)best;
                        }
                    }
                    if (TOTALS) {
                        t_level = __reduce_add_sync(0xffffffffu, t_level);
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) {
                            t_len += __shfl_xor_sync(0xffffffffu, t_len, o);
                            t_em += __shfl_xor_sync(0xffffffffu, t_em, o);
                            t_dist += __shfl_xor_sync(0xffffffffu, t_dist, o);
                        }
                        if (lane == 0) {
                            double *acc = sAcc + ((size_t)warp * L + lam) * VBQ_TOTALS;
                            acc[0] += (double)t_level;
                            acc[1] += t_len;
                            acc[2] += t_em;
                            acc[3] += t_dist;
                        }
                    }
                }
            }
        }
        cp_async_wait<0>();
    }

    if (TOTALS) {
        __syncthreads();
        // per-CTA partials, then the last CTA adds the partials of all CTAs in a fixed order (deterministic)
        for (int k = threadIdx.x; k < L * VBQ_TOTALS; k += kThreads) {
            double s = 0.0;
            for (int w = 0; w < kThreads / 32; ++w) s += sAcc[(size_t)w * L * VBQ_TOTALS + k];
            const int lam = k / VBQ_TOTALS, t = k % VBQ_TOTALS;
            a.partials[((size_t)lam * kMaxGrid + blockIdx.x) * VBQ_TOTALS + t] = s;
        }
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) {
            const unsigned t = atomicAdd(a.ticket, 1u);
            sLast = (t == gridDim.x - 1);
        }
        __syncthreads();
        if (sLast) {
            __threadfence();
            for (int k = threadIdx.x; k < L * VBQ_TOTALS; k += kThreads) {
                const int lam = k / VBQ_TOTALS, t = k % VBQ_TOTALS;
                const volatile double *p = a.partials + (size_t)lam * kMaxGrid * VBQ_TOTALS;
                double s = a.accumulate ? a.totals[k] : 0.0;
                for (unsigned b = 0; b < gridDim.x; ++b) s += p[b * VBQ_TOTALS + t];
                a.totals[k] = s;
            }
            if (threadIdx.x == 0) a.ticket[0] = 0u;
        }
    }
}

template <bool FAST, bool TOTALS, int T, int LP>
static int launch_sweep_t(QArgs a, int dev, int sms, cudaStream_t st) {
    constexpr int U = 2;
    constexpr int rows_per_pass = T / VBQ_GROUP;
    a.passes = (a.rows + rows_per_pass - 1) / rows_per_pass;
    a.total_units = a.passes * a.n_groups;
    long long gx = (a.total_units + U - 1) / U;
    if (gx > sms) gx = sms;
    if (gx > kMaxGrid) gx = kMaxGrid;
    // shared memory: tree + staging ring are fixed, penalties / lengths / accumulators grow with the lambda count;
    // calls with more lambdas than fit are served in lambda chunks
    const size_t fixed = ((size_t)kPadEntries * VBQ_GROUP + (size_t)kStages * 2 * U * T) * sizeof(float);
    const size_t per_lambda = (a.len ? 2 : 1) * (size_t)(a.N + 1) * VBQ_GROUP * sizeof(float) +
                              (TOTALS ? (size_t)(T / 32) * VBQ_TOTALS * sizeof(double) : 0);
    const int max_l = (int)((227 * 1024 - fixed) / per_lambda);
    if (max_l < 2) return -1;
    auto kern = vbq_sweep_kernel<FAST, TOTALS, T, LP>;
    const int n_lambda = a.n_lambda;
    const size_t pen_stride = (size_t)a.pen_channels * (a.N + 1);
    for (int l0 = 0; l0 < n_lambda; l0 += max_l) {
        QArgs b = a;
        b.n_lambda = n_lambda - l0 < max_l ? n_lambda - l0 : max_l;
        b.pen = a.pen + l0 * pen_stride;
        if (a.len) b.len = a.len + l0 * pen_stride;
        if (a.em) b.em = a.em + (size_t)l0 * a.C * a.Q;
        const size_t oo = (size_t)l0 * (size_t)a.lam_stride;
        if (a.zhat) b.zhat = a.zhat + oo;
        if (a.qidx) b.qidx = a.qidx + oo;
        if (a.level) b.level = a.level + oo;
        if (a.bits) b.bits = a.bits + oo;
        if (a.em_bits) b.em_bits = a.em_bits + oo;
        if (a.totals) {
            b.totals = a.totals + (size_t)l0 * VBQ_TOTALS;
            b.partials = a.partials + (size_t)l0 * kMaxGrid * VBQ_TOTALS;
        }
        const size_t smem = fixed + per_lambda * b.n_lambda;
        VBQ_ENSURE_MAX_SMEM(kern, dev);
        kern<<<dim3((int)gx, 1), T, smem, st>>>(b);
        CUDA_TRY(cudaGetLastError());
    }
    return VBQ_OK;
}

// returns -1 when the sweep does not apply (caller uses the per-lambda kernel), else a VBQ_* status
int vbq_launch_sweep(const QArgs &a, int dev, int sms, cudaStream_t st) {
    if (a.N > kSmemDepth || a.n_lambda < 2) return -1;
    const bool fast = (a.flags & VBQ_FLAG_FAST) != 0, tot = a.totals != nullptr;
    // development override (read once): VBQ_SWEEP_TUNE=<threads/128><lambdas per group>
    static const int tune = getenv("VBQ_SWEEP_TUNE") ? atoi(getenv("VBQ_SWEEP_TUNE")) : 61;
#define SWEEP_CASE(T, LP)                                                                                        \
    if (fast) return tot ? launch_sweep_t<true, true, T, LP>(a, dev, sms, st) : launch_sweep_t<true, false, T, LP>(a, dev, sms, st); \
    return tot ? launch_sweep_t<false, true, T, LP>(a, dev, sms, st) : launch_sweep_t<false, false, T, LP>(a, dev, sms, st);
    switch (tune) {
        case 51: { SWEEP_CASE(640, 1) }
        case 41: { SWEEP_CASE(512, 1) }
        default: { SWEEP_CASE(768, 1) }
    }
#undef SWEEP_CASE
}
