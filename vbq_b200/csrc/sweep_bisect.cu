// sweep_bisect.cu — rate-distortion SWEEP by certified bisection: all lambdas of a call from one tree walk (sm_100a).
//
// Reference behaviour reproduced (paths relative to mandt-lab/vbq): utils.py:387 computes the distortion term of every
// candidate once and utils.py:392-421 loops over `lambs`; quantizer.py:156-188 builds the candidates.  As in
// quantize_bisect.cu only the N+1 path nodes of a coordinate can win when the penalties are non-decreasing in depth,
// and they are ranked by an approximate loss with an integer guard band; here the lambda-independent part
// t_n^2 = ((z_n - mu) sqrt(1/2) / sigma)^2 of the 11 path nodes stays in registers and every lambda costs one packed
// add, one LOP3 per key, the 3-input minimum chain and the VIADDMNMX gap chain.  Coordinates whose ranking is not
// certified for some lambda are redone for that lambda by `reference_search` (literal two-ended walk, IEEE float32).
// Applies to raw code lengths (penalty = fl(lambda * n), identical for all channels), max_bits_per_coord <= 10; other
// calls use vbq_sweep_kernel (sweep.cu).
#include <stdlib.h>

#include "bisect.cuh"

constexpr int kPenSlots = 12;   // per lambda: penalties of depths 0..10 and the guard word, 48 bytes (three float4)

// OUTS: per-coordinate outputs are requested (otherwise the call returns only the per-lambda totals and the lambda loop
// carries no output pointers, masks or addresses)
template <bool TOTALS, bool OUTS, bool VEC, int kThreads>
__global__ void __launch_bounds__(kThreads, 1) vbq_bisect_sweep_kernel(const QArgs a) {
    constexpr int U = 2;
    constexpr int kWarps = kThreads / 32;
    extern __shared__ __align__(16) float smem[];
    const int N = a.N;                                  // <= kSmemDepth
    const int L = a.n_lambda;
    float *sT = smem;                                   // [kPadEntries][16] code points of depths 0..10
    float *sPenL = sT + kPadEntries * VBQ_GROUP;        // [L][kPenSlots]: pen_0..pen_10 (+inf beyond N), guard word
    float *sStage = sPenL + (size_t)L * kPenSlots;      // [kWarps][kStages][kTileFloats] staging rings
    double *sAcc = reinterpret_cast<double *>(sStage + kWarps * kStages * kTileFloats);   // [kWarps][L][2]: sum n, sum dist
    __shared__ int sNext;
    __shared__ bool sLast;

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col = lane & (VBQ_GROUP - 1);
    const int par = lane >> 4;
    const bool logvar = (a.flags & VBQ_FLAG_LOGVAR) != 0;
    const int C = a.C;
    const int rows = (int)a.rows;
    const long long tpg = a.passes;                     // tiles per group
    const long long vtotal = (tpg + kSwitchTiles) * a.n_groups;
    const long long u0 = span_cut(vtotal * blockIdx.x / gridDim.x, tpg, a.n_groups);
    const long long u1 = span_cut(vtotal * (blockIdx.x + 1) / gridDim.x, tpg, a.n_groups);
    const int pbi = (int)__cvta_generic_to_shared(sT + col);
    const float *sTc = sT + col;
    const unsigned kmask = a.keymask;
    float *wStage = sStage + warp * (kStages * kTileFloats);
    const float *myStage = wStage + par * VBQ_GROUP + col;
    double *wAcc = sAcc + (size_t)warp * L * 2;

    if (TOTALS) {
        for (int k = threadIdx.x; k < kWarps * L * 2; k += kThreads) sAcc[k] = 0.0;
    }
    pdl_wait();   // launched with programmatic stream serialization: nothing global is touched before this point
    // penalties are the same for every group (pen_channels == 1): staged once
    for (int lam = threadIdx.x; lam < L; lam += kThreads) {
        float prev = 0.0f;
        bool mono = true;
        for (int n = 0; n <= kSmemDepth; ++n) {
            const float p = n <= N ? a.pen[(size_t)lam * (N + 1) + n] : CUDART_INF_F;
            mono = mono && (p >= prev);
            prev = p;
            sPenL[lam * kPenSlots + n] = p;
        }
        sPenL[lam * kPenSlots + kSmemDepth + 1] = __uint_as_float(mono ? kKeyGuard : 0xffffffffu);
    }

    long long unit = u0;
    while (unit < u1) {
        const int g = (int)(unit / tpg);
        const int t0 = (int)(unit - (long long)g * tpg);
        const int n_tiles = (int)min(tpg - t0, u1 - unit);
        unit += n_tiles;

        __syncthreads();                     // every warp has left the previous segment
        if (threadIdx.x == 0) sNext = 0;
        __syncthreads();
        const int c = g * VBQ_GROUP + col;
        const bool c_ok = c < C;
        const int cc = min(c, C - 1);
        const unsigned thr_off = (unsigned)(t0 * kTileRows + par) * (unsigned)C + (unsigned)cc;
        const unsigned tile_step = (unsigned)(kTileRows * C), u_step = (unsigned)(2 * C);
        const int seg_row0 = t0 * kTileRows;
        const bool group_full = g * VBQ_GROUP + VBQ_GROUP <= C;
        const int full_tiles = group_full ? min(n_tiles, (rows - seg_row0) / kTileRows) : 0;

        const int prod_row = VEC ? ((lane >> 2) & 3) : par;
        const int prod_col = VEC ? g * VBQ_GROUP + (lane & 3) * 4 : cc;
        const float *prod_src = ((VEC && (lane >> 4)) ? a.sigma : a.mu) + ((size_t)(seg_row0 + prod_row) * C + prod_col);
        float *prod_dst = VEC ? wStage + (lane >> 4) * (kTileRows * VBQ_GROUP) + prod_row * VBQ_GROUP + (lane & 3) * 4
                              : wStage + par * VBQ_GROUP + col;
        const bool prod_col_ok = VEC ? prod_col < C : c_ok;
        auto claim = [&]() -> int { return claim_tile(&sNext, lane); };
        auto stage = [&](int j, int slot) {   // every call commits exactly one group (possibly empty)
            if (j < n_tiles) {
                const float *src = prod_src + (size_t)j * tile_step;
                float *dst = prod_dst + slot * kTileFloats;
                if (VEC) {
                    if (j < full_tiles || (prod_col_ok && seg_row0 + j * kTileRows + prod_row < rows)) cp_async_16(dst, src);
                } else {
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        if (j < full_tiles || (prod_col_ok && seg_row0 + j * kTileRows + 2 * u + par < rows)) {
                            cp_async_f32(dst + u * 2 * VBQ_GROUP, src + u * u_step);
                            cp_async_f32(dst + kTileRows * VBQ_GROUP + u * 2 * VBQ_GROUP, a.sigma + (src - a.mu) + u * u_step);
                        }
                    }
                }
            }
            cp_async_commit();
        };
        int q0 = claim(), q1 = claim(), q2 = claim();
        static_assert(kStages == 4, "the claim queue holds kStages - 1 = 3 tiles");
        stage(q0, 0);
        stage(q1, 1);
        stage(q2, 2);
        int slot = 0;

        {   // the group's tree, while the first tiles are in flight
            const float4 *src = reinterpret_cast<const float4 *>(a.packed + (size_t)g * kPadEntries * VBQ_GROUP);
            float4 *dst = reinterpret_cast<float4 *>(sT);
            for (int k = threadIdx.x; k < kPadEntries * (VBQ_GROUP / 4); k += kThreads) dst[k] = __ldg(src + k);
        }
        __syncthreads();
        const float z0 = sTc[entry_of(0, 0) * VBQ_GROUP];
        unsigned pen0 = (unsigned)__cvta_generic_to_shared(sPenL);
        asm volatile("" : "+r"(pen0));   // opaque: the penalty loads below stay behind the barrier above

        while (q0 < n_tiles) {
            const int nxt = claim();
            cp_async_wait<kStages - 2>();
            __syncwarp();
            const int tile = q0;
            const bool check = tile >= full_tiles;
            const int row = seg_row0 + tile * kTileRows + par;
            const unsigned off = thr_off + (unsigned)tile * tile_step;
            float mu[U], sg[U];
            bool ok[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                ok[u] = !check || (c_ok && row + 2 * u < rows);
                mu[u] = ok[u] ? myStage[slot * kTileFloats + u * 2 * VBQ_GROUP] : 0.0f;
                float s = ok[u] ? myStage[slot * kTileFloats + kTileRows * VBQ_GROUP + u * 2 * VBQ_GROUP] : 1.0f;
                if (logvar) s = sigma_of_logvar(s);
                sg[u] = s;
            }
            const float2 nmu2 = make_float2(-mu[0], -mu[1]);
            const float2 r2 = __fmul2_rn(make_float2(rcp_approx(sg[0]), rcp_approx(sg[1])),
                                         make_float2(0.70710678f, 0.70710678f));

            // ---- one walk: t^2 of the path node of every depth (lambda-independent) -------------------------
            float2 t2[kSmemDepth + 1];
            unsigned K[U];
#pragma unroll
            for (int n = 0; n <= kSmemDepth; ++n) t2[n] = make_float2(CUDART_INF_F, CUDART_INF_F);
            {
                const float2 d = __fadd2_rn(make_float2(z0, z0), nmu2);
                const float2 t = __fmul2_rn(d, r2);
                t2[0] = __fmul2_rn(t, t);
                K[0] = __funnelshift_l(__float_as_uint(d.x), 1u, 1);
                K[1] = __funnelshift_l(__float_as_uint(d.y), 1u, 1);
            }
#pragma unroll
            for (int n = 1; n <= kSmemDepth; ++n) {
                if (n > N) break;
                float z[U];
#pragma unroll
                for (int u = 0; u < U; ++u)
                    z[u] = lds_pure((unsigned)(imad((int)K[u], kRowStrideBytes, pbi) + 2 * n * kRowStrideBytes));
                const float2 d = __fadd2_rn(make_float2(z[0], z[1]), nmu2);
                K[0] = __funnelshift_l(__float_as_uint(d.x), K[0], 1);
                K[1] = __funnelshift_l(__float_as_uint(d.y), K[1], 1);
                const float2 t = __fmul2_rn(d, r2);
                t2[n] = __fmul2_rn(t, t);
            }
            const int kd = N + 1;   // depth of the node K points at

            // ---- every lambda from the registers ----------------------------------------------------------------
            // lane j of the warp keeps the tile's sums of lambda lb + j; they reach shared memory once per 32 lambdas
            for (int lb = 0; lb < L; lb += 32) {
            int my_level = 0;
            float my_dist = 0.0f;
            const int lend = min(L, lb + 32);
            for (int lam = lb; lam < lend; ++lam) {
                const unsigned pen_a = pen0 + (unsigned)lam * (kPenSlots * 4);   // 32-bit shared-memory address: no generic-pointer arithmetic
                const float4 pa = lds128_pure(pen_a), pb = lds128_pure(pen_a + 16), pc = lds128_pure(pen_a + 32);
                const float pen[kSmemDepth + 1] = {pa.x, pa.y, pa.z, pa.w, pb.x, pb.y, pb.z, pb.w, pc.x, pc.y, pc.z};
                const unsigned guard = __float_as_uint(pc.w);
                unsigned key[U][kSmemDepth + 1];
#pragma unroll
                for (int n = 0; n <= kSmemDepth; ++n) {
                    const float2 A = __fadd2_rn(t2[n], make_float2(pen[n], pen[n]));
                    key[0][n] = (__float_as_uint(A.x) & kmask) | (unsigned)n;
                    key[1][n] = (__float_as_uint(A.y) & kmask) | (unsigned)n;
                }
                int wn[U], wP[U];
                unsigned gapmin = 0xffffffffu;
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const unsigned *k_ = key[u];
                    unsigned m = __vimin3_u32(k_[0], k_[1], k_[2]);
                    m = __vimin3_u32(m, k_[3], k_[4]);
                    m = __vimin3_u32(m, k_[5], k_[6]);
                    m = __vimin3_u32(m, k_[7], k_[8]);
                    m = __vimin3_u32(m, k_[9], k_[10]);
                    const unsigned nm = ~m;
                    unsigned g0 = 0xffffffffu, g1 = 0xffffffffu;
#pragma unroll
                    for (int n = 0; n <= kSmemDepth; n += 2) g0 = __viaddmin_u32(k_[n], nm, g0);
#pragma unroll
                    for (int n = 1; n <= kSmemDepth; n += 2) g1 = __viaddmin_u32(k_[n], nm, g1);
                    gapmin = __vimin3_u32(gapmin, g0, g1);
                    wn[u] = (int)(m & 15u);
                    wP[u] = (int)(K[u] >> (kd - wn[u]));
                }
                if (gapmin <= guard) {   // not certified for this lambda (or penalties not monotone): literal search
#pragma unroll
                    for (int u = 0; u < U; ++u) {
                        const int r = reference_search(sTc, sPenL + lam * kPenSlots, 1, mu[u], sg[u], N);
                        wn[u] = r >> 24;
                        wP[u] = (1 << wn[u]) + (r & 0xffffff);
                    }
                }
                int t_level = 0;
                float t_dist = 0.0f;
                const size_t lam_off = (size_t)lam * (size_t)a.lam_stride;
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int n = wn[u], Pn = wP[u];
                    if ((TOTALS || OUTS) && ok[u]) {
                        const float zh = lds_pure((unsigned)(imad(n, 2 * kRowStrideBytes, imad(Pn, kRowStrideBytes, pbi))));
                        if (OUTS) {
                            const size_t o = lam_off + off + u * u_step;
                            const int q = ((2 * Pn + 1) << (N - n)) - (2 << N) - 1;
                            if (a.zhat) a.zhat[o] = zh;
                            if (a.qidx) a.qidx[o] = q;
                            if (a.level) a.level[o] = n;
                            if (a.bits) a.bits[o] = (float)n;
                        }
                        if (TOTALS) {
                            const float t = (zh - mu[u]) * (u ? r2.y : r2.x);
                            t_level += n;
                            t_dist += t * t;
                        }
                    }
                }
                if (TOTALS) {   // 64 float32 terms of the tile are added in float32, then accumulated in float64
                    t_level = __reduce_add_sync(0xffffffffu, t_level);
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) t_dist += __shfl_xor_sync(0xffffffffu, t_dist, o);
                    if (lane == lam - lb) {   // the butterfly left the sums in every lane
                        my_level = t_level;
                        my_dist = t_dist;
                    }
                }
            }
            if (TOTALS && lb + lane < L) {   // integers (distortion in units of 2^-16): the order of the tiles, which
                long long *wAccI = reinterpret_cast<long long *>(wAcc);   // depends on the claims, does not matter
                wAccI[(lb + lane) * 2 + 0] += my_level;
                wAccI[(lb + lane) * 2 + 1] += (long long)__float2ull_rn(my_dist * 65536.0f);   // 64-coordinate sums: exact to 2^-17
            }
            }

            __syncwarp();
            stage(nxt, slot == 0 ? kStages - 1 : slot - 1);
            slot = slot == kStages - 1 ? 0 : slot + 1;
            q0 = q1;
            q1 = q2;
            q2 = nxt;
        }
        cp_async_wait<0>();
    }

    if (TOTALS) {
        __syncthreads();
        // per-CTA partials, then the last CTA adds the partials of all CTAs in a fixed order (deterministic)
        for (int k = threadIdx.x; k < L * 2; k += kThreads) {
            long long si = 0;
            for (int w = 0; w < kWarps; ++w) si += reinterpret_cast<const long long *>(sAcc)[(size_t)w * L * 2 + k];
            const double s = (k & 1) ? (double)si * (1.0 / 65536.0) : (double)si;
            const int lam = k >> 1;
            double *part = a.partials + ((size_t)lam * kMaxGrid + blockIdx.x) * VBQ_TOTALS;
            if (k & 1) {
                part[3] = s;
            } else {   // raw-length mode: the code length of depth n is n itself; no entropy model on this path
                part[0] = s;
                part[1] = s;
                part[2] = 0.0;
            }
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

template <bool TOTALS, bool OUTS, bool VEC, int T>
static int launch_bisect_sweep(QArgs a, int dev, int sms, cudaStream_t st) {
    a.passes = (a.rows + kTileRows - 1) / kTileRows;
    a.total_units = a.passes * a.n_groups;
    long long gx = (a.total_units + (T / 32) - 1) / (T / 32);
    if (gx > sms) gx = sms;
    if (gx > kMaxGrid) gx = kMaxGrid;
    if (gx < 1) gx = 1;
    const size_t fixed = ((size_t)kPadEntries * VBQ_GROUP + (size_t)(T / 32) * kStages * kTileFloats) * sizeof(float);
    const size_t per_lambda = kPenSlots * sizeof(float) + (TOTALS ? (size_t)(T / 32) * 2 * sizeof(double) : 0);
    int max_l = (int)((220 * 1024 - fixed) / per_lambda);
    max_l &= ~3;   // keeps the accumulators behind the penalty block 16-byte aligned
    if (max_l < 4) return -1;
    auto kern = vbq_bisect_sweep_kernel<TOTALS, OUTS, VEC, T>;
    const int n_lambda = a.n_lambda;
    for (int l0 = 0; l0 < n_lambda; l0 += max_l) {   // lambdas beyond the shared-memory budget are served in chunks
        QArgs b = a;
        b.n_lambda = n_lambda - l0 < max_l ? n_lambda - l0 : max_l;
        b.pen = a.pen + (size_t)l0 * (a.N + 1);
        const size_t oo = (size_t)l0 * (size_t)a.lam_stride;
        if (a.zhat) b.zhat = a.zhat + oo;
        if (a.qidx) b.qidx = a.qidx + oo;
        if (a.level) b.level = a.level + oo;
        if (a.bits) b.bits = a.bits + oo;
        if (a.totals) {
            b.totals = a.totals + (size_t)l0 * VBQ_TOTALS;
            b.partials = a.partials + (size_t)l0 * kMaxGrid * VBQ_TOTALS;
        }
        // round the penalty block up to a multiple of 16 bytes so that the double accumulators behind the staging ring
        // stay 8-byte aligned: kPenSlots * 4 = 48 bytes per lambda is already a multiple of 16
        const size_t smem = fixed + per_lambda * b.n_lambda;
        VBQ_ENSURE_MAX_SMEM(kern, dev);
        CUDA_TRY(launch_pdl(kern, dim3((int)gx, 1), T, smem, st, b));
    }
    return VBQ_OK;
}

// returns -1 when this kernel does not apply (the caller then uses vbq_sweep_kernel), else a VBQ_* status
int vbq_launch_sweep_bisect(const QArgs &a, int dev, int sms, cudaStream_t st) {
    if (a.N > kSmemDepth || a.n_lambda < 2 || a.len || a.em || a.pen_channels != 1) return -1;
    if (a.flags & (VBQ_FLAG_FAST | VBQ_FLAG_REFERENCE_WALK | VBQ_FLAG_BRACKET_WALK)) return -1;
    const bool tot = a.totals != nullptr;
    const bool vec = a.C % 4 == 0 && (((uintptr_t)a.mu | (uintptr_t)a.sigma) & 15) == 0;
    constexpr int T = 768;
    const bool outs = a.zhat || a.qidx || a.level || a.bits;
    if (!tot && !outs) return VBQ_OK;   // nothing requested
    if (vec) {
        if (!outs) return launch_bisect_sweep<true, false, true, T>(a, dev, sms, st);
        return tot ? launch_bisect_sweep<true, true, true, T>(a, dev, sms, st) : launch_bisect_sweep<false, true, true, T>(a, dev, sms, st);
    }
    return tot ? launch_bisect_sweep<true, true, false, T>(a, dev, sms, st) : launch_bisect_sweep<false, true, false, T>(a, dev, sms, st);
}
