// sweep_both.cu — rate-distortion SWEEP for ARBITRARY per-channel penalties (corrected code lengths n + R_lambda[c, n],
// quantizer.py:170-180): all lambdas of a call from one tree walk, like sweep_bisect.cu, with the second bracket end where
// it can win (sm_100a).
//
// Reference behaviour reproduced (paths relative to mandt-lab/vbq): quantizer.py:156-188 builds the 2N+1 candidates
// left_0..left_N, right_1..right_N and the (Lambda, 2N+1, B, C) code lengths, utils.py:387 computes the distortion term of
// every candidate once, utils.py:392-421 loops over `lambs` (score, first argmax, gather), quantizer.py:223-228 looks up the
// sorted index and the entropy-model bits.  Here one walk per coordinate leaves the squared scaled distance of ONE
// candidate per depth in registers: the path node, or — at the depths where the penalties of some lambda and some channel
// of the group dip below an earlier depth's (quantize_tma.cuh, iteration_both, explains why only there) — the nearer of the
// path node and its in-level neighbour on the side of mu.  Every lambda then costs one packed add and one LOP3 per key, the
// 3-input minimum chain and the VIADDMNMX gap chain with this thread's channel's penalties (a [Lambda][16][24] table of
// penalties and code lengths in shared memory).  Which end it is gets decided for the winning depth only, and only where that
// lambda's own mask says the neighbour can win: the left end unless the right end is strictly nearer AND the key of the left
// end lies beyond the guard band (the left end comes first in the reference's candidate order, so the right end needs a
// strictly better float32 score).  A ranking that is not certified for some lambda is redone for that lambda by
// `reference_search` (literal two-ended walk, IEEE float32).  Entropy-model bits: summed in the kernel (loads consumed one
// lambda later than issued) when only totals are wanted; as an output they are left to em_gather_kernel
// (quantize_tma_both.cu) through the winner's heap index parked in the entropy-model plane.  max_bits_per_coord <= 10,
// C % 4 == 0, 16-byte aligned inputs, finite non-negative penalties known on the host; other calls use one both-ends launch
// per lambda or vbq_sweep_kernel.
#include <stdlib.h>

#include "bisect.cuh"

constexpr int kPenSlots = 24;   // per (lambda, channel): penalties of depths 0..10 (three float4), then the code lengths of depths 0..10
constexpr int kAccPerLambda = 4;

// OUTS: per-coordinate outputs are requested (otherwise the call returns only the per-lambda totals); EM: entropy-model bits
// (an output and / or column 2 of the totals)
template <bool TOTALS, bool OUTS, bool EM, int kThreads>
__global__ void __launch_bounds__(kThreads, 1) vbq_both_sweep_kernel(const QArgs a) {
    constexpr bool VEC = true;
    constexpr int U = 2;
    constexpr int kWarps = kThreads / 32;
    extern __shared__ __align__(16) float smem[];
    const int N = a.N;                                  // <= kSmemDepth
    const int L = a.n_lambda;
    float *sT = smem;                                   // [kPadEntries][16] code points of depths 0..10
    float *sPenL = sT + kPadEntries * VBQ_GROUP;        // [L][16][kPenSlots]: pen_0..pen_10 of the group's channels (+inf beyond N)
    float *sStage = sPenL + (size_t)L * VBQ_GROUP * kPenSlots;   // [kWarps][kStages][kTileFloats] staging rings
    long long *sAcc = reinterpret_cast<long long *>(sStage + kWarps * kStages * kTileFloats);   // [kWarps][L][4], integers
    unsigned *sMask = reinterpret_cast<unsigned *>(sAcc + (TOTALS ? (size_t)kWarps * L * kAccPerLambda : 0));   // [L]
    __shared__ int sNext, sBig;   // sBig: some code length exceeds 512 bits (the integer warp sums below would overflow)
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
    long long *wAcc = sAcc + (size_t)warp * L * kAccPerLambda;

    if (TOTALS) {
        for (int k = threadIdx.x; k < kWarps * L * kAccPerLambda; k += kThreads) sAcc[k] = 0;
    }
    if (threadIdx.x == 0) sBig = 0;
    __syncthreads();
    pdl_wait();   // launched with programmatic stream serialization: nothing global is touched before this point
    long long unit = u0;
    while (unit < u1) {
        const int g = (int)(unit / tpg);
        const int t0 = (int)(unit - (long long)g * tpg);
        const int n_tiles = (int)min(tpg - t0, u1 - unit);
        unit += n_tiles;

        __syncthreads();                     // every warp has left the previous segment
        if (threadIdx.x == 0) sNext = 0;
        // the penalties of the group's channels for every lambda (quantizer.py:170-180: lambda * (n + R_lambda[c, n]))
        for (int k = threadIdx.x; k < L * VBQ_GROUP * kPenSlots; k += kThreads) {
            const int n = k % 12, what = (k / 12) & 1, j = (k / kPenSlots) % VBQ_GROUP, lam = k / (kPenSlots * VBQ_GROUP);
            const int ch = a.pen_channels == 1 ? 0 : min(g * VBQ_GROUP + j, C - 1);
            const size_t src = ((size_t)lam * a.pen_channels + ch) * (N + 1) + n;
            float v = what ? (float)n : CUDART_INF_F;          // no length table: raw code lengths
            if (n <= N) v = what ? (a.len ? __ldg(a.len + src) : (float)n) : __ldg(a.pen + src);
            sPenL[k] = v;
            if (what && !(v <= 512.0f)) sBig = 1;
        }
        __syncthreads();
        // depths at which the in-level neighbour can win for some lambda and some channel of the group: pen_n below the
        // running maximum of the shallower depths (warp-uniform; every warp computes the same mask)
        // sMask[lam]: the same per lambda (the walk serves all lambdas and uses the union; the decision between the two ends
        // of a winning depth uses the lambda's own mask)
        const bool big = sBig != 0;
        unsigned pen0 = (unsigned)__cvta_generic_to_shared(sPenL) + (unsigned)col * (kPenSlots * 4);   // this channel, lambda 0
        unsigned mask0 = (unsigned)__cvta_generic_to_shared(sMask);
        asm volatile("" : "+r"(pen0), "+r"(mask0));   // new values per segment as far as the compiler knows
        unsigned umask = 0;
        for (int lam = 0; lam < L; ++lam) {
            const float *pr = sPenL + (lam * VBQ_GROUP + col) * kPenSlots;
            unsigned below = 0;
            float pmax = pr[0];
            for (int n = 1; n <= N; ++n) {
                below |= pr[n] < pmax ? 1u << n : 0u;
                pmax = fmaxf(pmax, pr[n]);
            }
            below = (a.flags & VBQ_FLAG_NEIGHBOUR_EVERY_DEPTH) ? 0x7feu : __reduce_or_sync(0xffffffffu, below);
            if (threadIdx.x == 0) sMask[lam] = below;
            umask |= below;
        }
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
                unsigned addr[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    addr[u] = (unsigned)(imad((int)K[u], kRowStrideBytes, pbi) + 2 * n * kRowStrideBytes);
                    z[u] = lds_pure(addr[u]);
                }
                float2 d = __fadd2_rn(make_float2(z[0], z[1]), nmu2);
                K[0] = __funnelshift_l(__float_as_uint(d.x), K[0], 1);
                K[1] = __funnelshift_l(__float_as_uint(d.y), K[1], 1);
                if ((umask >> n) & 1u) {   // the nearer of the path node and its neighbour on the side of mu (pads repeat the level ends)
                    const float zn0 = lds_pure(addr[0] + ((K[0] & 1u) ? kRowStrideBytes : -kRowStrideBytes));
                    const float zn1 = lds_pure(addr[1] + ((K[1] & 1u) ? kRowStrideBytes : -kRowStrideBytes));
                    const float2 dn = __fadd2_rn(make_float2(zn0, zn1), nmu2);
                    d = make_float2(fminf(fabsf(d.x), fabsf(dn.x)), fminf(fabsf(d.y), fabsf(dn.y)));
                }
                const float2 t = __fmul2_rn(d, r2);
                t2[n] = __fmul2_rn(t, t);
            }
            const int kd = N + 1;   // depth of the node K points at

            // ---- every lambda from the registers ----------------------------------------------------------------
            // lane j of the warp keeps the tile's sums of lambda lb + j; they reach shared memory once per 32 lambdas
            for (int lb = 0; lb < L; lb += 32) {
            int my_level = 0;
            unsigned long long my_bits = 0, my_em = 0;   // units of 2^-16
            float my_dist = 0.0f;
            const int lend = min(L, lb + 32);
            // entropy-model bits (quantizer.py:226-228): one L2 sector per coordinate and lambda.  The loads of a lambda are
            // consumed (stored, summed) after the ranking of the NEXT lambda, which hides their latency.
            float em_pend[U] = {0.0f, 0.0f};
            int em_lam = -1;
            auto retire_em = [&]() {
                if (em_lam < 0) return;
                float t_em = 0.0f;
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (ok[u]) {
                        if (OUTS && a.em_bits) __stcs(a.em_bits + (size_t)em_lam * (size_t)a.lam_stride + off + u * u_step, em_pend[u]);
                        t_em += em_pend[u];
                    }
                if (TOTALS) {
                    // entropy-model bits are -log2 of frequencies: the saturating conversion only matters for garbage tables
                    const unsigned w_em = __reduce_add_sync(0xffffffffu, __float2uint_rn(fminf(t_em, 1024.0f) * 65536.0f));
                    if (lane == em_lam - lb) my_em = w_em;
                }
                em_lam = -1;
            };
            size_t o_lam = (size_t)lb * (size_t)a.lam_stride + off;   // this thread's first output element of lambda lam
            unsigned pen_a = pen0 + (unsigned)lb * (VBQ_GROUP * kPenSlots * 4);   // this channel's penalties, then code lengths
            for (int lam = lb; lam < lend; ++lam, o_lam += (size_t)a.lam_stride, pen_a += VBQ_GROUP * kPenSlots * 4) {
                const unsigned lmask = __float_as_uint(lds_pure(mask0 + 4u * (unsigned)lam));
                const float4 pa = lds128_pure(pen_a), pb = lds128_pure(pen_a + 16), pc = lds128_pure(pen_a + 32);
                const float pen[kSmemDepth + 1] = {pa.x, pa.y, pa.z, pa.w, pb.x, pb.y, pb.z, pb.w, pc.x, pc.y, pc.z};
                unsigned key[U][kSmemDepth + 1];
#pragma unroll
                for (int n = 0; n <= kSmemDepth; ++n) {
                    const float2 A = __fadd2_rn(t2[n], make_float2(pen[n], pen[n]));
                    key[0][n] = (__float_as_uint(A.x) & kmask) | (unsigned)n;
                    key[1][n] = (__float_as_uint(A.y) & kmask) | (unsigned)n;
                }
                int wn[U], wP[U];   // winning depth, heap index 2^n + i of the winner
                unsigned mkey[U], gap[U];
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
                    gap[u] = min(g0, g1);
                    mkey[u] = m;
                    wn[u] = (int)(m & 15u);
                    wP[u] = (int)(K[u] >> (kd - wn[u]));
                }
                // The depth is certified if the gap exceeds the guard.  Where the neighbour can win, the two bracket ends of
                // the winning depth (same penalty) are told apart by their distances: the left end comes first in the
                // reference's candidate order (quantizer.py:183, utils.py:401), so the right end wins only with a strictly
                // better float32 score — certified through the key of the left end, like the gap between depths.
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int n = wn[u];
                    if (gap[u] > kKeyGuard && ((lmask >> n) & 1u)) {
                        const int fg = wP[u] - (1 << n) + (int)((K[u] >> (kd - n - 1)) & 1u);
                        const int il = clamp_index(fg, n, N, false), ir = clamp_index(fg, n, N, true);
                        const int lvl = imad(n, 2 * kRowStrideBytes, pbi) + (kRowStrideBytes << n);   // entry_of(n, 0)
                        const float dl = fabsf(lds_pure((unsigned)imad(il, kRowStrideBytes, lvl)) - mu[u]);
                        const float dr = fabsf(lds_pure((unsigned)imad(ir, kRowStrideBytes, lvl)) - mu[u]);
                        int iw = il;
                        if (dr < dl) {
                            const float tf = dl * (u ? r2.y : r2.x);
                            const int dfar = (int)(__float_as_uint(__fmaf_rn(tf, tf, lds_pure(pen_a + 4u * (unsigned)n))) & kmask) - (int)(mkey[u] & kmask);
                            if (dfar > (int)kKeyGuard) iw = ir;
                            else gap[u] = 0u;
                        }
                        wP[u] = (1 << n) + iw;
                    }
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (gap[u] <= kKeyGuard) {   // not certified for this lambda: literal search
                        const int r = reference_search(sTc, sPenL + (lam * VBQ_GROUP + col) * kPenSlots, 1, mu[u], sg[u], N);
                        wn[u] = r >> 24;
                        wP[u] = (1 << wn[u]) + (r & 0xffffff);
                    }
                }
                int t_level = 0, qv[U] = {0, 0};
                float t_bits = 0.0f, t_dist = 0.0f;
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int n = wn[u], Pn = wP[u];
                    if ((TOTALS || OUTS) && ok[u]) {
                        const float zh = lds_pure((unsigned)(imad(n, 2 * kRowStrideBytes, imad(Pn, kRowStrideBytes, pbi))));
                        const float len = lds_pure(pen_a + 48u + 4u * (unsigned)n);
                        const int q = ((2 * Pn + 1) << (N - n)) - (2 << N) - 1;
                        qv[u] = q;
                        if (OUTS) {
                            const size_t o = o_lam + u * u_step;
                            // streaming stores: the outputs of a sweep are many times the L2 and must not evict the
                            // entropy-model tables that every tile gathers from
                            if (a.zhat) __stcs(a.zhat + o, zh);
                            if (a.qidx) __stcs(a.qidx + o, q);
                            if (a.level) __stcs(a.level + o, n);
                            if (a.bits) __stcs(a.bits + o, len);
                            if (a.kout) __stcs(a.em_bits + o, __int_as_float(Pn));   // for em_gather_kernel
                        }
                        if (TOTALS) {
                            const float t = (zh - mu[u]) * (u ? r2.y : r2.x);
                            t_level += n;
                            t_bits += len;
                            t_dist += t * t;
                        }
                    }
                }
                if (EM) {
                    retire_em();   // the previous lambda's loads have long arrived
#pragma unroll
                    for (int u = 0; u < U; ++u) em_pend[u] = ok[u] ? __ldg(a.em + ((size_t)lam * C + cc) * a.Q + qv[u]) : 0.0f;
                    em_lam = lam;
                }
                if (TOTALS) {
                    // code lengths: this thread's two terms in units of 2^-16, then an integer warp sum (one REDUX); the
                    // distortion (unbounded) keeps the float32 butterfly over the 64 terms of the tile
                    t_level = __reduce_add_sync(0xffffffffu, t_level);
                    unsigned long long w_bits;
                    if (!big) w_bits = __reduce_add_sync(0xffffffffu, __float2uint_rn(t_bits * 65536.0f));
                    else {   // absurdly long codes: float32 butterfly like the distortion
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) t_bits += __shfl_xor_sync(0xffffffffu, t_bits, o);
                        w_bits = __float2ull_rn(t_bits * 65536.0f);
                    }
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) t_dist += __shfl_xor_sync(0xffffffffu, t_dist, o);
                    if (lane == lam - lb) {   // the sums are in every lane
                        my_level = t_level;
                        my_bits = w_bits;
                        my_dist = t_dist;
                    }
                }
            }
            if (EM) retire_em();
            if (TOTALS && lb + lane < L) {   // integers (units of 2^-16): the order of the tiles, which depends on the claims,
                long long *w4 = wAcc + (size_t)(lb + lane) * kAccPerLambda;   // does not matter
                w4[0] += my_level;
                w4[1] += (long long)my_bits;
                w4[2] += (long long)my_em;
                w4[3] += (long long)__float2ull_rn(my_dist * 65536.0f);   // 64-coordinate sums: exact to 2^-17
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
        for (int k = threadIdx.x; k < L * kAccPerLambda; k += kThreads) {
            long long si = 0;
            for (int w = 0; w < kWarps; ++w) si += sAcc[(size_t)w * L * kAccPerLambda + k];
            const int lam = k / kAccPerLambda, t = k % kAccPerLambda;
            a.partials[((size_t)lam * kMaxGrid + blockIdx.x) * VBQ_TOTALS + t] = t == 0 ? (double)si : (double)si * (1.0 / 65536.0);
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

template <bool TOTALS, bool OUTS, bool EM, int T>
static int launch_both_sweep(QArgs a, int dev, int sms, cudaStream_t st) {
    a.passes = (a.rows + kTileRows - 1) / kTileRows;
    a.total_units = a.passes * a.n_groups;
    long long gx = (a.total_units + (T / 32) - 1) / (T / 32);
    if (gx > sms) gx = sms;
    if (gx > kMaxGrid) gx = kMaxGrid;
    if (gx < 1) gx = 1;
    const size_t fixed = ((size_t)kPadEntries * VBQ_GROUP + (size_t)(T / 32) * kStages * kTileFloats) * sizeof(float);
    const size_t per_lambda = (size_t)VBQ_GROUP * kPenSlots * sizeof(float) + sizeof(unsigned) +
                              (TOTALS ? (size_t)(T / 32) * kAccPerLambda * sizeof(long long) : 0);
    int max_l = (int)((220 * 1024 - fixed) / per_lambda);
    if (max_l < 2) return -1;
    auto kern = vbq_both_sweep_kernel<TOTALS, OUTS, EM, T>;
    const int n_lambda = a.n_lambda;
    for (int l0 = 0; l0 < n_lambda; l0 += max_l) {   // lambdas beyond the shared-memory budget are served in chunks
        QArgs b = a;
        b.n_lambda = n_lambda - l0 < max_l ? n_lambda - l0 : max_l;
        b.pen = a.pen + (size_t)l0 * a.pen_channels * (a.N + 1);
        if (a.len) b.len = a.len + (size_t)l0 * a.pen_channels * (a.N + 1);
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
        // 1536 bytes of penalties and code lengths per lambda: the 8-byte accumulators behind the staging ring stay aligned
        const size_t smem = fixed + per_lambda * b.n_lambda;
        VBQ_ENSURE_MAX_SMEM(kern, dev);
        CUDA_TRY(launch_pdl(kern, dim3((int)gx, 1), T, smem, st, b));
    }
    return VBQ_OK;
}

// returns -1 when this kernel does not apply (the caller then launches the both-ends kernel once per lambda or uses
// vbq_sweep_kernel), else a VBQ_* status
int vbq_launch_sweep_both(const QArgs &a, int dev, int sms, cudaStream_t st) {
    if (a.N > kSmemDepth || a.n_lambda < 2 || !a.h_pen) return -1;
    if (a.flags & (VBQ_FLAG_FAST | VBQ_FLAG_REFERENCE_WALK | VBQ_FLAG_BRACKET_WALK | VBQ_FLAG_NO_TMA)) return -1;
    if (a.C % 4 != 0 || (((uintptr_t)a.mu | (uintptr_t)a.sigma) & 15) != 0) return -1;
    if (a.em_bits && !a.em) return -1;
    const size_t n_pen = (size_t)a.n_lambda * a.pen_channels * (a.N + 1);
    for (size_t i = 0; i < n_pen; ++i)   // keys are the bit patterns of non-negative floats
        if (!(a.h_pen[i] >= 0.0f && a.h_pen[i] < 3.0e38f)) return -1;
    const bool tot = a.totals != nullptr, em = a.em != nullptr;
    constexpr int T = 768;
    const bool outs = a.zhat || a.qidx || a.level || a.bits || a.em_bits;
    if (!tot && !outs) return VBQ_OK;   // nothing requested
    // Entropy-model bits as an OUTPUT: gathering them here costs an L2 sector per coordinate and lambda while the output
    // stream of the sweep keeps evicting the tables (measured 1.64 ms for 16 lambdas on the Kodak batch); instead the
    // entropy-model planes receive the winners' heap indices and em_gather_kernel (quantize_tma_both.cu) replaces them in all
    // lambda planes by the table entries from shared memory.
    static const bool in_kernel = getenv("VBQ_EM_IN_KERNEL") != nullptr;
    if (em && a.em_bits && !in_kernel && a.N == kSmemDepth && a.C % 4 == 0 && a.n_groups <= 2 * kMaxGrid &&
        a.n_lambda <= 65535 &&   // the conditions of vbq_launch_em_gather
        (((uintptr_t)a.em_bits | (uintptr_t)a.em) & 15) == 0) {
        QArgs b = a;
        b.em = nullptr;   // no gather in the sweep kernel: the entropy-model planes receive the heap indices
        b.kout = 1;
        RETURN_IF(tot ? (launch_both_sweep<true, true, false, T>(b, dev, sms, st)) : (launch_both_sweep<false, true, false, T>(b, dev, sms, st)));
        return vbq_launch_em_gather(a, dev, sms, st);
    }
    if (!outs) return em ? launch_both_sweep<true, false, true, T>(a, dev, sms, st) : launch_both_sweep<true, false, false, T>(a, dev, sms, st);
    if (tot) return em ? launch_both_sweep<true, true, true, T>(a, dev, sms, st) : launch_both_sweep<true, true, false, T>(a, dev, sms, st);
    return em ? launch_both_sweep<false, true, true, T>(a, dev, sms, st) : launch_both_sweep<false, true, false, T>(a, dev, sms, st);
}
