// quantize_bisect.cu — the single-lambda rate-distortion search as a certified BISECTION (sm_100a).
//
// Reference behaviour reproduced (paths relative to mandt-lab/vbq): the same as quantize.cu —
//   img-compression/quantizer.py:65-80, :156-188   bracket of mu at every bit depth, candidates left_0..left_N,
//                                                  right_1..right_N with code length n
//   img-compression/utils.py:318-320, :392-415     score fl(fl(-0.5 fl(t^2)) - fl(lambda n)), t = fl(fl(z-mu)/sigma),
//                                                  first argmax
//
// Why one candidate per depth is enough.  The code points of depths <= n form the nested dyadic grid
// G_n = {F^-1(k 2^-(n+1))}.  Walking the tree keeps the open interval (lo, hi) of G_(n-1) that contains mu; the PATH
// NODE z_n is the only depth-n point inside it.  The reference's depth-n bracket is {z_n, z'} where z' is the next
// depth-n point beyond lo or hi — or z_n itself / the clipped edge point when there is none.  z' lies beyond a bracket
// end `a` that (i) is a path node of a shallower depth m < n, (ii) is at least as close to mu, (iii) has
// pen_m <= pen_n when the penalties are non-decreasing in depth, and (iv) precedes z' in the reference's candidate
// order (same side, smaller depth).  Every float32 operation of the score is monotone, so score(z') <= score(a) and
// z' can never be the first maximiser.  Hence the winner is always one of the N+1 path nodes: one shared-memory load,
// one compare and one score per depth — the neighbour load, the nearer-end selection and the left/right decision of
// the bracket walk (quantize_kernel.cuh) disappear.
//
// Certified approximate scoring.  Only the IDENTITY of the winner is returned, so the path nodes are ranked with a
// cheap loss  A_n = fma(t, t, pen_n),  t = (z_n - mu) * (sqrt(1/2) / sigma)  (3 packed f32x2 instructions per two
// coordinates) instead of the 6-instruction IEEE-division chain.  A_n and the reference's -score E_n are both
// non-negative floats that differ by < 15 float32 roundings (error analysis in DESIGN.md §4), i.e. their bit patterns
// differ by < 30 as integers.  The depth is embedded in the 4 low bits of the pattern (key_n); the winner is the
// integer minimum (VIMNMX3), and a second pass (VIADDMNMX) measures the gap to the runner-up.  If the gap exceeds
// kKeyGuard = 192 > 2*(30+15) the reference's float32 scores are strictly ordered the same way and the result is
// certified identical; otherwise (3-6 coordinates in 10^5 on Kodak-shaped inputs), or when the penalties are not non-decreasing and
// non-negative, the coordinate is redone by `reference_search`, the literal two-ended walk with IEEE arithmetic.
#include <stdlib.h>

#include "bisect.cuh"

// NT > 0: max_bits_per_coord == NT at compile time; NT == 0: runtime depth (<= kSmemDepth).
// OUT >= 0: the set of requested outputs (bit 0 zhat, 1 qidx, 2 level, 3 bits) is known at compile time; OUT < 0: runtime.
// VEC: C % 4 == 0 and 16-byte aligned latents: a warp stages its tile (256 B of mu, 256 B of sigma) with ONE 16-byte
// cp.async per lane; otherwise every thread copies its own two coordinates with 4-byte cp.async.
// NT < 0 (DEEP): max_bits_per_coord up to VBQ_MAX_DEPTH at run time; the path nodes of depths 11..N come from the
// heap-order table in global memory (one 4-byte gather per depth; the bracket walk needs up to three), the depth takes
// 5 key bits instead of 4.
template <bool PRUNE, bool TOTALS, int NT, int OUT, bool VEC, int kThreads>
__global__ void __launch_bounds__(kThreads, 1) vbq_bisect_kernel(const QArgs a) {
    constexpr int U = 2, P = 1;
    constexpr bool DEEP = NT < 0;
    constexpr int kKeys = DEEP ? VBQ_MAX_DEPTH + 1 : kSmemDepth + 1;   // candidates (depths) per coordinate
    constexpr unsigned kDepthBits = DEEP ? 31u : 15u;                   // low key bits that hold the depth
    extern __shared__ __align__(16) float smem[];
    float *sT = smem;                                   // [kPadEntries][16] code points of depths 0..10
    float *sPen = sT + kPadEntries * VBQ_GROUP;         // [kKeys][16] penalties (+inf beyond N)
    float *sStage = sPen + kKeys * VBQ_GROUP;           // [kWarps][kStages][kTileFloats] staging rings
    __shared__ double sRed[VBQ_TOTALS][kMaxThreads / 32];
    __shared__ unsigned sGuard[VBQ_GROUP];
    __shared__ int sNext;                               // next unclaimed tile of the current segment
    __shared__ bool sLast;

    const int N = NT > 0 ? NT : a.N;
    const int lam = blockIdx.y;
    const unsigned outm = OUT >= 0 ? (unsigned)OUT : (a.outm & 15u);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col = lane & (VBQ_GROUP - 1);
    const int par = lane >> 4;                          // row parity inside the tile
    const bool logvar = (a.flags & VBQ_FLAG_LOGVAR) != 0;
    const int C = a.C;
    const int rows = (int)a.rows;                       // the host splits calls so that rows*C < 2^29
    const long long tpg = a.passes;                     // tiles per group = ceil(rows / 4)
    const long long vtotal = (tpg + kSwitchTiles) * a.n_groups;
    const long long u0 = span_cut(vtotal * blockIdx.x / gridDim.x, tpg, a.n_groups);
    const long long u1 = span_cut(vtotal * (blockIdx.x + 1) / gridDim.x, tpg, a.n_groups);
    const size_t lam_off = (size_t)lam * (size_t)a.lam_stride;
    // shared-memory byte address of padded entry (n, i) of this thread's channel = pbi + 64*K + 128*n, K = 2^n + i
    // (entry_of(n, i) = K + 2n): K is the 1-based heap index of the node, children 2K and 2K+1
    const int pbi = (int)__cvta_generic_to_shared(sT + col);
    const float *sTc = sT + col;
    const unsigned kmask = a.keymask;                   // 0xfffffff0 as a runtime value: stays in one register
    float *wStage = sStage + warp * (kStages * kTileFloats);
    const float *myStage = wStage + par * VBQ_GROUP + col;   // + slot*kTileFloats + arr*64 + u*32

    Acc128 acc_dist = {0, 0};   // distortion terms in units of 2^-24: an integer sum does not depend on which warp claimed
                                // which tile
    int acc_level = 0;   // < 2^31: at most 2^29 coordinates per launch, depth <= 10
    pdl_wait();   // launched with programmatic stream serialization: nothing global is touched before this point
#ifdef VBQ_TRACE
    unsigned long long tr_t0 = 0, tr_t1 = 0, tr_t2 = 0;
    int tr_segs = 0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_t0));
    const long long tr_c0 = clock64();
#endif

    long long unit = u0;
    while (unit < u1) {
#ifdef VBQ_TRACE
        ++tr_segs;
#endif
        // ---- segment: a run of tiles inside one 16-channel group -----------------------------------------------
        const int g = (int)(unit / tpg);
        const int t0 = (int)(unit - (long long)g * tpg);
        const int n_tiles = (int)min(tpg - t0, u1 - unit);   // tiles t0 .. t0 + n_tiles - 1 of group g
        unit += n_tiles;

        __syncthreads();                     // every warp has left the previous segment
        if (threadIdx.x == 0) sNext = 0;
        __syncthreads();
        const int c = g * VBQ_GROUP + col;
        const bool c_ok = c < C;
        const int cc = min(c, C - 1);
        // element offset of this thread's first coordinate inside tile 0 of the segment; tile j adds j * 4C
        const unsigned thr_off = (unsigned)(t0 * kTileRows + par) * (unsigned)C + (unsigned)cc;
        const unsigned tile_step = (unsigned)(kTileRows * C), u_step = (unsigned)(2 * C);
        const int seg_row0 = t0 * kTileRows;
        float *zhat_c = a.zhat ? a.zhat + lam_off : nullptr;
        int *qidx_c = a.qidx ? a.qidx + lam_off : nullptr;
        int *level_c = a.level ? a.level + lam_off : nullptr;
        float *bits_c = a.bits ? a.bits + lam_off : nullptr;
        // tiles below full_tiles have all 4 rows inside the matrix; a group with 16 real channels needs no predicates
        const bool group_full = g * VBQ_GROUP + VBQ_GROUP <= C;
        const int full_tiles = group_full ? min(n_tiles, (rows - seg_row0) / kTileRows) : 0;

        // producer role of this lane.  VEC: array (lane>>4), tile row ((lane>>2)&3), 16-byte chunk (lane&3)
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
        int q0 = claim(), q1 = claim(), q2 = claim();   // tiles in flight (kStages - 1 = 3)
        static_assert(kStages == 4, "the claim queue below holds kStages - 1 = 3 tiles");
        stage(q0, 0);
        stage(q1, 1);
        stage(q2, 2);
        int slot = 0;

        // the group's tree and penalties, while the first tiles are in flight
        {
            const float4 *src = reinterpret_cast<const float4 *>(a.packed + (size_t)g * kPadEntries * VBQ_GROUP);
            float4 *dst = reinterpret_cast<float4 *>(sT);
            for (int k = threadIdx.x; k < kPadEntries * (VBQ_GROUP / 4); k += kThreads) dst[k] = __ldg(src + k);
            if (threadIdx.x < VBQ_GROUP) {
                const int j = threadIdx.x;
                const int cj = min(g * VBQ_GROUP + j, C - 1);
                const size_t po = ((size_t)lam * a.pen_channels + (a.pen_channels == 1 ? 0 : cj)) * (N + 1);
                float prev = 0.0f;
                bool mono = true;   // certified ranking needs 0 <= pen_0 <= pen_1 <= ... (false for NaN)
                for (int n = 0; n < kKeys; ++n) {
                    const float p = n <= N ? a.pen[po + n] : CUDART_INF_F;
                    mono = mono && (p >= prev);
                    prev = p;
                    sPen[n * VBQ_GROUP + j] = p;
                }
                sGuard[j] = mono ? kKeyGuard : 0xffffffffu;   // 0xffffffff: every coordinate takes the slow path
            }
        }
        __syncthreads();
        float pen[kKeys];
#pragma unroll
        for (int n = 0; n < kKeys; ++n) pen[n] = sPen[n * VBQ_GROUP + col];
        const float *gT = a.table + (size_t)cc * a.Q - 1;   // DEEP: heap index K (1-based) -> gT[K]
        const unsigned guard = sGuard[col];
        const float z0 = sTc[entry_of(0, 0) * VBQ_GROUP];

        // one tile: U coordinates of this thread (tile rows par and 2 + par); CHECK = bounds must be tested
        auto iteration = [&](auto check_tag, const int tile) {
            constexpr bool CHECK = decltype(check_tag)::value;
            const int row = seg_row0 + tile * kTileRows + par;          // row of coordinate u = 0
            const unsigned off = thr_off + (unsigned)tile * tile_step;
            float mu[U], sg[U];
            float2 nmu2[P], r2[P];   // r2 = sqrt(1/2)/sigma
            bool ok[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                ok[u] = !CHECK || (c_ok && row + 2 * u < rows);
                mu[u] = ok[u] ? myStage[slot * kTileFloats + u * 2 * VBQ_GROUP] : 0.0f;
                float s = ok[u] ? myStage[slot * kTileFloats + kTileRows * VBQ_GROUP + u * 2 * VBQ_GROUP] : 1.0f;
                if (logvar) s = sigma_of_logvar(s);
                sg[u] = s;
            }
#pragma unroll
            for (int k = 0; k < P; ++k) {
                nmu2[k] = make_float2(-mu[2 * k], -mu[2 * k + 1]);
                r2[k] = __fmul2_rn(make_float2(rcp_approx(sg[2 * k]), rcp_approx(sg[2 * k + 1])),
                                   make_float2(0.70710678f, 0.70710678f));
            }

            unsigned key[U][kKeys];
            unsigned K[U];   // 1-based heap index of the path node at the current depth
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int n = 0; n < kKeys; ++n) key[u][n] = (0x7fffffffu & ~kDepthBits) | (unsigned)n;

            // ---- depth 0: the median ---------------------------------------------------------------------
#pragma unroll
            for (int k = 0; k < P; ++k) {
                const float2 d = __fadd2_rn(make_float2(z0, z0), nmu2[k]);
                const float2 t = __fmul2_rn(d, r2[k]);
                const float2 A = __ffma2_rn(t, t, make_float2(pen[0], pen[0]));
                key[2 * k][0] = make_key<0>(A.x, kmask);
                key[2 * k + 1][0] = make_key<0>(A.y, kmask);
                K[2 * k] = __funnelshift_l(__float_as_uint(d.x), 1u, 1);       // 2 + (mu > z0)
                K[2 * k + 1] = __funnelshift_l(__float_as_uint(d.y), 1u, 1);
            }
            int m_done = 0;   // deepest level scored (warp-uniform)

            bool alive[U];            // DEEP: the coordinate still gathers from the global-memory depths
            unsigned run_deep[U];     // DEEP: minimum of its keys so far
#pragma unroll
            for (int u = 0; u < U; ++u) { alive[u] = true; run_deep[u] = 0xffffffffu; }
            auto deep_seed = [&](int u) -> unsigned {   // minimum over the shared-memory depths 0..kSmemDepth
                unsigned m = key[u][0];
#pragma unroll
                for (int j = 1; j <= kSmemDepth; ++j) m = min(m, key[u][j]);
                return m;
            };
            // ---- depths 1..N, fully unrolled -------------------------------------------------------------
            auto depth = [&](auto n_tag) {
                constexpr int n = decltype(n_tag)::value;
                float z[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (n <= kSmemDepth) {
                        z[u] = lds_pure((unsigned)(imad((int)K[u], kRowStrideBytes, pbi) + 2 * n * kRowStrideBytes));
                    } else {
                        // Global-memory depths: a coordinate whose best key so far is more than the guard below the key of
                        // pen_n cannot be won, or brought within the guard, by any deeper candidate (sound, like the
                        // warp-wide early exit, but per coordinate): it stops gathering.  The gathers are the cost of
                        // these depths (one 32-byte sector each), so this is what lambda >= 0.1 or so runs on.
                        run_deep[u] = min(run_deep[u], n == kSmemDepth + 1 ? deep_seed(u) : key[u][n - 1]);
                        const unsigned floor_key = __float_as_uint(pen[n]) & kmask;
                        alive[u] = alive[u] && !(guard == kKeyGuard && floor_key > kKeyGuard + 32u &&
                                                 run_deep[u] < floor_key - (kKeyGuard + 32u));
                        z[u] = alive[u] ? __ldg(gT + K[u]) : CUDART_INF_F;
                    }
                }
#pragma unroll
                for (int k = 0; k < P; ++k) {
                    const float2 d = __fadd2_rn(make_float2(z[2 * k], z[2 * k + 1]), nmu2[k]);
                    if (!(NT > 0 && n == NT)) {   // the branch of the deepest compile-time depth is never used
                        K[2 * k] = __funnelshift_l(__float_as_uint(d.x), K[2 * k], 1);          // 2K + (mu > z)
                        K[2 * k + 1] = __funnelshift_l(__float_as_uint(d.y), K[2 * k + 1], 1);
                    }
                    const float2 t = __fmul2_rn(d, r2[k]);
                    const float2 A = __ffma2_rn(t, t, make_float2(pen[n], pen[n]));
                    key[2 * k][n] = make_key<n>(A.x, kmask);
                    key[2 * k + 1][n] = make_key<n>(A.y, kmask);
                }
                m_done = n;
            };
            unsigned run_min[U];   // PRUNE: minimum of the keys of the depths scored so far, updated at every test
#pragma unroll
            for (int u = 0; u < U; ++u) run_min[u] = 0xffffffffu;
            auto prune_here = [&](auto n_tag) -> bool {
                constexpr int n = decltype(n_tag)::value;
                // sound early exit: every deeper loss is >= pen_n, so once the best key plus the guard is below the
                // key of pen_n no deeper candidate can win or come within the guard.  Tested at depths 3, 6, 9 and
                // before every global-memory depth.
                const unsigned floor_key = __float_as_uint(pen[n]) & kmask;
                bool done = guard == kKeyGuard && floor_key > kKeyGuard + 32u;
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    if (n <= 9) {
                        run_min[u] = __vimin3_u32(run_min[u], key[u][n - 3], key[u][n - 2]);
                        run_min[u] = min(run_min[u], key[u][n - 1]);
                    } else if (n == kSmemDepth + 1) {
                        run_min[u] = __vimin3_u32(run_min[u], key[u][n - 2], key[u][n - 1]);
                    } else {
                        run_min[u] = min(run_min[u], key[u][n - 1]);
                    }
                    done = done && run_min[u] < floor_key - (kKeyGuard + 32u);
                }
                return __all_sync(0xffffffffu, done);
            };
#define VBQ_DEPTH(n_)                                                                                          \
    if constexpr (n_ <= kSmemDepth || DEEP) {                                                                  \
        if ((NT > 0 ? n_ <= NT : n_ <= N) && !stop) {                                                          \
            if (PRUNE && ((n_ <= 9 && n_ % 3 == 0) || n_ > kSmemDepth) &&                                      \
                prune_here(std::integral_constant<int, n_>{}))                                                 \
                stop = true;                                                                                   \
            else                                                                                               \
                depth(std::integral_constant<int, n_>{});                                                      \
        }                                                                                                      \
    }
            bool stop = false;
            VBQ_DEPTH(1) VBQ_DEPTH(2) VBQ_DEPTH(3) VBQ_DEPTH(4) VBQ_DEPTH(5)
            VBQ_DEPTH(6) VBQ_DEPTH(7) VBQ_DEPTH(8) VBQ_DEPTH(9) VBQ_DEPTH(10)
            VBQ_DEPTH(11) VBQ_DEPTH(12) VBQ_DEPTH(13) VBQ_DEPTH(14) VBQ_DEPTH(15)
            VBQ_DEPTH(16) VBQ_DEPTH(17) VBQ_DEPTH(18) VBQ_DEPTH(19) VBQ_DEPTH(20)
#undef VBQ_DEPTH
            static_assert(kSmemDepth == 10 && VBQ_MAX_DEPTH == 20, "the depth macro lists above cover depths 1..10 and 11..20");
            const int kd = (NT > 0 && m_done == NT) ? NT : m_done + 1;   // depth of the node K points at

            // ---- winner and certificate -----------------------------------------------------------------------
            int wn[U], wP[U];          // winning depth and heap index 2^n + i of the winning path node
            unsigned gapmin = 0xffffffffu;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const unsigned *k_ = key[u];
                unsigned m = k_[0];
#pragma unroll
                for (int n = 1; n + 1 < kKeys; n += 2) m = __vimin3_u32(m, k_[n], k_[n + 1]);
                if (kKeys % 2 == 0) m = min(m, k_[kKeys - 1]);
                const unsigned nm = ~m;   // key + ~m = key - m - 1: 0xffffffff for the winner itself
                unsigned g0 = 0xffffffffu, g1 = 0xffffffffu;   // two chains for instruction-level parallelism
#pragma unroll
                for (int n = 0; n < kKeys; n += 2) g0 = __viaddmin_u32(k_[n], nm, g0);
#pragma unroll
                for (int n = 1; n < kKeys; n += 2) g1 = __viaddmin_u32(k_[n], nm, g1);
                gapmin = __vimin3_u32(gapmin, g0, g1);
                wn[u] = (int)(m & kDepthBits);
                wP[u] = (int)(K[u] >> (kd - wn[u]));
            }
            if (gapmin <= guard) {   // some coordinate is not certified (or penalties not monotone): literal search
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int r = DEEP ? reference_search_deep(sTc, gT + 1, sPen + col, VBQ_GROUP, mu[u], sg[u], N)
                                       : reference_search(sTc, sPen + col, VBQ_GROUP, mu[u], sg[u], N);
                    wn[u] = r >> 24;
                    wP[u] = (1 << wn[u]) + (r & 0xffffff);
                }
            }
            float dist[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int n = wn[u], Pn = wP[u];
                dist[u] = 0.0f;
                if (ok[u]) {
                    const unsigned o = off + u * u_step;
                    // sorted index q = (2i+1) 2^(N-n) - 1 with i = Pn - 2^n:  (2 Pn + 1) 2^(N-n) - 2^(N+1) - 1
                    const int q = ((2 * Pn + 1) << (N - n)) - (2 << N) - 1;
                    if (outm & 2u) qidx_c[o] = q;
                    if (outm & 4u) level_c[o] = n;
                    if (outm & 8u) bits_c[o] = (float)n;
                    if (TOTALS || (outm & 1u)) {
                        float zh;
                        if (DEEP && n > kSmemDepth) zh = __ldg(gT + Pn);
                        else zh = lds_pure((unsigned)(imad(n, 2 * kRowStrideBytes, imad(Pn, kRowStrideBytes, pbi))));
                        if (outm & 1u) zhat_c[o] = zh;
                        if (TOTALS) {
                            const float r1 = u & 1 ? r2[u / 2].y : r2[u / 2].x;
                            const float t = (zh - mu[u]) * r1;
                            acc_level += n;
                            dist[u] = t * t;
                        }
                    }
                }
            }
            if (TOTALS) {   // the float32 terms of this thread's part of a tile, then an exact (integer) sum
                float dsum = dist[0];
#pragma unroll
                for (int u = 1; u < U; ++u) dsum += dist[u];
                acc_dist.add_q24(dsum);
            }
        };

        while (q0 < n_tiles) {
            const int nxt = claim();             // used at the end of the iteration: the atomic's latency is hidden
            cp_async_wait<kStages - 2>();        // tile q0 has landed ...
            __syncwarp();                        // ... for every lane of the warp (the tile is staged cooperatively)
            if (q0 < full_tiles) iteration(std::false_type{}, q0);
            else iteration(std::true_type{}, q0);
            __syncwarp();                        // all lanes have read slot `slot`; (slot + 3) % 4 was read one tile ago
            stage(nxt, slot == 0 ? kStages - 1 : slot - 1);
            slot = slot == kStages - 1 ? 0 : slot + 1;
            q0 = q1;
            q1 = q2;
            q2 = nxt;
        }
        cp_async_wait<0>();
    }

#ifdef VBQ_TRACE
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_t1));
    __syncthreads();
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_t2));
    if (TOTALS && (threadIdx.x & 31) == 0) {   // per warp: start, own end, CTA end, segments, SM id
        unsigned smid;
        asm("mov.u32 %0, %%smid;" : "=r"(smid));
        double *tr = a.partials + (size_t)kMaxGrid * VBQ_TOTALS * a.n_lambda + ((size_t)blockIdx.x * 32 + (threadIdx.x >> 5)) * 5;
        tr[0] = (double)tr_t0; tr[1] = (double)tr_t1; tr[2] = (double)tr_t2; tr[3] = tr_segs + 1e-9 * (double)(clock64() - tr_c0); tr[4] = smid;
    }
#endif
    if (TOTALS) {
        // raw-length mode: the code length of depth n is n itself; no entropy model on this path
        double v[VBQ_TOTALS] = {(double)acc_level, (double)acc_level, 0.0, acc_dist.value()};
        finish_totals<kThreads>(a, lam, v, sRed, &sLast);
    }
}

template <bool PRUNE, bool TOTALS, int NT, int OUT, bool VEC, int T>
static int launch_bisect(QArgs a, int dev, int sms, cudaStream_t st) {
    a.passes = (a.rows + kTileRows - 1) / kTileRows;   // tiles per group
    a.total_units = a.passes * a.n_groups;
    long long gx = (a.total_units + (T / 32) - 1) / (T / 32);   // at least one tile per warp
    if (gx > sms) gx = sms;
    if (gx > kMaxGrid) gx = kMaxGrid;
    if (gx < 1) gx = 1;
    const size_t smem = ((size_t)kPadEntries * VBQ_GROUP + (size_t)(NT < 0 ? VBQ_MAX_DEPTH + 1 : kSmemDepth + 1) * VBQ_GROUP +
                         (size_t)(T / 32) * kStages * kTileFloats) * sizeof(float);
    auto kern = vbq_bisect_kernel<PRUNE, TOTALS, NT, OUT, VEC, T>;
    VBQ_ENSURE_MAX_SMEM(kern, dev);
    CUDA_TRY(launch_pdl(kern, dim3((int)gx, a.n_lambda), T, smem, st, a));
    return VBQ_OK;
}

template <bool PRUNE, bool TOTALS, int NT, int T>
static int launch_bisect3(const QArgs &a, int dev, int sms, cudaStream_t st) {
    // the two output sets the facade and the benchmark ask for are compiled in; anything else tests the mask at run time
    const bool vec = a.C % 4 == 0 && (((uintptr_t)a.mu | (uintptr_t)a.sigma) & 15) == 0;
    if (!vec) return launch_bisect<PRUNE, TOTALS, NT, -1, false, T>(a, dev, sms, st);
    switch (a.outm & 15u) {
        case 2u | 8u: return launch_bisect<PRUNE, TOTALS, NT, 2 | 8, true, T>(a, dev, sms, st);   // sorted index + code length
        case 1u | 4u: return launch_bisect<PRUNE, TOTALS, NT, 1 | 4, true, T>(a, dev, sms, st);   // z_hat + depth
        case 1u: return launch_bisect<PRUNE, TOTALS, NT, 1, true, T>(a, dev, sms, st);            // z_hat (word embeddings)
        default: return launch_bisect<PRUNE, TOTALS, NT, -1, true, T>(a, dev, sms, st);
    }
}

template <bool PRUNE, int T>
static int launch_bisect2(const QArgs &a, int dev, int sms, cudaStream_t st) {
    const bool tot = a.totals != nullptr;
    if (a.N == kSmemDepth)
        return tot ? launch_bisect3<PRUNE, true, kSmemDepth, T>(a, dev, sms, st)
                   : launch_bisect3<PRUNE, false, kSmemDepth, T>(a, dev, sms, st);
    return tot ? launch_bisect3<PRUNE, true, 0, T>(a, dev, sms, st) : launch_bisect3<PRUNE, false, 0, T>(a, dev, sms, st);
}

// raw code lengths (no length table, no entropy model), max_bits_per_coord <= 10; returns -1 if not applicable
int vbq_launch_quantize_bisect(const QArgs &a, int dev, int sms, cudaStream_t st) {
    if (a.len || a.em) return -1;
    const bool prune = !(a.flags & VBQ_FLAG_NO_PRUNE);
    if (a.N > kSmemDepth) {   // deep tables: 512 threads (21 keys and penalties per coordinate pair: > 100 registers)
        QArgs b = a;
        b.keymask = 0xffffffe0u;
        const bool tot = a.totals != nullptr;
        if (prune) return tot ? launch_bisect3<true, true, -1, 512>(b, dev, sms, st) : launch_bisect3<true, false, -1, 512>(b, dev, sms, st);
        return tot ? launch_bisect3<false, true, -1, 512>(b, dev, sms, st) : launch_bisect3<false, false, -1, 512>(b, dev, sms, st);
    }
    // 768 threads (24 warps, 80 registers): measured best of 512 / 640 / 768 / 896
    return prune ? launch_bisect2<true, 768>(a, dev, sms, st) : launch_bisect2<false, 768>(a, dev, sms, st);
}

// Self-test helper (host only, no GPU): the tile range [out[b], out[b+1]) CTA b of a `grid`-CTA launch takes, for
// `rows` rows and C channels — the same span_cut arithmetic the kernels run.
extern "C" int vbq_selftest_span_cuts(long long rows, int C, int grid, long long *out) {
    if (rows < 0 || C < 1 || grid < 1 || !out) return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_selftest_span_cuts: bad argument");
    const long long tpg = (rows + kTileRows - 1) / kTileRows;
    const int n_groups = (C + VBQ_GROUP - 1) / VBQ_GROUP;
    const long long vtotal = (tpg + kSwitchTiles) * n_groups;
    for (int b = 0; b <= grid; ++b) out[b] = span_cut(vtotal * b / grid, tpg, n_groups);
    return VBQ_OK;
}
