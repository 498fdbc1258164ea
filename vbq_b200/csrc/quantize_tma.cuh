// quantize_tma.cuh — the single-lambda certified bisection (quantize_bisect.cu explains the search and why its result is
// the reference's) as a warp-specialised TMA pipeline for sm_100a.
//
// Reference behaviour reproduced (paths relative to mandt-lab/vbq): img-compression/quantizer.py:65-80, :156-188 and
// img-compression/utils.py:318-320, :392-415 — identical results to vbq_bisect_kernel; data movement, the tree walk and
// the work decomposition differ.
//
// Structure.  One persistent CTA per SM: W consumer warps + one producer warp (one elected lane).
//   * tile = W quads; a quad = 4 consecutive rows x the 16 channels of one group = one warp iteration (lane = (row
//     parity, channel), two coordinates per thread: rows parity and parity + 2).  Warp w ALWAYS computes quad w of a
//     tile: nothing is claimed, the thread -> coordinate map is static, so every thread adds its distortion terms in a
//     fixed order and the totals are bit-reproducible.
//   * the producer brings the mu box and the sigma box of a tile (4W rows x 16 channels, 64-byte rows) into one of S
//     shared-memory slots with two cp.async.bulk.tensor loads (TMA) that complete on the slot's `full` mbarrier.  The
//     consumers read their coordinates from the slot, search, and write the two outputs BACK INTO THE SAME slot words
//     (a thread only ever touches its own words); after fence.proxy.async + one arrive per warp on the slot's `done`
//     mbarrier the producer sends the slot to global memory with two TMA stores and refills it.  No consumer thread
//     computes a global address, tests a bound or issues a global load / store for the latents and the outputs.
//   * the CTA's share of the work is a contiguous range of rows (multiples of 4) in (group, row) order; the last tile of
//     a range is cut to its rows: its quads beyond the cut are skipped and its outputs leave through 4-row boxes.
//   * the group's code points arrive by ONE plain bulk copy (UBLKCP, 160 KB) in the "walk tree" layout made by
//     pack_walk_tree_kernel (quantize.cu): heap order (node K has children 2K, 2K+1), every value scaled by 2^24,
//     rows of 16 channels; bit depths 1..7 a second time with rows of 32 words = one private copy per half-warp, so a
//     tree load of these depths touches 32 different banks (the single copy costs two wavefronts per load: the two
//     half-warps of a warp hit the same 16 banks whenever their path bits agree).
//   * the walk runs on the FMA pipe.  The shared-memory BYTE ADDRESS of the path node is kept as a float whose bit
//     pattern is that address — a subnormal number, on which FMA arithmetic is exact integer arithmetic up to 2^24 —:
//     addr' = 2 addr + stride [mu > z] - base  is  fma(step, stride, fma(addr, 2, -base))  with
//     step = sat(-(z - mu) * 2^127) in {0, 1} (FMUL.SAT; the 2^24 scaling of the tree and of mu makes every non-zero
//     difference at least 2^-125, so the product saturates).  The integer pipe (2 cycles per warp instruction, the
//     saturated unit of vbq_bisect_kernel) keeps only the keys, the minimum and the certificate.
#include <math.h>
#include <stdlib.h>

#pragma once
#include "bisect.cuh"
#include "tma.cuh"

constexpr int kQuadRows = 4;
constexpr int kTmaRows = 128;                // rows of a tile = one TMA box per array
constexpr int kSlots = 4;                  // tiles in flight per CTA
constexpr int kDblDepth = 7;               // bit depths 1..kDblDepth also exist as one copy per half-warp
constexpr int kSingleRows = 1 << (kSmemDepth + 1);               // heap index K = 1 .. 2047, row 0 unused
constexpr int kDblRows = (1 << (kDblDepth + 1)) + 1;             // K = 2 .. 255 (rows 0 and 1 unused) + node 256: the "neighbour"
                                                                 // that the both-ends variant reads beyond the last node of depth 7
constexpr int kTmaSmemBytes = 229376 + 128 + 512;   // walk tree + kSlots x (mu box + sigma box) + barriers, descriptors, ticket counter, penalties
constexpr int kWalkFloats = kSingleRows * VBQ_GROUP + kDblRows * 2 * VBQ_GROUP;   // 40992 floats = 160 KB per group
constexpr float kWalkScale = 16777216.0f;                        // 2^24
constexpr float kWalkUnscale = 1.0f / 16777216.0f;
constexpr long long kSwitchRows = 448;     // a second range (new tree) costs a CTA about as much as this many rows

struct TmaMaps {
    CUtensorMap in[2];       // mu, sigma: box of 4W rows
    CUtensorMap out[2][2];   // [first, second output array of the compiled output set][0: 4W-row box, 1: 4-row box]
};

struct UniformPen { float v[kSmemDepth + 1]; };   // warp-uniform penalties as launch constants (constant bank operands)

// first real row position (group-major: position = group * rows4 + row) of virtual position v: every group but the
// first is preceded by kSwitchRows virtual rows — what a second range (drain, new tree, refill) costs the CTA whose
// share crosses the group boundary; the first tree load is the same for every CTA
__host__ __device__ __forceinline__ long long row_cut(long long v, long long rows4, int n_groups) {
    const long long vg = rows4 + kSwitchRows;
    long long g = (v + kSwitchRows) / vg;
    if (g > n_groups) g = n_groups;
    const long long o = v + kSwitchRows - g * vg;
    return g * rows4 + (o > kSwitchRows ? (o - kSwitchRows) & ~3ll : 0);
}

#ifdef VBQ_TRACE   // development: %globaltimer stamps into the workspace behind the partial totals (scripts/trace_tma.py)
__device__ __forceinline__ unsigned long long gtime() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#define TRACE_P(tile, k) do { if ((tile) < 64) tr[8 + (tile) * 4 + (k)] = (double)gtime(); } while (0)
#define TRACE_C(tile, k) do {} while (0)
#else
#define TRACE_P(tile, k) do {} while (0)
#define TRACE_C(tile, k) do {} while (0)
#endif

__device__ __forceinline__ void sts_u32(unsigned addr, unsigned v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void sts_v4(unsigned addr, int x, int y, int z, int w) {
    asm volatile("st.shared.v4.s32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ unsigned lds_u32i(unsigned addr) {
    unsigned v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ int4 lds_v4(unsigned addr) {
    int4 v;
    asm volatile("ld.shared.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}
// lane 0 takes the next ticket of the CTA-wide counter (atom.inc with wrap bound 2^31-1 = a plain increment: for
// atom.add ptxas emits its 17-instruction warp-aggregation sequence around this single-lane atomic); the other lanes get
// the value by a shuffle from lane 0 later
__device__ __forceinline__ int claim_ticket(unsigned counter_addr, int lane) {
    int j = 0;
    if (lane == 0) asm volatile("atom.shared.inc.u32 %0, [%1], 0x7fffffff;" : "=r"(j) : "r"(counter_addr) : "memory");
    return j;
}

// the dynamic tile queues: one counter per group in global memory
__device__ __forceinline__ unsigned queue_claim(unsigned *q) {
    unsigned v;
    asm volatile("atom.add.relaxed.gpu.global.u32 %0, [%1], 1;" : "=r"(v) : "l"(q) : "memory");
    return v;
}
__device__ __forceinline__ unsigned queue_peek(const unsigned *q) {
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(q) : "memory");
    return v;
}

__device__ __forceinline__ float mul_sat(float a, float b) {
    float r;
    asm("mul.rn.sat.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
    return r;
}

// the literal search (slow path) on the walk tree: code point (n, i) = single[(2^n + i) * 16 + c] / 2^24
static __device__ __noinline__ int reference_search_walk(const float *sSc, const float *sPen, float mu, float sg, int N) {
    const float rs = rcp_rn(sg);
    auto point = [&](int n, int i) -> float { return sSc[((1 << n) + i) * VBQ_GROUP] * kWalkUnscale; };
    const float z0 = point(0, 0);
    float bestL = score_exact(z0, mu, sg, rs, -sPen[0]), bestR = -CUDART_INF_F;
    int nL = 0, iL = 0, nR = 0, iR = 0;
    int ip = mu > z0 ? 1 : 0;
    for (int n = 1; n <= N; ++n) {
        const float zp = point(n, ip);
        const int b = mu > zp ? 1 : 0;
        const int fg = ip + b;   // number of depth-n points below mu = searchsorted(side='left'), quantizer.py:74
        const int il = clamp_index(fg, n, N, false), ir = clamp_index(fg, n, N, true);
        const float npn = -sPen[n];
        const float sl = score_exact(il == ip ? zp : point(n, il), mu, sg, rs, npn);
        const float sr = score_exact(ir == ip ? zp : point(n, ir), mu, sg, rs, npn);
        if (sl > bestL) { bestL = sl; nL = n; iL = il; }
        if (sr > bestR) { bestR = sr; nR = n; iR = ir; }
        ip = 2 * ip + b;
    }
    return bestR > bestL ? (nR << 24 | iR) : (nL << 24 | iL);
}

// The same search done by a whole warp for ONE coordinate (channel column sSc) whose walk ended at heap node Kd of depth
// kd >= N: lane j scores candidate j of the reference's order left_0..left_N, right_1..right_N; the first maximum wins.
// Every lane returns depth << 24 | index.  (A coordinate that the certificate rejects used to hold its warp, and with
// it the tile's slot, for microseconds.)
static __device__ __forceinline__ int reference_search_warp(const float *sSc, const float *sPen, float mu, float sg,
                                                            int N, int Kd, int kd, int lane) {
    const float rs = rcp_rn(sg);
    const bool right = lane > N;
    const int n = min(right ? lane - N : lane, N);
    auto point = [&](int i) -> float { return sSc[((1 << n) + i) * VBQ_GROUP] * kWalkUnscale; };
    const int ip = (Kd >> (kd - n)) - (1 << n);
    const float zp = point(ip);
    const int fg = ip + (mu > zp ? 1 : 0);
    const int idx = clamp_index(fg, n, N, right);
    float s = score_exact(idx == ip ? zp : point(idx), mu, sg, rs, -sPen[n]);
    // sequential semantics: candidate 0 starts as the best whatever its score; a NaN never replaces anything
    if (lane == 0) s = s != s ? CUDART_INF_F : s;
    else if (s != s || lane > 2 * N) s = -CUDART_INF_F;
    int who = lane;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float so = __shfl_xor_sync(0xffffffffu, s, o);
        const int wo = __shfl_xor_sync(0xffffffffu, who, o);
        if (so > s || (so == s && wo < who)) { s = so; who = wo; }
    }
    const int wi = __shfl_sync(0xffffffffu, idx, who);
    const int wn = who > N ? who - N : who;
    return wn << 24 | wi;
}

// The literal search for the coordinates of a unit that the certificate rejected, out of line (both-ends kernel: four
// unrolled inline copies cost 2 % of the step through registers and code size although they run for 5 coordinates in 10^5;
// the raw kernel measured no difference and keeps them inline).  Everything travels by value; r[u] < 0 means "unchanged",
// else depth << 24 | index within the level.  The whole warp serves one coordinate when they are few (lane j scores
// candidate j), else every lane searches for itself.  pen: penalties, pen_off: this lane's channel's offset into them.
template <int U>
struct SlowIO {
    int Kd[U];
    unsigned gap[U];
    int r[U];
};
template <int U>
static __device__ __noinline__ SlowIO<U> slow_search(SlowIO<U> io, const float *sSingle, const float *pen, int pen_off,
                                                     unsigned mine, unsigned sg_off_bytes, int N, int kd, int lane) {
#pragma unroll 1
    for (int u = 0; u < U; ++u) {
        io.r[u] = -1;
        const float m_ = lds_u32(mine + u * 128), s_ = lds_u32(mine + sg_off_bytes + u * 128);
        unsigned todo = __ballot_sync(0xffffffffu, io.gap[u] <= kKeyGuard);
        if (__popc(todo) <= 6) {
            while (todo) {
                const int L = __ffs(todo) - 1;
                todo &= todo - 1;
                const int r = reference_search_warp(sSingle + (L & (VBQ_GROUP - 1)), pen + __shfl_sync(0xffffffffu, pen_off, L),
                                                    __shfl_sync(0xffffffffu, m_, L), __shfl_sync(0xffffffffu, s_, L), N,
                                                    __shfl_sync(0xffffffffu, io.Kd[u], L), kd, lane);
                if (lane == L) io.r[u] = r;
            }
        } else if (io.gap[u] <= kKeyGuard) {
            io.r[u] = reference_search_walk(sSingle + (lane & (VBQ_GROUP - 1)), pen + pen_off, m_, s_, N);
        }
    }
    return io;
}

// OUT: compiled output set (bit 0 zhat, 1 qidx, 2 level, 3 bits), at most two arrays, in ascending bit order.
// NT > 0: max_bits_per_coord == NT at compile time; NT == 0: run time (<= kSmemDepth).
// W = consumer warps (the CTA has W + 1 warps); P = coordinate pairs per thread: a warp iteration ("unit") covers
// 4P consecutive rows x 16 channels, lane = (row parity, channel), coordinates at rows parity + 2u, u < 2P.
template <bool BOTH, int EM, bool PRUNE, bool TOTALS, int NT, int OUT, int W, int P>
__global__ void __launch_bounds__(32 * (W + 1), 1)
    vbq_bisect_tma_kernel(const QArgs a, const __grid_constant__ TmaMaps maps, const UniformPen up) {
    constexpr int U = 2 * P, S = kSlots;
    constexpr int kUnitRows = kQuadRows * P;
    constexpr int kUnits = kTmaRows / kUnitRows;               // units (tickets) per tile
    constexpr int kLogUnits = P == 1 ? 5 : (P == 2 ? 4 : 3);
    constexpr int kUnitFloats = kUnitRows * VBQ_GROUP;
    constexpr int kBoxFloats = kTmaRows * VBQ_GROUP;           // one array of one slot
    constexpr int kSgOff = S * kBoxFloats;                     // sigma word = mu word + kSgOff
    constexpr int kKeys = kSmemDepth + 1;
    constexpr unsigned kDepthBits = 15u;
    constexpr int kNOut = ((OUT & 1) ? 1 : 0) + ((OUT & 2) ? 1 : 0) + ((OUT & 4) ? 1 : 0) + ((OUT & 8) ? 1 : 0);
    static_assert(kNOut <= 2, "a slot has room for two output arrays");
    static_assert((P == 1 || P == 2 || P == 4) && S == 4 && kTmaRows == 128, "ticket bit fields");
    constexpr unsigned kTreeBytes = kWalkFloats * sizeof(float);

    // dynamic shared memory, byte offsets (everything the main loop touches sits at a constant offset from ONE base
    // register; left to itself the compiler re-derives the window address of every __shared__ object in every iteration)
    constexpr unsigned kOffDbl = kSingleRows * VBQ_GROUP * 4;             // [256][2][16] depths 1..7, one copy per half-warp
    constexpr unsigned kOffMu = kOffDbl + kDblRows * 2 * VBQ_GROUP * 4;   // [S][128][16] mu boxes, later first outputs
    constexpr unsigned kOffSg = kOffMu + kSgOff * 4;                      // [S][128][16] sigma boxes, later second outputs
    constexpr unsigned kOffBar = kOffSg + kSgOff * 4;                     // full[S], done[S], tree: 8 bytes each
    constexpr unsigned kOffDesc = kOffBar + 128;                          // int4[S]: (valid rows, range index, group, 0)
    constexpr unsigned kOffNext = kOffDesc + 16 * S;                      // next unclaimed ticket; + 4: number of tickets
    constexpr unsigned kOffPen = kOffNext + 16;                           // float[kKeys]
    static_assert(kOffPen + 4 * kKeys <= kTmaSmemBytes, "shared-memory layout");
    extern __shared__ __align__(1024) float smem[];
    float *sSingle = smem;                                      // [2048][16]   heap order, all depths
    float *sPen = smem + kOffPen / 4;
    __shared__ bool sLast;
    unsigned sm0 = smem_u32(smem);
    asm volatile("" : "+r"(sm0));   // opaque: keep it in a register

    const int N = NT > 0 ? NT : a.N;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col = lane & (VBQ_GROUP - 1);
    const int par = lane >> 4;
    const bool logvar = (a.flags & VBQ_FLAG_LOGVAR) != 0;
    const int C = a.C;
    const int rows = (int)a.rows;
    const long long rows4 = (a.rows + 3) & ~3ll;
    const long long vtotal = (rows4 + kSwitchRows) * a.n_groups - kSwitchRows;
    const long long p0 = row_cut(vtotal * blockIdx.x / gridDim.x, rows4, a.n_groups);
    const long long p1 = row_cut(vtotal * (blockIdx.x + 1) / gridDim.x, rows4, a.n_groups);
    const unsigned bar_full = sm0 + kOffBar, bar_done = bar_full + 8 * S, bar_tree = bar_full + 16 * S;

    // the next range of this CTA: rows [row_a, row_b) of group g (row_b a multiple of 4 or the padded end of the group)
    auto next_range = [&](long long &pos, int &g, int &row_a, int &row_b) {
        g = (int)(pos / rows4);
        row_a = (int)(pos - (long long)g * rows4);
        const long long end = min((long long)(g + 1) * rows4, p1);
        row_b = (int)(end - (long long)g * rows4);
        pos = end;
    };

#ifdef VBQ_TRACE
    double *tr = a.partials + (size_t)kMaxGrid * VBQ_TOTALS * a.n_lambda + (size_t)blockIdx.x * 1024;
    if (threadIdx.x == 0) tr[0] = (double)gtime();
#endif
    if (threadIdx.x == 0) {
        for (int s = 0; s < S; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_done + 8 * s, kUnits);   // one arrival per unit of the tile
        }
        mbar_init(bar_tree, 1);
        mbar_fence_init();
        sts_u32(sm0 + kOffNext, 0u);
    }
    if (threadIdx.x < kKeys) sPen[threadIdx.x] = up.v[threadIdx.x];
    __syncthreads();
    // programmatic stream serialization: nothing global is touched before pdl_wait() — except the code points of the
    // first range when the caller vouches that they were complete before the previous kernel of the stream started
    const int home_g = a.queue ? (int)((long long)blockIdx.x * a.n_groups / gridDim.x) : (int)min(p0 / rows4, (long long)a.n_groups - 1);
    const bool early_tree = (a.flags & VBQ_FLAG_TABLE_STABLE) != 0;
    if (early_tree && threadIdx.x == 32 * W) {
        mbar_arrive_expect_tx(bar_tree, kTreeBytes);
        bulk_load(sm0, a.packed + (size_t)a.n_groups * kPadEntries * VBQ_GROUP + (size_t)home_g * kWalkFloats, kTreeBytes, bar_tree);
    }
    pdl_wait();
#ifdef VBQ_TRACE
    if (threadIdx.x == 0) tr[1] = (double)gtime();
#endif

    Acc128 acc_dist = {0, 0};   // sum of the distortion terms in units of 2^-24: integer, so the order does not matter
    Acc128 acc_bits = {0, 0}, acc_em = {0, 0};   // BOTH: corrected code lengths / entropy-model bits, same units
    int acc_level = 0;

    if (warp == W) {
        // =============================== producer warp (one lane) =======================================================
        if (lane == 0) {
            tma_prefetch_map(&maps.in[0]);
            tma_prefetch_map(&maps.in[1]);
            if (kNOut > 0) { tma_prefetch_map(&maps.out[0][0]); tma_prefetch_map(&maps.out[0][1]); }
            if (kNOut > 1) { tma_prefetch_map(&maps.out[1][0]); tma_prefetch_map(&maps.out[1][1]); }
            int t_issue = 0, t_retire = 0;     // CTA-wide tile counters: tile t lives in slot t % S
            int ring_g[S], ring_row[S], ring_valid[S];
            auto retire = [&](int t) {         // slot -> global once every unit of the tile has been computed
                const int s = t & (S - 1);
                mbar_wait_sleepy(bar_done + 8 * s, (unsigned)(t / S) & 1u, 20000u);
                TRACE_P(t, 1);
                if (kNOut > 0) {
                    // the consumers fenced their st.shared into the async proxy before arriving
                    int g = 0, r0 = 0, valid = 0;
#pragma unroll
                    for (int j = 0; j < S; ++j)
                        if (j == s) { g = ring_g[j]; r0 = ring_row[j]; valid = ring_valid[j]; }
                    const unsigned base = sm0 + kOffMu + s * (kBoxFloats * 4);
                    if (valid == kTmaRows) {
                        tma_store_3d(&maps.out[0][0], base, g * VBQ_GROUP, r0, 0);
                        if (kNOut > 1) tma_store_3d(&maps.out[1][0], base + kSgOff * 4, g * VBQ_GROUP, r0, 0);
                    } else {   // cut tile: only its first `valid` rows belong to this CTA
                        for (int r = 0; r < valid; r += kQuadRows) {
                            const unsigned o = (unsigned)r * VBQ_GROUP * 4;
                            tma_store_3d(&maps.out[0][1], base + o, g * VBQ_GROUP, r0 + r, 0);
                            if (kNOut > 1) tma_store_3d(&maps.out[1][1], base + kSgOff * 4 + o, g * VBQ_GROUP, r0 + r, 0);
                        }
                    }
                    tma_store_commit();
                    TRACE_P(t, 2);
                    tma_store_wait_read<0>();   // the slot may be overwritten
                    TRACE_P(t, 3);
                }
            };
            auto load = [&](int t, int g, int r0, int valid, int range) {
                const int s = t & (S - 1);
                const unsigned base = sm0 + kOffMu + s * (kBoxFloats * 4);
                const unsigned bar = bar_full + 8 * s;
#pragma unroll
                for (int j = 0; j < S; ++j)
                    if (j == s) { ring_g[j] = g; ring_row[j] = r0; ring_valid[j] = valid; }
                sts_v4(sm0 + kOffDesc + 16 * s, valid, range, g, r0);
                TRACE_P(t, 0);
                mbar_arrive_expect_tx(bar, 2 * kBoxFloats * 4);
                tma_load_3d(base, &maps.in[0], g * VBQ_GROUP, r0, 0, bar);
                tma_load_3d(base + kSgOff * 4, &maps.in[1], g * VBQ_GROUP, r0, 0, bar);
            };
            int n_trees = early_tree ? 1 : 0;   // tree loads so far; the consumers wait for phase (range index) & 1
            int cur_g = early_tree ? home_g : -1;   // group whose tree is (being) loaded
            auto use_group = [&](int g) {   // -> range index of the tiles that follow
                if (g != cur_g) {
                    // every tile of the previous range has to be retired before its tree is overwritten
                    while (t_retire < t_issue) retire(t_retire++);
                    // ... and the previous tree has to have arrived (an unused prefetch may still be in flight)
                    if (n_trees > 0) mbar_wait(bar_tree, (unsigned)(n_trees - 1) & 1u);
                    mbar_arrive_expect_tx(bar_tree, kTreeBytes);
                    bulk_load(sm0, a.packed + (size_t)a.n_groups * kPadEntries * VBQ_GROUP + (size_t)g * kWalkFloats, kTreeBytes,
                              bar_tree);
                    ++n_trees;
                    cur_g = g;
                }
                return n_trees - 1;
            };
            if (a.queue == nullptr) {
                // static shares: rows [p0, p1) of the (group, row) order
                for (long long pos = p0; pos < p1;) {
                    int g, row_a, row_b;
                    next_range(pos, g, row_a, row_b);
                    const int range = use_group(g);
                    for (int r0 = row_a; r0 < row_b; r0 += kTmaRows) {
                        if (t_issue - t_retire == S) retire(t_retire++);
                        load(t_issue++, g, r0, min(kTmaRows, min(row_b, rows) - r0), range);
                    }
                }
            } else {
                // dynamic: every group is a queue of 128-row tiles (one global counter each).  A CTA starts with its home
                // group and, when that queue is empty, moves to a group nobody has touched yet or one with enough work left
                // to be worth a second tree; whoever has touched a queue stays until it is empty, so nothing is left over.
                const unsigned n_tiles_g = (unsigned)((rows + kTmaRows - 1) / kTmaRows);
                const unsigned worth = max(2u, 3u * gridDim.x / (2u * (unsigned)a.n_groups));
                int g = home_g;
                unsigned idx = queue_claim(a.queue + g);
                for (;;) {
                    if (idx >= n_tiles_g) {
                        int found = -1;
                        for (int j = 1; j < a.n_groups && found < 0; ++j) {
                            const int g2 = g + j < a.n_groups ? g + j : g + j - a.n_groups;
                            const unsigned taken = queue_peek(a.queue + g2);
                            if (taken == 0u || (taken < n_tiles_g && n_tiles_g - taken > worth)) found = g2;
                        }
                        if (found < 0) break;
                        g = found;
                        idx = queue_claim(a.queue + g);
                        continue;
                    }
                    const int range = use_group(g);
                    if (t_issue - t_retire == S) retire(t_retire++);
                    const int r0 = (int)idx * kTmaRows;
                    load(t_issue++, g, r0, min(kTmaRows, rows - r0), range);
                    idx = queue_claim(a.queue + g);   // in flight while the consumers work
                }
            }
            while (t_retire < t_issue) retire(t_retire++);
            // every store has READ its slot (retire waits for that), which is all the CTA owes the copies before it
            // exits; their global writes complete before the grid does.  Stop signs for the tickets still in flight (a
            // warp holds at most two: fewer than S tiles in all).
            for (int j = 0; j < S; ++j) {
                const int s_ = (t_issue + j) & (S - 1);
                sts_v4(sm0 + kOffDesc + 16 * s_, -1, 0, 0, 0);
                mbar_arrive(bar_full + 8 * s_);
            }
        } else if (lane == 1 && blockIdx.x == gridDim.x - 1 && a.peer_world > 0) {
            // Multi-GPU exchange of the totals (peer.cu), hidden behind this launch's search: an idle lane delivers the
            // sums of an EARLIER call (complete: the wait above covers every earlier kernel of the stream) to every
            // rank's inbox over NVLink (plain peer stores, then a system-scope release of the sequence number), and
            // collects a still earlier call: waits for every rank's entry and adds them in rank order.
            if (a.peer_seq) {
                double v[VBQ_TOTALS];
#pragma unroll
                for (int k = 0; k < VBQ_TOTALS; ++k) v[k] = __ldcv(a.peer_src + k);
                for (int p = 0; p < a.peer_world; ++p)
#pragma unroll
                    for (int k = 0; k < VBQ_TOTALS; ++k) a.peer_inbox[p][a.peer_off + k] = v[k];
                __threadfence_system();
                for (int p = 0; p < a.peer_world; ++p)
                    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(a.peer_inbox[p] + a.peer_flag), "l"(a.peer_seq) : "memory");
            }
            if (a.peer_cseq) {
                for (int r = 0; r < a.peer_world; ++r) {
                    const double *f = a.peer_own + a.peer_coff + (long long)r * a.peer_entry + (a.peer_entry - 1);
                    unsigned long long v;
                    do {
                        asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
                    } while (v < a.peer_cseq);
                }
#pragma unroll
                for (int k = 0; k < VBQ_TOTALS; ++k) {
                    double sum = 0.0;
                    for (int r = 0; r < a.peer_world; ++r) sum += __ldcv(a.peer_own + a.peer_coff + (long long)r * a.peer_entry + k);
                    a.peer_cout[k] = sum;
                }
            }
        }
        __syncwarp();
    } else {
        // =============================== consumers =======================================================================
        const unsigned kmask = a.keymask;
        const unsigned t_sg = sm0, t_db = sm0 + kOffDbl;
        // walk constants (see the header): floats whose bit patterns are (signed) byte addresses
        const float A1 = __uint_as_float(t_db + 2 * 128 + 4 * lane);                      // node 2 of this lane's copy
        const float Ec1 = __uint_as_float(0x80000000u | (t_db + 4 * lane));               // -(base of the double rows)
        const float Ec2 = __uint_as_float(0x80000000u | (t_sg + 4 * col));                // -(base of the single rows)
        const int esw = (int)(t_sg + 4 * col) - (int)(t_db + 4 * lane);
        const float Esw = __uint_as_float(esw < 0 ? 0x80000000u | (unsigned)(-esw) : (unsigned)esw);
        const float c128 = __uint_as_float(128u), c64 = __uint_as_float(64u);
        const float *sSc = sSingle + col;
        const unsigned lane_mu = sm0 + kOffMu + 4 * lane;   // coordinate u of a unit: + u * 128 bytes; sigma: + 4 kSgOff
        float z0s = 0.0f;
        int range = -1, cur_tile = -1, valid = 0, tile_r0 = 0, chan = 0;
        bool c_ok = false, group_full = false;
        float penc[kKeys];   // BOTH: this thread's channel's penalties (per range)
        // BOTH: depths at which the in-level neighbour of the path node can win for some channel of the group (see
        // iteration_both); warp-uniform
        unsigned bmask = 0;
        const float *lenp = nullptr;   // BOTH: this thread's channel's row of the code-length table
#pragma unroll
        for (int n = 0; n < kKeys; ++n) penc[n] = CUDART_INF_F;

        // one unit: U coordinates of this thread (unit rows par + 2u, channel col).  `mine` points at this thread's mu
        // word of coordinate 0; bit u of `okm`: coordinate u exists (the others were given harmless inputs by `prepare`).
        auto iteration = [&](const unsigned mine, const unsigned okm) {
            float2 nmu2[P], r2[P];
            bool ok[U];
            {
                float mu[U], sg[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    ok[u] = (okm >> u) & 1u;
                    mu[u] = lds_u32(mine + u * 128);
                    sg[u] = lds_u32(mine + 4 * kSgOff + u * 128);
                }
#pragma unroll
                for (int k = 0; k < P; ++k) {
                    nmu2[k] = __fmul2_rn(make_float2(mu[2 * k], mu[2 * k + 1]), make_float2(-kWalkScale, -kWalkScale));
                    r2[k] = __fmul2_rn(make_float2(rcp_approx(sg[2 * k]), rcp_approx(sg[2 * k + 1])),
                                       make_float2(0.70710678f * kWalkUnscale, 0.70710678f * kWalkUnscale));
                }
            }
            unsigned key[U][kKeys];
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int n = 0; n < kKeys; ++n) key[u][n] = (0x7fffffffu & ~kDepthBits) | (unsigned)n;
            float2 G[P];   // bit patterns = shared-memory byte addresses of the path nodes of the next depth
#pragma unroll
            for (int k = 0; k < P; ++k) {
                const float2 d = __fadd2_rn(make_float2(z0s, z0s), nmu2[k]);
                const float2 st = make_float2(mul_sat(d.x, -1.7014118e38f), mul_sat(d.y, -1.7014118e38f));
                G[k] = __ffma2_rn(st, make_float2(c128, c128), make_float2(A1, A1));
                const float2 t = __fmul2_rn(d, r2[k]);
                const float2 A = __ffma2_rn(t, t, make_float2(up.v[0], up.v[0]));
                key[2 * k][0] = make_key<0>(A.x, kmask);
                key[2 * k + 1][0] = make_key<0>(A.y, kmask);
            }
            auto depth = [&](auto n_tag) {
                constexpr int n = decltype(n_tag)::value;
                float2 z[P];
#pragma unroll
                for (int k = 0; k < P; ++k)
                    z[k] = make_float2(lds_pure(__float_as_uint(G[k].x)), lds_pure(__float_as_uint(G[k].y)));
#pragma unroll
                for (int k = 0; k < P; ++k) {
                    const float2 d = __fadd2_rn(z[k], nmu2[k]);
                    if (n < kSmemDepth && (NT > 0 ? n < NT : true)) {   // the address of the next path node
                        float2 GL;
                        if (n < kDblDepth) GL = __ffma2_rn(G[k], make_float2(2.0f, 2.0f), make_float2(Ec1, Ec1));
                        else if (n == kDblDepth) GL = __fadd2_rn(G[k], make_float2(Esw, Esw));
                        else GL = __ffma2_rn(G[k], make_float2(2.0f, 2.0f), make_float2(Ec2, Ec2));
                        const float2 st = make_float2(mul_sat(d.x, -1.7014118e38f), mul_sat(d.y, -1.7014118e38f));
                        const float stride = n < kDblDepth ? c128 : c64;
                        G[k] = __ffma2_rn(st, make_float2(stride, stride), GL);
                    }
                    const float2 t = __fmul2_rn(d, r2[k]);
                    const float2 A = __ffma2_rn(t, t, make_float2(up.v[n], up.v[n]));
                    key[2 * k][n] = make_key<n>(A.x, kmask);
                    key[2 * k + 1][n] = make_key<n>(A.y, kmask);
                }
            };
            int m_done = 0;   // deepest depth visited
            // sound early exit (PRUNE): every deeper key is >= key(pen_n), so the walk may stop once the best key so far
            // is more than the certificate's guard below it for every coordinate of the warp (tested every third depth)
            unsigned run_min[U];
#pragma unroll
            for (int u = 0; u < U; ++u) run_min[u] = 0xffffffffu;
            auto prune_here = [&](auto n_tag) -> bool {
                constexpr int n = decltype(n_tag)::value;
                const unsigned floor_key = __float_as_uint(up.v[n]) & kmask;
                bool done = floor_key > kKeyGuard + 32u;
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    run_min[u] = __vimin3_u32(run_min[u], key[u][n - 3], key[u][n - 2]);
                    run_min[u] = min(run_min[u], key[u][n - 1]);
                    done = done && run_min[u] < floor_key - (kKeyGuard + 32u);
                }
                return __all_sync(0xffffffffu, done);
            };
            bool stop = false;
#define VBQ_DEPTH(n_)                                                                                          \
    if constexpr (n_ <= kSmemDepth) {                                                                          \
        if ((NT > 0 ? n_ <= NT : n_ <= N) && !stop) {                                                          \
            if (PRUNE && (n_ <= 9 && n_ % 3 == 0) && prune_here(std::integral_constant<int, n_>{})) {          \
                stop = true;                                                                                   \
            } else {                                                                                           \
                depth(std::integral_constant<int, n_>{});                                                      \
                m_done = n_;                                                                                   \
            }                                                                                                  \
        }                                                                                                      \
    }
            VBQ_DEPTH(1) VBQ_DEPTH(2) VBQ_DEPTH(3) VBQ_DEPTH(4) VBQ_DEPTH(5)
            VBQ_DEPTH(6) VBQ_DEPTH(7) VBQ_DEPTH(8) VBQ_DEPTH(9) VBQ_DEPTH(10)
#undef VBQ_DEPTH
            static_assert(kSmemDepth == 10, "the depth macro list above covers depths 1..10");
            // G addresses the node of depth kd: kd = m_done + 1 if the walk stopped above the last tree level (N <
            // kSmemDepth: it then points at one of the repeated ancestors), else the depth-10 path node itself
            const int kd = m_done < kSmemDepth ? m_done + 1 : kSmemDepth;

            int wn[U], wP[U], Kd[U];
            unsigned gap[U], gap_min = 0xffffffffu;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const unsigned *k_ = key[u];
                unsigned m = k_[0];
#pragma unroll
                for (int n = 1; n + 1 < kKeys; n += 2) m = __vimin3_u32(m, k_[n], k_[n + 1]);
                if (kKeys % 2 == 0) m = min(m, k_[kKeys - 1]);
                const unsigned nm = ~m;
                unsigned g0 = 0xffffffffu, g1 = 0xffffffffu;
#pragma unroll
                for (int n = 0; n < kKeys; n += 2) g0 = __viaddmin_u32(k_[n], nm, g0);
#pragma unroll
                for (int n = 1; n < kKeys; n += 2) g1 = __viaddmin_u32(k_[n], nm, g1);
                gap[u] = min(g0, g1);
                gap_min = min(gap_min, gap[u]);
                wn[u] = (int)(m & kDepthBits);
                // heap index of the node G addresses, then of its ancestor at the winning depth
                const unsigned gb = __float_as_uint(u & 1 ? G[u / 2].y : G[u / 2].x);
                Kd[u] = kd <= kDblDepth ? (int)((gb - (t_db + 4 * lane)) >> 7) : (int)((gb - (t_sg + 4 * col)) >> 6);
                wP[u] = Kd[u] >> (kd - wn[u]);
            }
            if (__any_sync(0xffffffffu, gap_min <= kKeyGuard)) {
                // rare (a few coordinates in 10^5): the coordinates that are not certified redo the literal search on
                // the reloaded inputs — the whole warp for one coordinate when they are few, else every lane for itself
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const float m_ = lds_u32(mine + u * 128), s_ = lds_u32(mine + 4 * kSgOff + u * 128);
                    unsigned todo = __ballot_sync(0xffffffffu, gap[u] <= kKeyGuard);
                    if (__popc(todo) <= 6) {
                        while (todo) {
                            const int L = __ffs(todo) - 1;
                            todo &= todo - 1;
                            const int r = reference_search_warp(sSingle + (L & (VBQ_GROUP - 1)), sPen,
                                                                __shfl_sync(0xffffffffu, m_, L), __shfl_sync(0xffffffffu, s_, L),
                                                                N, __shfl_sync(0xffffffffu, Kd[u], L), kd, lane);
                            if (lane == L) {
                                wn[u] = r >> 24;
                                wP[u] = (1 << wn[u]) + (r & 0xffffff);
                            }
                        }
                    } else if (gap[u] <= kKeyGuard) {
                        const int r = reference_search_walk(sSc, sPen, m_, s_, N);
                        wn[u] = r >> 24;
                        wP[u] = (1 << wn[u]) + (r & 0xffffff);
                    }
                }
            }
            float dsum = 0.0f;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int n = wn[u], Pn = wP[u];
                // sorted index q = (2i+1) 2^(N-n) - 1 with i = Pn - 2^n
                const int q = ((2 * Pn + 1) << (N - n)) - (2 << N) - 1;
                float zh = 0.0f;   // scaled by 2^24
                if (TOTALS || (OUT & 1)) zh = lds_pure((unsigned)imad(Pn, kRowStrideBytes, (int)(t_sg + 4 * col)));
                // the outputs replace this thread's own inputs in the slot (first output array in the mu box)
                int slot_word = 0;
                if (OUT & 1) { sts_u32(mine + slot_word * 4 * kSgOff + u * 128, __float_as_uint(zh * kWalkUnscale)); ++slot_word; }
                if (OUT & 2) { sts_u32(mine + slot_word * 4 * kSgOff + u * 128, (unsigned)q); ++slot_word; }
                if (OUT & 4) { sts_u32(mine + slot_word * 4 * kSgOff + u * 128, (unsigned)n); ++slot_word; }
                if (OUT & 8) { sts_u32(mine + slot_word * 4 * kSgOff + u * 128, __float_as_uint((float)n)); ++slot_word; }
                if (TOTALS && ok[u]) {
                    const float t = (zh + (u & 1 ? nmu2[u / 2].y : nmu2[u / 2].x)) * (u & 1 ? r2[u / 2].y : r2[u / 2].x);
                    acc_level += n;
                    dsum = __fmaf_rn(t, t, dsum);
                }
            }
            // float32 within the thread's coordinates of the unit, then an exact integer sum (saturating conversion):
            // whichever warp computes whichever unit, the total is the same
            if (TOTALS) acc_dist.add_q24(dsum);
        };

        // The same for arbitrary non-negative penalties (corrected code lengths n + R_lambda[c, n], quantizer.py:170-180):
        // without monotone penalties the in-level neighbour of the path node on the side of mu — the other end of the
        // reference's bracket — stays a candidate.  Both ends of a depth carry the same penalty, so only the NEARER one
        // can win (every float32 operation of the score is monotone): per depth the kernel loads the neighbour as well,
        // keeps min(|z - mu|, |z' - mu|) and ranks ONE key, exactly as above.  Which end it was is decided for the
        // winning depth alone, in the epilogue, where the farther end also enters the certificate (it is the only
        // candidate that the per-depth keys do not cover: the farther end of any other depth loses to its own nearer
        // end).  Level ends need no test: there the "neighbour" read through the heap order is the extreme point of
        // the adjacent level, which lies on the path node's side of mu and farther away (quantizer.py:50-63: the
        // bracket's second point is the path node itself).  The one exception is mu above the highest point of depth
        // N, where the reference pairs the highest with the SECOND-highest point: those coordinates take the literal
        // search.
        //   Most depths do not need the neighbour at all.  Between the path node of depth n and its neighbour lies exactly
        // one coarser point, their lowest common ancestor A (depth a < n), which is on the search path; mu lies between the
        // path node and A, so A is nearer to mu than the neighbour.  If pen[a] <= pen[n], A's float32 score is at least as
        // good (monotone operations) and A comes first in the reference's candidate order: the neighbour cannot win.
        // bmask holds the depths n with pen[n] < max(pen[0..n-1]) for some channel of the group — for fitted corrected
        // lengths one to three shallow depths — and every other depth takes the raw-length step (one load).
        auto penc_at = [&](int n) -> float {   // penc[n] for a run-time n without moving the array to local memory
            float v = penc[0];
#pragma unroll
            for (int j = 1; j < kKeys; ++j) v = n == j ? penc[j] : v;
            return v;
        };
        auto iteration_both = [&](const unsigned mine, const unsigned okm, const int unit_row) {
            float2 nmu2[P], r2[P];
            bool ok[U];
            {
                float mu[U], sg[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    ok[u] = (okm >> u) & 1u;
                    mu[u] = lds_u32(mine + u * 128);
                    sg[u] = lds_u32(mine + 4 * kSgOff + u * 128);
                }
#pragma unroll
                for (int k = 0; k < P; ++k) {
                    nmu2[k] = __fmul2_rn(make_float2(mu[2 * k], mu[2 * k + 1]), make_float2(-kWalkScale, -kWalkScale));
                    r2[k] = __fmul2_rn(make_float2(rcp_approx(sg[2 * k]), rcp_approx(sg[2 * k + 1])),
                                       make_float2(0.70710678f * kWalkUnscale, 0.70710678f * kWalkUnscale));
                }
            }
            unsigned key[U][kKeys];
#pragma unroll
            for (int u = 0; u < U; ++u)
#pragma unroll
                for (int n = 0; n < kKeys; ++n) key[u][n] = (0x7fffffffu & ~kDepthBits) | (unsigned)n;
            float2 G[P], st_last[P];
#pragma unroll
            for (int k = 0; k < P; ++k) {
                const float2 d = __fadd2_rn(make_float2(z0s, z0s), nmu2[k]);
                const float2 st = make_float2(mul_sat(d.x, -1.7014118e38f), mul_sat(d.y, -1.7014118e38f));
                G[k] = __ffma2_rn(st, make_float2(c128, c128), make_float2(A1, A1));
                st_last[k] = st;
                const float2 t = __fmul2_rn(d, r2[k]);
                const float2 A = __ffma2_rn(t, t, make_float2(penc[0], penc[0]));
                key[2 * k][0] = make_key<0>(A.x, kmask);
                key[2 * k + 1][0] = make_key<0>(A.y, kmask);
            }
            auto depth = [&](auto n_tag, auto raw_tag) {
                constexpr int n = decltype(n_tag)::value;
                constexpr bool kRawOnly = decltype(raw_tag)::value;       // the caller knows that bit n of bmask is clear
                const float stride = n <= kDblDepth ? c128 : c64;         // row pitch of the level the node sits in
                float2 z[P];
#pragma unroll
                for (int k = 0; k < P; ++k)
                    z[k] = make_float2(lds_pure(__float_as_uint(G[k].x)), lds_pure(__float_as_uint(G[k].y)));
                if (kRawOnly || !((bmask >> n) & 1u)) {   // the neighbour of this depth cannot win: the step of the raw-length search
#pragma unroll
                    for (int k = 0; k < P; ++k) {
                        const float2 d = __fadd2_rn(z[k], nmu2[k]);
                        const float2 st = make_float2(mul_sat(d.x, -1.7014118e38f), mul_sat(d.y, -1.7014118e38f));
                        st_last[k] = st;
                        if (n < kSmemDepth && (NT > 0 ? n < NT : true)) {
                            float2 GL;
                            if (n < kDblDepth) GL = __ffma2_rn(G[k], make_float2(2.0f, 2.0f), make_float2(Ec1, Ec1));
                            else if (n == kDblDepth) GL = __fadd2_rn(G[k], make_float2(Esw, Esw));
                            else GL = __ffma2_rn(G[k], make_float2(2.0f, 2.0f), make_float2(Ec2, Ec2));
                            const float nstride = n < kDblDepth ? c128 : c64;
                            G[k] = __ffma2_rn(st, make_float2(nstride, nstride), GL);
                        }
                        const float2 t = __fmul2_rn(d, r2[k]);
                        const float2 A = __ffma2_rn(t, t, make_float2(penc[n], penc[n]));
                        key[2 * k][n] = make_key<n>(A.x, kmask);
                        key[2 * k + 1][n] = make_key<n>(A.y, kmask);
                    }
                    return;
                }
#pragma unroll
                for (int k = 0; k < P; ++k) {
                    const float2 d = __fadd2_rn(z[k], nmu2[k]);
                    const float2 st = make_float2(mul_sat(d.x, -1.7014118e38f), mul_sat(d.y, -1.7014118e38f));
                    st_last[k] = st;
                    // the neighbour on the side of the branch: address +- one row
                    const float2 Gm = __fadd2_rn(G[k], make_float2(-stride, -stride));
                    const float2 Gn = __ffma2_rn(st, make_float2(2.0f * stride, 2.0f * stride), Gm);
                    const float2 zn = make_float2(lds_pure(__float_as_uint(Gn.x)), lds_pure(__float_as_uint(Gn.y)));
                    if (n < kSmemDepth && (NT > 0 ? n < NT : true)) {   // the address of the next path node
                        float2 GL;
                        if (n < kDblDepth) GL = __ffma2_rn(G[k], make_float2(2.0f, 2.0f), make_float2(Ec1, Ec1));
                        else if (n == kDblDepth) GL = __fadd2_rn(G[k], make_float2(Esw, Esw));
                        else GL = __ffma2_rn(G[k], make_float2(2.0f, 2.0f), make_float2(Ec2, Ec2));
                        const float nstride = n < kDblDepth ? c128 : c64;
                        G[k] = __ffma2_rn(st, make_float2(nstride, nstride), GL);
                    }
                    const float2 dn = __fadd2_rn(zn, nmu2[k]);
                    const float2 dm = make_float2(fminf(fabsf(d.x), fabsf(dn.x)), fminf(fabsf(d.y), fabsf(dn.y)));
                    const float2 t = __fmul2_rn(dm, r2[k]);
                    const float2 A = __ffma2_rn(t, t, make_float2(penc[n], penc[n]));
                    key[2 * k][n] = make_key<n>(A.x, kmask);
                    key[2 * k + 1][n] = make_key<n>(A.y, kmask);
                }
            };
            int m_done = 0;
#define VBQ_DEPTH(n_, raw_)                                                                                    \
    if constexpr (n_ <= kSmemDepth) {                                                                          \
        if (NT > 0 ? n_ <= NT : n_ <= N) {                                                                     \
            depth(std::integral_constant<int, n_>{}, std::integral_constant<bool, raw_>{});                    \
            m_done = n_;                                                                                       \
        }                                                                                                      \
    }
            // fitted corrected lengths dip at the shallow depths only: from depth 4 on, one test selects a branch-free run of
            // raw-length steps (which the compiler schedules across depths) or the per-depth tests
            VBQ_DEPTH(1, false) VBQ_DEPTH(2, false) VBQ_DEPTH(3, false)
            if ((bmask >> 4) == 0u) {
                VBQ_DEPTH(4, true) VBQ_DEPTH(5, true) VBQ_DEPTH(6, true) VBQ_DEPTH(7, true)
                VBQ_DEPTH(8, true) VBQ_DEPTH(9, true) VBQ_DEPTH(10, true)
            } else {
                VBQ_DEPTH(4, false) VBQ_DEPTH(5, false) VBQ_DEPTH(6, false) VBQ_DEPTH(7, false)
                VBQ_DEPTH(8, false) VBQ_DEPTH(9, false) VBQ_DEPTH(10, false)
            }
#undef VBQ_DEPTH
            const int kd = m_done < kSmemDepth ? m_done + 1 : kSmemDepth;

            int wn[U], wP[U], Kd[U];
            unsigned gap[U], mkey[U], gap_min = 0xffffffffu;
            int wn_min = kKeys;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const unsigned *k_ = key[u];
                unsigned m = k_[0];
#pragma unroll
                for (int n = 1; n + 1 < kKeys; n += 2) m = __vimin3_u32(m, k_[n], k_[n + 1]);
                if (kKeys % 2 == 0) m = min(m, k_[kKeys - 1]);
                const unsigned nm = ~m;
                unsigned g0 = 0xffffffffu, g1 = 0xffffffffu;
#pragma unroll
                for (int n = 0; n < kKeys; n += 2) g0 = __viaddmin_u32(k_[n], nm, g0);
#pragma unroll
                for (int n = 1; n < kKeys; n += 2) g1 = __viaddmin_u32(k_[n], nm, g1);
                gap[u] = min(g0, g1);
                wn[u] = (int)(m & kDepthBits);
                const unsigned gb = __float_as_uint(u & 1 ? G[u / 2].y : G[u / 2].x);
                Kd[u] = kd <= kDblDepth ? (int)((gb - (t_db + 4 * lane)) >> 7) : (int)((gb - (t_sg + 4 * col)) >> 6);
                wP[u] = Kd[u] >> (kd - wn[u]);
                mkey[u] = m;
                wn_min = min(wn_min, wn[u]);
            }
            // mu above the highest point of the deepest level: the reference's bracket is (second highest, highest)
            if (kd == N && ((bmask >> N) & 1u)) {
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const float sl = u & 1 ? st_last[u / 2].y : st_last[u / 2].x;
                    if (Kd[u] == (2 << kd) - 1 && sl != 0.0f) gap[u] = 0u;
                }
            }
            const bool nb_any = wn_min < 32 - __clz(bmask);   // some winner is no deeper than the deepest masked depth
            // the two ends of the bracket at the winning depth, where the neighbour can win (else the path node: its
            // neighbour lost to an ancestor): the path node and its neighbour on the side of the branch taken there (a path
            // bit, or the last comparison at the deepest level)
            if (__any_sync(0xffffffffu, nb_any)) {
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const bool nb = (bmask >> wn[u]) & 1u;
                    const float sl = u & 1 ? st_last[u / 2].y : st_last[u / 2].x;
                    const int b = wn[u] < kd ? (Kd[u] >> (kd - wn[u] - 1)) & 1 : (sl != 0.0f ? 1 : 0);
                    const int Pp = wP[u], Pq = Pp + 2 * b - 1;
                    const float nm_ = u & 1 ? nmu2[u / 2].y : nmu2[u / 2].x, r_ = u & 1 ? r2[u / 2].y : r2[u / 2].x;
                    const float dp = lds_pure((unsigned)imad(Pp, kRowStrideBytes, (int)(t_sg + 4 * col))) + nm_;
                    const float dq = wn[u] > 0 ? lds_pure((unsigned)imad(Pq, kRowStrideBytes, (int)(t_sg + 4 * col))) + nm_ : CUDART_INF_F;
                    // the nearer one wins; at equal distance the scores are equal and the left end comes first in the
                    // reference's candidate order.  Near-equal scores of the two ends: not certified.
                    const float ap = fabsf(dp), aq = fabsf(dq);
                    const bool take_q = nb && (aq < ap || (aq == ap && b == 0 && wn[u] > 0));
                    wP[u] = take_q ? Pq : Pp;
                    const float tf = fmaxf(ap, aq) * r_;
                    const int dfar = (int)(__float_as_uint(__fmaf_rn(tf, tf, penc_at(wn[u]))) & kmask) - (int)(mkey[u] & kmask);
                    if (nb) gap[u] = min(gap[u], dfar < 0 ? 0u : (unsigned)dfar);   // both keys are patterns of non-negative floats
                }
            }
#pragma unroll
            for (int u = 0; u < U; ++u) gap_min = min(gap_min, gap[u]);
            if (__any_sync(0xffffffffu, gap_min <= kKeyGuard)) {   // rare: a few coordinates in 10^5
                SlowIO<U> io;
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    io.Kd[u] = Kd[u];
                    io.gap[u] = gap[u];
                    io.r[u] = -1;
                }
                io = slow_search<U>(io, sSingle, a.pen, (a.pen_channels == 1 ? 0 : chan) * (N + 1), mine, 4 * kSgOff, N, kd, lane);
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (io.r[u] >= 0) {
                        wn[u] = io.r[u] >> 24;
                        wP[u] = (1 << wn[u]) + (io.r[u] & 0xffffff);
                    }
            }
            float dsum = 0.0f, bsum = 0.0f, esum = 0.0f;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const int n = wn[u], Pn = wP[u];
                const int q = ((2 * Pn + 1) << (N - n)) - (2 << N) - 1;
                float zh = 0.0f;   // scaled by 2^24
                if (TOTALS || (OUT & 1)) zh = lds_pure((unsigned)imad(Pn, kRowStrideBytes, (int)(t_sg + 4 * col)));
                const float len = lenp ? __ldg(lenp + n) : (float)n;
                float em = 0.0f;
                if (EM == 1) em = __ldg(a.em + (size_t)chan * a.Q + q);
                int slot_word = 0;
                if (OUT & 1) { sts_u32(mine + slot_word * 4 * kSgOff + u * 128, __float_as_uint(zh * kWalkUnscale)); ++slot_word; }
                if (OUT & 2) { sts_u32(mine + slot_word * 4 * kSgOff + u * 128, (unsigned)q); ++slot_word; }
                if (OUT & 4) { sts_u32(mine + slot_word * 4 * kSgOff + u * 128, (unsigned)n); ++slot_word; }
                // EM == 2: the heap index of the winner travels in the code-length box; em_gather_kernel (quantize_tma_both.cu)
                // turns it into the code length and entropy_model[c][q], the latter from a shared-memory copy of the group's table
                if (OUT & 8) { sts_u32(mine + slot_word * 4 * kSgOff + u * 128, EM == 2 ? (unsigned)Pn : __float_as_uint(len)); ++slot_word; }
                if (EM == 1 && a.em_bits && ok[u])
                    a.em_bits[((size_t)(tile_r0 + unit_row + par + 2 * u)) * C + chan] = em;
                if (TOTALS && ok[u]) {
                    const float t = (zh + (u & 1 ? nmu2[u / 2].y : nmu2[u / 2].x)) * (u & 1 ? r2[u / 2].y : r2[u / 2].x);
                    acc_level += n;
                    dsum = __fmaf_rn(t, t, dsum);
                    bsum += len;
                    esum += em;
                }
            }
            if (TOTALS) {
                acc_dist.add_q24(dsum);
                acc_bits.add_q24(bsum);
                if (EM == 1) acc_em.add_q24(esum);
            }
        };

        // Partial units (rows beyond the tile's share, channels beyond C) and log-variance inputs are handled BEFORE the
        // search, in the slot: a thread rewrites its own words — sigma = sqrt(exp(logvar)) (quantizer.py:193-198), and
        // mu = 0, sigma = 1 for coordinates that do not exist — so that ONE instance of the search serves every case.
        auto prepare = [&](const unsigned mine, const int my_rows, const bool full) -> unsigned {
            unsigned okm = 0;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const bool ok = full || (c_ok && par + 2 * u < my_rows);
                float m = lds_u32(mine + u * 128), sd = lds_u32(mine + 4 * kSgOff + u * 128);
                if (logvar) sd = sigma_of_logvar(sd);
                if (!ok) { m = 0.0f; sd = 1.0f; }
                sts_u32(mine + u * 128, __float_as_uint(m));
                sts_u32(mine + 4 * kSgOff + u * 128, __float_as_uint(sd));
                okm |= ok ? 1u << u : 0u;
            }
            return okm;
        };
        {
            int kk = __shfl_sync(0xffffffffu, claim_ticket(sm0 + kOffNext, lane), 0);
            for (;;) {
                // the next ticket one iteration ahead; its value is read at the end of this iteration, so the atomic's
                // latency never stalls the warp
                const int nxt_raw = claim_ticket(sm0 + kOffNext, lane);
                const int tile = kk >> kLogUnits;
                const unsigned sb = ((unsigned)tile & (S - 1)) * 8u;
                if (tile != cur_tile) {
                    cur_tile = tile;
                    mbar_wait_sleepy(bar_full + sb, ((unsigned)tile >> 2) & 1u, 20000u);
                    const int4 d = lds_v4(sm0 + kOffDesc + 2 * sb);
                    if (d.x < 0) break;   // stop sign: no more tiles
                    valid = d.x;
                    tile_r0 = d.w;
                    if (d.y != range) {   // a new range: its tree, first code point and channel
                        range = d.y;
                        mbar_wait(bar_tree, (unsigned)range & 1u);
                        z0s = lds_u32(sm0 + 4 * (VBQ_GROUP + col));
                        c_ok = d.z * VBQ_GROUP + col < C;
                        group_full = d.z * VBQ_GROUP + VBQ_GROUP <= C;
                        chan = min(d.z * VBQ_GROUP + col, C - 1);
                        if (BOTH) {
#pragma unroll
                            for (int n = 0; n < kKeys; ++n)
                                penc[n] = n <= N ? __ldg(a.pen + (size_t)(a.pen_channels == 1 ? 0 : chan) * (N + 1) + n) : CUDART_INF_F;
                            lenp = a.len ? a.len + (size_t)(a.pen_channels == 1 ? 0 : chan) * (N + 1) : nullptr;
                            unsigned below = 0;
                            float pmax = penc[0];
#pragma unroll
                            for (int n = 1; n < kKeys; ++n)
                                if (n <= N) {
                                    below |= penc[n] < pmax ? 1u << n : 0u;
                                    pmax = fmaxf(pmax, penc[n]);
                                }
                            bmask = (a.flags & VBQ_FLAG_NEIGHBOUR_EVERY_DEPTH) ? 0x7feu : __reduce_or_sync(0xffffffffu, below);
                        }
                    }
                }
                const int my_rows = valid - (kk & (kUnits - 1)) * kUnitRows;   // rows of this unit that belong to the tile
                const unsigned mine = lane_mu + (kk & (S * kUnits - 1)) * (kUnitFloats * 4);
                if (my_rows > 0) {
                    const bool full = my_rows >= kUnitRows && group_full;
                    const unsigned okm = (full && !logvar) ? (1u << U) - 1u : prepare(mine, my_rows, full);
                    if constexpr (BOTH) iteration_both(mine, okm, (kk & (kUnits - 1)) * kUnitRows);
                    else iteration(mine, okm);
                }
                if (kNOut > 0) fence_proxy_async();   // this thread's st.shared -> visible to the TMA store
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_done + sb);
                kk = __shfl_sync(0xffffffffu, nxt_raw, 0);
            }
        }
    }

#ifdef VBQ_TRACE
    if (threadIdx.x == 0) tr[2] = (double)gtime();
    if (threadIdx.x == 32 * W) tr[3] = (double)gtime();
#endif
    if (TOTALS) {
        // integer sums inside the CTA, integer partials of the CTAs added by the last CTA to arrive (ticket counter):
        // exact, so neither the arrival order nor the distribution of the tiles over warps and CTAs matters
        Acc128 v[VBQ_TOTALS];
        v[0].lo = (unsigned long long)acc_level; v[0].hi = 0;
        v[1] = acc_bits;
        if (!BOTH) { v[1].lo = (unsigned long long)acc_level << 24; v[1].hi = 0; }
        v[2] = acc_em;
        v[3] = acc_dist;
        Acc128(*sQ)[kMaxThreads / 32] = reinterpret_cast<Acc128(*)[kMaxThreads / 32]>(smem + kOffMu / 4);   // the slots are idle
        __syncthreads();
#pragma unroll
        for (int k = 0; k < VBQ_TOTALS; ++k) {
            v[k].warp_sum();
            if (lane == 0) sQ[k][warp] = v[k];
        }
        __syncthreads();
        Acc128 *part = reinterpret_cast<Acc128 *>(a.partials);
        if (warp == 0) {
#pragma unroll
            for (int k = 0; k < VBQ_TOTALS; ++k) {
                if (lane <= W) v[k] = sQ[k][lane];
                else v[k].lo = v[k].hi = 0;
                v[k].warp_sum();
            }
            if (lane == 0) {
#pragma unroll
                for (int k = 0; k < VBQ_TOTALS; ++k) part[VBQ_TOTALS * blockIdx.x + k] = v[k];
                unsigned t;   // release: the partials above are visible to whoever acquires the counter after this increment
                asm volatile("atom.add.acq_rel.gpu.global.u32 %0, [%1], 1;" : "=r"(t) : "l"(a.ticket) : "memory");
                sLast = (t == gridDim.x - 1);
            }
        }
        __syncthreads();
        if (sLast && warp == 0) {
            __threadfence();
            const volatile unsigned long long *vp = reinterpret_cast<const volatile unsigned long long *>(part);
#pragma unroll
            for (int k = 0; k < VBQ_TOTALS; ++k) {
                Acc128 x = {0, 0};
                for (unsigned b = lane; b < gridDim.x; b += 32) {
                    Acc128 t;
                    t.lo = vp[2 * (VBQ_TOTALS * b + k)];
                    t.hi = vp[2 * (VBQ_TOTALS * b + k) + 1];
                    x.add(t);
                }
                x.warp_sum();
                if (lane == 0) {
                    const double d_ = k == 0 ? (double)x.lo : x.value();
                    a.totals[k] = a.accumulate ? a.totals[k] + d_ : d_;
                }
            }
            if (lane == 0) a.ticket[0] = 0u;
            if (a.queue)
                for (int g = lane; g < a.n_groups; g += 32) a.queue[g] = 0u;
        }
    }
#ifdef VBQ_TRACE
    if (threadIdx.x == 0) tr[4] = (double)gtime();
#endif
}

template <bool BOTH, int EM, bool PRUNE, bool TOTALS, int NT, int OUT, int W, int P>
static int launch_tma(const QArgs &a0, const void *out0, const void *out1, int dev, int sms, cudaStream_t st) {
    constexpr int kTile = kTmaRows;
    const long long rows4 = (a0.rows + 3) & ~3ll;
    long long gx = rows4 / kQuadRows * a0.n_groups;   // quads
    gx = gx < sms ? gx : sms;
    if (gx > kMaxGrid) gx = kMaxGrid;
    if (gx < 1) gx = 1;
    auto kern = vbq_bisect_tma_kernel<BOTH, EM, PRUNE, TOTALS, NT, OUT, W, P>;
    VBQ_ENSURE_MAX_SMEM(kern, dev);
    static_assert(((size_t)kWalkFloats + (size_t)kSlots * 2 * kTile * VBQ_GROUP) * sizeof(float) + 512 == kTmaSmemBytes, "slots");
    const size_t smem = kTmaSmemBytes;
    const long long plane = a0.rows * (long long)a0.C;
    for (int lam = 0; lam < a0.n_lambda; ++lam) {   // one launch per lambda (several lambdas normally take the sweep kernel)
        QArgs a = a0;
        const size_t lo = (size_t)lam * a0.lam_stride;
        const char *o0 = out0 ? (const char *)out0 + lo * 4 : nullptr, *o1 = out1 ? (const char *)out1 + lo * 4 : nullptr;
        if (a.totals) a.totals = a0.totals + (size_t)lam * VBQ_TOTALS;
        a.n_lambda = 1;
        a.pen = a0.pen + (size_t)lam * a0.pen_channels * (a0.N + 1);
        if (a.len) a.len = a0.len + (size_t)lam * a0.pen_channels * (a0.N + 1);
        if (a.em) a.em = a0.em + (size_t)lam * a0.C * a0.Q;
        if (a.em_bits) a.em_bits = a0.em_bits + lo;
        TmaMaps maps;
        RETURN_IF(vbq_make_tensor_map(&maps.in[0], a.mu, a.C, a.rows, 1, plane, kTile));
        RETURN_IF(vbq_make_tensor_map(&maps.in[1], a.sigma, a.C, a.rows, 1, plane, kTile));
        for (int k = 0; k < 2; ++k) {   // unused output maps repeat an input map so that the parameter block is initialised
            const int br = k == 0 ? kTile : kQuadRows;
            RETURN_IF(vbq_make_tensor_map(&maps.out[0][k], o0 ? o0 : (const void *)a.mu, a.C, a.rows, 1, plane, br));
            RETURN_IF(vbq_make_tensor_map(&maps.out[1][k], o1 ? o1 : (const void *)a.mu, a.C, a.rows, 1, plane, br));
        }
        UniformPen up;
        const float *hp = a0.h_pen + (size_t)lam * a0.pen_channels * (a0.N + 1);
        for (int n = 0; n <= kSmemDepth; ++n) up.v[n] = (!BOTH && n <= a.N) ? hp[n] : HUGE_VALF;
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((int)gx);
        cfg.blockDim = dim3(32 * (W + 1));
        cfg.dynamicSmemBytes = smem;
        cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        attr[0].val.programmaticStreamSerializationAllowed = 1;
        static const bool pdl = !getenv("VBQ_NO_PDL");
        cfg.attrs = attr;
        cfg.numAttrs = pdl ? 1 : 0;
        CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, a, maps, up));
    }
    return VBQ_OK;
}

