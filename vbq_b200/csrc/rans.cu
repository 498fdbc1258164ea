// rans.cu — entropy coding of the sorted quantile indices: a 32-lane interleaved rANS coder with one frequency table
// per (plane, channel).  The reference stops at ideal code lengths (-log2 of the fitted frequency, quantizer.py:226-228);
// this turns the symbols of the search kernels into bytes and the bytes back into symbols and z_hat.
//
// Stream layout (normative; tests/rans_reference.py restates it in NumPy):
//   * a plane is (items, item_rows, C) symbols q in [0, Q), Q = 2^(N+1)-1; a GROUP is (item, row segment of seg_rows
//     rows, 32-channel group g); lane j of group g codes channel 32g+j (only lanes with 32g+j < C exist) over the
//     segment's rows in increasing order;
//   * rANS with a 32-bit state x in [2^16, 2^32), 16-bit words, probabilities of P = prob_bits <= 16 bits: a symbol
//     moves at most one word per lane, so a warp finds every lane's word offset with one ballot and popc;
//   * the decoder defines the format: read the active lanes' initial states (two words each, low half first); for each
//     row, for each active lane in increasing order: slot = x & (2^P-1), s the symbol with cum[s] <= slot < cum[s]+f[s],
//     x = f[s] (x >> P) + slot - cum[s], and if x < 2^16 then x = (x << 16) | next word of the group.  After the last
//     row every state equals 2^16 and every word of the group has been read;
//   * the payload of a plane is its group end offset table (uint32 per group, in 16-bit words from the start of the
//     plane's group data, groups in (item, segment, channel group) order) followed by the groups, each its states and
//     then its words.  The payload of a call is its planes' payloads back to back.
#include <climits>

#include "common.h"

namespace {

constexpr int kRansWarps = 8;
constexpr unsigned kRansL = 1u << 16;
constexpr int kRansBuckets = 256;   // coarse decode index: slot >> (P - 8) -> first candidate symbol

struct RansShape {
    int n_planes, items, C, CG, P, Q;
    long long item_rows, seg_rows, n_segs, G;   // G = groups per plane
};

int rans_shape(const char *fn, int n_planes, int items, long long item_rows, int C, long long seg_rows, int N,
               int prob_bits, RansShape *s) {
    if (n_planes < 1 || n_planes > 65535 || items < 0 || item_rows < 0 || C < 1 || C > 32 * 65535 || seg_rows < 1)
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "%s: n_planes=%d items=%d item_rows=%lld C=%d seg_rows=%lld", fn, n_planes,
                        items, item_rows, C, seg_rows);
    if (N < 0 || N > 10) return vbq_fail(VBQ_ERR_BAD_DEPTH, "%s: N=%d (the coder holds N <= 10)", fn, N);
    const int Q = (1 << (N + 1)) - 1;
    if (prob_bits < 12 || prob_bits > 16 || Q > (1 << prob_bits))
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "%s: prob_bits=%d (12..16 with Q=%d <= 2^prob_bits)", fn, prob_bits, Q);
    s->n_planes = n_planes; s->items = items; s->C = C; s->CG = (C + 31) / 32; s->P = prob_bits; s->Q = Q;
    s->item_rows = item_rows; s->seg_rows = seg_rows;
    s->n_segs = (item_rows + seg_rows - 1) / seg_rows;
    s->G = (long long)items * s->n_segs * s->CG;
    // worst-case words of a plane: every lane emits a word on every row, plus its state, plus the offset table
    const double words = (double)items * s->n_segs * C * ((double)seg_rows + 2.0) + 2.0 * (double)s->G;
    if (words >= 4294967296.0 || (double)items * s->n_segs >= 2147483647.0 * kRansWarps ||
        (double)n_planes * s->G >= 2147483647.0)
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "%s: a plane of %d x %lld x %d symbols in segments of %lld rows exceeds "
                        "the 32-bit offset table", fn, items, item_rows, C, seg_rows);
    return VBQ_OK;
}

long long rans_plane_scratch_words(const RansShape &s) {
    return (long long)s.items * s.n_segs * s.C * (s.seg_rows + 2);
}

long long align256(long long b) { return (b + 255) & ~255ll; }

// The 32 channels of a group are consecutive rows of the (n_planes, C, Q) cum table: one linear copy.
__device__ __forceinline__ void load_group_cum(unsigned short *sh_cum, const unsigned short *__restrict__ cum,
                                               int plane, int cg, const RansShape &s) {
    const int nact = min(32, s.C - 32 * cg);
    const unsigned short *src = cum + ((size_t)plane * s.C + 32 * cg) * s.Q;
    const int n = nact * s.Q;
    for (int i = threadIdx.x; i < n; i += blockDim.x) sh_cum[i] = __ldg(src + i);
}

__device__ __forceinline__ unsigned lanemask_lt() {
    unsigned m;
    asm("mov.u32 %0, %%lanemask_lt;" : "=r"(m));
    return m;
}

constexpr int kEncBlock = 16;   // rows whose symbols are loaded together (the next block's loads overlap the coding)

// One warp encodes one group of len rows and nact lanes: rows last to first, lanes high to low, words written back to
// front into scratch below `end`, then the lanes' final states.  src (already offset to the lane's channel) + t C is
// the lane's symbol of row t, tab the lane's cum table.  Returns the group's first word (its states, then its words);
// `bad` becomes 1 on a lane that met a symbol outside [0, Q) (coded as symbol 0).
__device__ __forceinline__ long long rans_encode_group(const int *__restrict__ src, int C, long long len, int nact,
                                                       const unsigned short *tab, int P, int Q,
                                                       unsigned short *__restrict__ scratch, long long end,
                                                       int &bad) {
    const int lane = threadIdx.x & 31;
    const bool active = lane < nact;
    const unsigned top = 1u << P;
    const int fshift = 32 - P;
    long long pos = end;
    unsigned x = kRansL;
    const unsigned lt = lanemask_lt();

    int cur[kEncBlock], nxt[kEncBlock];
#pragma unroll
    for (int k = 0; k < kEncBlock; ++k) {
        const long long t = len - 1 - k;
        cur[k] = (active && t >= 0) ? __ldg(src + t * C) : 0;
    }
    for (long long t0 = len - 1; t0 >= 0; t0 -= kEncBlock) {
#pragma unroll
        for (int k = 0; k < kEncBlock; ++k) {
            const long long t = t0 - kEncBlock - k;
            nxt[k] = (active && t >= 0) ? __ldg(src + t * C) : 0;
        }
#pragma unroll
        for (int k = 0; k < kEncBlock; ++k) {
            if (t0 - k < 0) break;                         // warp-uniform
            int sym = cur[k];
            if (sym < 0 || sym >= Q) { bad = 1; sym = 0; }
            const unsigned lo = tab[sym];
            const unsigned f = (sym + 1 < Q ? (unsigned)tab[sym + 1] : top) - lo;
            const bool emit = active && (unsigned long long)x >= ((unsigned long long)f << fshift);
            const unsigned mask = __ballot_sync(0xffffffffu, emit);
            pos -= __popc(mask);
            if (emit) {
                scratch[pos + __popc(mask & lt)] = (unsigned short)(x & 0xffffu);
                x >>= 16;
            }
            if (active) x = ((x / f) << P) + (x % f) + lo;
        }
#pragma unroll
        for (int k = 0; k < kEncBlock; ++k) cur[k] = nxt[k];
    }
    pos -= 2 * nact;
    if (active) {
        scratch[pos + 2 * lane] = (unsigned short)(x & 0xffffu);
        scratch[pos + 2 * lane + 1] = (unsigned short)(x >> 16);
    }
    return pos;
}

// One warp per (item, segment) of the CTA's channel group, coded into the group's scratch region
// [base, base + nact (seg_rows + 2)).
__global__ void __launch_bounds__(kRansWarps * 32) vbq_rans_encode_kernel(const int *__restrict__ qidx,
                                                                         const unsigned short *__restrict__ cum,
                                                                         RansShape s,
                                                                         unsigned short *__restrict__ scratch,
                                                                         long long *__restrict__ sizes,
                                                                         int *__restrict__ status) {
    extern __shared__ unsigned short sh_cum[];   // [nact][Q]
    const int cg = blockIdx.y, plane = blockIdx.z;
    load_group_cum(sh_cum, cum, plane, cg, s);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const long long unit = (long long)blockIdx.x * kRansWarps + (threadIdx.x >> 5);   // item * n_segs + segment
    if (unit >= (long long)s.items * s.n_segs) return;
    const int item = (int)(unit / s.n_segs);
    const long long r0 = (unit % s.n_segs) * s.seg_rows;
    const long long len = min(s.seg_rows, s.item_rows - r0);
    const int nact = min(32, s.C - 32 * cg);
    const bool active = lane < nact;
    const int c = 32 * cg + lane;
    const int *src = qidx + (((long long)plane * s.items + item) * s.item_rows + r0) * s.C + c;
    const long long base = ((long long)plane * s.items * s.n_segs + unit) * s.C * (s.seg_rows + 2) +
                           32ll * cg * (s.seg_rows + 2);
    const long long end = base + (long long)nact * (s.seg_rows + 2);
    int bad = 0;
    const long long pos = rans_encode_group(src, s.C, len, nact, sh_cum + (active ? lane : 0) * s.Q, s.P, s.Q, scratch,
                                            end, bad);
    const long long g = (((long long)plane * s.items * s.n_segs + unit) * s.CG + cg);
    if (lane == 0) sizes[g] = end - pos;
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr(status, 1);
}

// The work-list encoder of many images (vbq_rans_encode_batch): CTA i stages the table set (table, cg) of descriptor i
// and its warp w codes unit first + w into the unit's scratch range, then records the group's size and scratch end.
// Every field of the descriptor and the unit comes from the caller's memory and is checked before it is used: a bad
// one sets status bit 8 (of the unit's blob if its blob id is in range, else of blob 0) and writes nothing.
__global__ void __launch_bounds__(kRansWarps * 32) vbq_rans_encode_batch_kernel(
        const int *__restrict__ in, long long n_in, const unsigned short *__restrict__ cum,
        const int *__restrict__ prob_bits, int n_tables, int C, int Q, const vbq_rans_encode_unit *__restrict__ units,
        long long n_units, const vbq_rans_batch_cta *__restrict__ ctas, int n_blobs, long long n_groups,
        unsigned short *__restrict__ scratch, long long scratch_words, long long *__restrict__ sizes,
        long long *__restrict__ ends, int *__restrict__ status) {
    extern __shared__ unsigned short sh_cum[];   // [nact][Q]
    const vbq_rans_batch_cta d = ctas[blockIdx.x];
    const int CG = (C + 31) / 32;
    bool ok = d.count >= 1 && d.count <= kRansWarps && d.first >= 0 && d.first <= n_units - d.count &&
              d.table >= 0 && d.table < n_tables && d.cg >= 0 && d.cg < CG;
    const int P = ok ? __ldg(prob_bits + d.table) : 0;
    ok = ok && P >= 12 && P <= 16 && Q <= (1 << P);
    if (!ok) {                                                         // CTA-uniform
        if (threadIdx.x == 0) atomicOr(status, 8);
        return;
    }
    const int cg = (int)d.cg;
    const int nact = min(32, C - 32 * cg);
    const unsigned short *src_cum = cum + ((size_t)d.table * C + 32 * cg) * Q;
    for (int i = threadIdx.x; i < nact * Q; i += blockDim.x) sh_cum[i] = __ldg(src_cum + i);
    __syncthreads();

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (warp >= d.count) return;
    const vbq_rans_encode_unit u = units[d.first + warp];
    const bool blob_ok = u.blob >= 0 && u.blob < n_blobs;
    // the rows lie in the input (in + (rows - 1) C + nact <= n_in) and the worst case in the scratch
    const bool bad = !blob_ok || u.table != d.table || u.cg != d.cg || u.rows < 1 || u.in < 0 || u.rows > n_in / C ||
                     u.in > n_in - ((u.rows - 1) * C + nact) || u.group < 0 || u.group >= n_groups ||
                     u.scratch < 0 || u.scratch > scratch_words - nact * (u.rows + 2);
    int *st = status + (blob_ok ? u.blob : 0);
    if (bad) {
        if (lane == 0) atomicOr(st, 8);
        return;
    }
    const bool active = lane < nact;
    const long long end = u.scratch + nact * (u.rows + 2);
    int sym_bad = 0;
    const long long pos = rans_encode_group(in + u.in + lane, C, u.rows, nact, sh_cum + (active ? lane : 0) * Q, P, Q,
                                            scratch, end, sym_bad);
    if (lane == 0) {
        sizes[u.group] = end - pos;
        ends[u.group] = end;
    }
    if (__any_sync(0xffffffffu, sym_bad) && lane == 0) atomicOr(st, 1);
}

// Block-wide inclusive sum of one value per thread (blockDim.x a multiple of 32, at most 1024).
__device__ long long block_inclusive_sum(long long v, long long *sh_warp, long long *total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long u = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += u;
    }
    if (lane == 31) sh_warp[warp] = v;
    __syncthreads();
    if (warp == 0) {
        long long w = lane < nw ? sh_warp[lane] : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long u = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += u;
        }
        if (lane < nw) sh_warp[lane] = w;
    }
    __syncthreads();
    if (warp > 0) v += sh_warp[warp - 1];
    *total = sh_warp[nw - 1];
    __syncthreads();
    return v;
}

// Block-wide exclusive scan of one plane's G group sizes: writes the plane's offset table at out[plane_start..] and
// each group's destination word; returns the word where the next plane starts.
__device__ long long scan_plane(const long long *__restrict__ sizes, long long *__restrict__ dst, long long G,
                                long long plane_start, unsigned short *__restrict__ out, long long *sh_warp) {
    long long carry = 0;
    for (long long c0 = 0; c0 < G; c0 += blockDim.x) {
        const long long i = c0 + threadIdx.x;
        const long long v = i < G ? sizes[i] : 0;
        long long chunk;
        const long long incl = block_inclusive_sum(v, sh_warp, &chunk);
        if (i < G) {
            const unsigned long long e = (unsigned long long)(carry + incl);
            out[plane_start + 2 * i] = (unsigned short)(e & 0xffffu);
            out[plane_start + 2 * i + 1] = (unsigned short)(e >> 16);
            dst[i] = plane_start + 2 * G + carry + incl - v;
        }
        carry += chunk;
    }
    return plane_start + 2 * G + carry;
}

// One CTA: exclusive scan of the group sizes of every plane -> each group's destination, the planes' offset tables
// and the payload size in bytes.
__global__ void __launch_bounds__(1024) vbq_rans_scan_kernel(const long long *__restrict__ sizes,
                                                            long long *__restrict__ dst, int n_planes, long long G,
                                                            unsigned short *__restrict__ out,
                                                            long long *__restrict__ out_bytes) {
    __shared__ long long sh_warp[32];
    long long plane_start = 0;   // in words
    for (int p = 0; p < n_planes; ++p)
        plane_start = scan_plane(sizes + (long long)p * G, dst + (long long)p * G, G, plane_start, out, sh_warp);
    if (threadIdx.x == 0) *out_bytes = 2 * plane_start;
}

// One CTA per group: move its words from the end of its scratch region to their place in the payload.
__global__ void vbq_rans_compact_kernel(const unsigned short *__restrict__ scratch, const long long *__restrict__ sizes,
                                        const long long *__restrict__ dst, RansShape s,
                                        unsigned short *__restrict__ out) {
    const long long g = blockIdx.x;                  // (plane, item, segment, channel group)
    const int cg = (int)(g % s.CG);
    const long long unit = g / s.CG;                 // (plane, item, segment)
    const int nact = min(32, s.C - 32 * cg);
    const long long end = unit * s.C * (s.seg_rows + 2) + (32ll * cg + nact) * (s.seg_rows + 2);
    const long long n = sizes[g];
    const unsigned short *src = scratch + end - n;
    unsigned short *d = out + dst[g];
    for (long long i = threadIdx.x; i < n; i += blockDim.x) d[i] = src[i];
}

// One CTA: the blobs of vbq_rans_encode_batch back to back.  blob_groups (n_blobs + 1) gives each blob's first group
// in blob-major order; it comes from the caller's memory, so unless it runs from 0 to n_groups without decreasing the
// kernel sets bit 8 of blob 0, zeroes blob_starts and marks every group as not to be moved (dst = -1).  Otherwise:
// dst[g] = the exclusive prefix of the sizes (first pass), blob_starts[b] = 2 (first group) + prefix at the first group
// (second pass), then each group's offset-table entry and its destination word (third pass; a group finds its blob by
// binary search).  Table words that would fall outside the payload are not written.
__global__ void __launch_bounds__(1024) vbq_rans_encode_batch_scan_kernel(
        const long long *__restrict__ sizes, long long *__restrict__ dst, long long n_groups,
        const long long *__restrict__ blob_groups, int n_blobs, unsigned short *__restrict__ out, long long out_words,
        long long *__restrict__ blob_starts, int *__restrict__ status) {
    __shared__ long long sh_warp[32];
    bool bad = false;
    for (int b = threadIdx.x; b <= n_blobs; b += blockDim.x) {
        const long long g = blob_groups[b];
        bad = bad || (b == 0 ? g != 0 : g < blob_groups[b - 1]) || (b == n_blobs && g != n_groups);
    }
    if (__syncthreads_or(bad)) {
        for (int b = threadIdx.x; b <= n_blobs; b += blockDim.x) blob_starts[b] = 0;
        for (long long g = threadIdx.x; g < n_groups; g += blockDim.x) dst[g] = -1;
        if (threadIdx.x == 0) atomicOr(status, 8);
        return;
    }
    long long total = 0;
    for (long long c0 = 0; c0 < n_groups; c0 += blockDim.x) {
        const long long i = c0 + threadIdx.x;
        const long long v = i < n_groups ? sizes[i] : 0;
        long long chunk;
        const long long incl = block_inclusive_sum(v, sh_warp, &chunk);
        if (i < n_groups) dst[i] = total + incl - v;
        total += chunk;
    }
    __syncthreads();
    for (int b = threadIdx.x; b <= n_blobs; b += blockDim.x) {
        const long long g = blob_groups[b];
        blob_starts[b] = 2 * g + (g < n_groups ? dst[g] : total);
    }
    __syncthreads();
    for (long long g = threadIdx.x; g < n_groups; g += blockDim.x) {
        int lo = 0, hi = n_blobs - 1;                      // the last blob whose first group is <= g holds g
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (blob_groups[mid] <= g) lo = mid; else hi = mid - 1;
        }
        const long long g0 = blob_groups[lo], start = blob_starts[lo];
        const long long data = start + 2 * (blob_groups[lo + 1] - g0);   // the blob's group data
        const long long excl = dst[g] - (start - 2 * g0);                // words of the blob's groups before g
        const unsigned long long e = (unsigned long long)(excl + sizes[g]);
        const long long w = start + 2 * (g - g0);
        if (w + 1 < out_words) {
            out[w] = (unsigned short)(e & 0xffffu);
            out[w + 1] = (unsigned short)(e >> 16);
        }
        dst[g] = data + excl;
    }
}

// One CTA per group of vbq_rans_encode_batch: move its words from the end of its scratch range to their place in the
// payload.  A group of size 0 (no unit, or a bad one) moves nothing; the clamps keep every access inside the scratch
// and the payload even when duplicate units of one group left the size of one and the scratch end of another.
__global__ void vbq_rans_encode_batch_compact_kernel(const unsigned short *__restrict__ scratch,
                                                     const long long *__restrict__ sizes,
                                                     const long long *__restrict__ ends,
                                                     const long long *__restrict__ dst,
                                                     unsigned short *__restrict__ out, long long out_words) {
    const long long g = blockIdx.x;
    const long long size = sizes[g];
    if (size <= 0) return;                           // ends[g] is written together with a nonzero size
    const long long end = ends[g], d = dst[g];
    const long long n = min(size, end);
    if (d < 0) return;
    const unsigned short *src = scratch + end - n;
    const long long m = min(n, out_words - d);
    for (long long i = threadIdx.x; i < m; i += blockDim.x) out[d + i] = src[i];
}

constexpr int kDecBlock = 8;   // rows per unrolled block; z_hat gathers of a block are stored one block later

__device__ __forceinline__ unsigned short ld_word(const unsigned short *__restrict__ w, long long i, long long end) {
    return i < end ? __ldg(w + i) : (unsigned short)0;
}

// Shared memory of the VBQ2 decoders: the 32-channel group's cum tables [nact][Q] (a linear copy of nact Q entries
// from src) and the coarse index [32][257]: idx[j][b] = the symbol whose slot range holds b << (P - 8), and
// idx[j][256] = Q - 1.  Every thread of the CTA takes part (two barriers).
__device__ __forceinline__ void stage_group_table(unsigned short *sh_cum, unsigned short *sh_idx,
                                                  const unsigned short *__restrict__ src, int nact, int Q, int P) {
    for (int i = threadIdx.x; i < nact * Q; i += blockDim.x) sh_cum[i] = __ldg(src + i);
    __syncthreads();
    const int bshift = P - 8;
    const unsigned top = 1u << P;
    // every bucket start lies in exactly one symbol
    for (int k = threadIdx.x; k < nact * Q; k += blockDim.x) {
        const int j = k / Q, q = k - j * Q;
        const unsigned lo = sh_cum[k], hi = q + 1 < Q ? (unsigned)sh_cum[k + 1] : top;
        for (unsigned b = (lo + (1u << bshift) - 1) >> bshift; (b << bshift) < hi && b < kRansBuckets; ++b)
            sh_idx[j * (kRansBuckets + 1) + b] = (unsigned short)q;
    }
    for (int j = threadIdx.x; j < nact; j += blockDim.x) sh_idx[j * (kRansBuckets + 1) + kRansBuckets] = (unsigned short)(Q - 1);
    __syncthreads();
}

// One warp decodes one VBQ2 group of len rows and nact state lanes from its word range [start, end) (err = 4 with
// start = end = 0 for a range the caller rejected): symbol of row t, lane j goes to qidx / zhat[out0 + t C] of lane j,
// with out0 and cp (the lane's code points) already offset to the lane's channel.  tab / cidx are the lane's table and
// coarse index.  A warp keeps the next 128 words of its group in registers (4 windows of 32, one word per lane) and
// reads each row's words with shuffles; a window is refilled 64..96 words before it is needed.  Returns the status
// bits 1, 2 and 4 of vbq_rans_decode, the same on every lane.
__device__ __forceinline__ int vbq2_decode_group(const unsigned short *__restrict__ words, long long start,
                                                 long long end, int err, const unsigned short *tab,
                                                 const unsigned short *cidx, int P, int Q, int nact, long long len,
                                                 int C, long long out0, const float *__restrict__ cp,
                                                 int *__restrict__ qidx, float *__restrict__ zhat) {
    const int lane = threadIdx.x & 31;
    const bool active = lane < nact;
    const int bshift = P - 8;
    const unsigned top = 1u << P;
    const unsigned lt = lanemask_lt();

    unsigned x = kRansL;
    if (!err && active) x = (unsigned)__ldg(words + start + 2 * lane) | ((unsigned)__ldg(words + start + 2 * lane + 1) << 16);
    if (__any_sync(0xffffffffu, active && x < kRansL)) err |= 4;
    long long pos = start + 2 * nact;
    long long wbase = pos;
    unsigned w0 = ld_word(words, wbase + lane, end), w1 = ld_word(words, wbase + 32 + lane, end);
    unsigned w2 = ld_word(words, wbase + 64 + lane, end), w3 = ld_word(words, wbase + 96 + lane, end);

    // z_hat of a block is gathered after the block and stored after the next one, so the gather's latency never stalls
    // the state chain
    float zprev[kDecBlock];
    long long tprev = -1;
    for (long long t0 = 0; t0 < len && !err; t0 += kDecBlock) {
        int sy[kDecBlock];
#pragma unroll
        for (int k = 0; k < kDecBlock; ++k) {
            sy[k] = 0;
            if (t0 + k >= len) break;                      // warp-uniform
            const unsigned slot = x & (top - 1);
            int lo = min((int)cidx[slot >> bshift], Q - 1), hi = min((int)cidx[(slot >> bshift) + 1], Q - 1);
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (tab[mid] <= slot) lo = mid; else hi = mid - 1;
            }
            const unsigned c0 = tab[lo];
            const unsigned f = (lo + 1 < Q ? (unsigned)tab[lo + 1] : top) - c0;
            x = f * (x >> P) + slot - c0;
            const bool need = active && x < kRansL;
            const unsigned mask = __ballot_sync(0xffffffffu, need);
            const int n = __popc(mask);
            if (pos + n > end) { err |= 1; break; }
            const int rel = (int)(pos - wbase) + __popc(mask & lt);   // < 64 for the lanes that read
            const unsigned a = __shfl_sync(0xffffffffu, w0, rel & 31), b = __shfl_sync(0xffffffffu, w1, rel & 31);
            if (need) x = (x << 16) | (rel < 32 ? a : b);
            pos += n;
            if (pos - wbase >= 32) {
                w0 = w1; w1 = w2; w2 = w3;
                wbase += 32;
                w3 = ld_word(words, wbase + 96 + lane, end);
            }
            sy[k] = lo;
        }
        if (zhat && tprev >= 0) {
#pragma unroll
            for (int k = 0; k < kDecBlock; ++k)
                if (active) zhat[out0 + (tprev + k) * C] = zprev[k];   // a previous block is always full
        }
        if (err) break;
#pragma unroll
        for (int k = 0; k < kDecBlock; ++k) {
            if (active && t0 + k < len) {
                if (qidx) qidx[out0 + (t0 + k) * C] = sy[k];
                if (zhat) zprev[k] = __ldg(cp + sy[k]);
            }
        }
        tprev = t0;
    }
    if (zhat && tprev >= 0 && !err) {
#pragma unroll
        for (int k = 0; k < kDecBlock; ++k)
            if (active && tprev + k < len) zhat[out0 + (tprev + k) * C] = zprev[k];
    }
    if (!err && (__any_sync(0xffffffffu, active && x != kRansL) || pos != end)) err |= 2;
    return err;
}

// Same CTA layout as the encoder: CTA (x, cg, plane), one warp per (item, segment) of its channel group.
__global__ void __launch_bounds__(kRansWarps * 32) vbq_rans_decode_kernel(const unsigned short *__restrict__ words,
                                                                         long long n_words,
                                                                         const long long *__restrict__ bounds,
                                                                         const unsigned short *__restrict__ cum,
                                                                         RansShape s,
                                                                         const float *__restrict__ code_points,
                                                                         int *__restrict__ qidx,
                                                                         float *__restrict__ zhat,
                                                                         int *__restrict__ status) {
    extern __shared__ unsigned short sh_cum[];   // [32][Q] then [32][kRansBuckets + 1]
    const int cg = blockIdx.y, plane = blockIdx.z;
    unsigned short *sh_idx = sh_cum + 32 * s.Q;
    const int nact = min(32, s.C - 32 * cg);
    stage_group_table(sh_cum, sh_idx, cum + ((size_t)plane * s.C + 32 * cg) * s.Q, nact, s.Q, s.P);

    const int lane = threadIdx.x & 31;
    const long long unit = (long long)blockIdx.x * kRansWarps + (threadIdx.x >> 5);
    if (unit >= (long long)s.items * s.n_segs) return;
    const int item = (int)(unit / s.n_segs);
    const long long r0 = (unit % s.n_segs) * s.seg_rows;
    const long long len = min(s.seg_rows, s.item_rows - r0);
    const bool active = lane < nact;
    const int c = 32 * cg + lane;
    const long long g = (((long long)plane * s.items * s.n_segs + unit) * s.CG + cg);
    long long start = bounds[2 * g], end = bounds[2 * g + 1];
    int err = 0;
    if (start < 0 || end > n_words || end - start < 2ll * nact) { err = 4; end = start = 0; }
    err = vbq2_decode_group(words, start, end, err, sh_cum + (active ? lane : 0) * s.Q,
                            sh_idx + (active ? lane : 0) * (kRansBuckets + 1), s.P, s.Q, nact, len, s.C,
                            (((long long)plane * s.items + item) * s.item_rows + r0) * s.C + c,
                            code_points + (size_t)(active ? c : 0) * s.Q, qidx, zhat);
    if (err && lane == 0) atomicOr(status, err);
}

// The work-list decoder of many VBQ2 streams (vbq_rans_decode_batch): CTA i stages the table set (table, cg) of
// descriptor i and its warp w decodes unit first + w.  Every field of the descriptor and the unit comes from the
// caller's memory and is checked before it is used: a bad one sets status bit 8 (of the unit's blob if its blob id is
// in range, else of blob 0) and writes nothing.
__global__ void __launch_bounds__(kRansWarps * 32) vbq_rans_decode_batch_kernel(
        const unsigned short *__restrict__ words, long long n_words, const unsigned short *__restrict__ cum,
        const int *__restrict__ prob_bits, int n_tables, int C, int Q, const vbq_rans_batch_unit *__restrict__ units,
        long long n_units, const vbq_rans_batch_cta *__restrict__ ctas, int n_blobs,
        const float *__restrict__ code_points, long long n_out, int *__restrict__ qidx, float *__restrict__ zhat,
        int *__restrict__ status) {
    extern __shared__ unsigned short sh_cum[];   // [32][Q] then [32][kRansBuckets + 1]
    unsigned short *sh_idx = sh_cum + 32 * Q;
    const vbq_rans_batch_cta d = ctas[blockIdx.x];
    const int CG = (C + 31) / 32;
    bool ok = d.count >= 1 && d.count <= kRansWarps && d.first >= 0 && d.first <= n_units - d.count &&
              d.table >= 0 && d.table < n_tables && d.cg >= 0 && d.cg < CG;
    const int P = ok ? __ldg(prob_bits + d.table) : 0;
    ok = ok && P >= 12 && P <= 16 && Q <= (1 << P);
    if (!ok) {                                                         // CTA-uniform
        if (threadIdx.x == 0) atomicOr(status, 8);
        return;
    }
    const int cg = (int)d.cg;
    const int nact = min(32, C - 32 * cg);
    stage_group_table(sh_cum, sh_idx, cum + ((size_t)d.table * C + 32 * cg) * Q, nact, Q, P);

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (warp >= d.count) return;
    const vbq_rans_batch_unit u = units[d.first + warp];
    const bool blob_ok = u.blob >= 0 && u.blob < n_blobs;
    // the word range holds the states, the rows fit the output: out + (rows - 1) C + nact <= n_out
    const bool bad = !blob_ok || u.table != d.table || u.cg != d.cg || u.start < 0 || u.end > n_words ||
                     u.end - u.start < 2ll * nact || u.rows < 1 || u.out < 0 || u.rows > n_out / C ||
                     u.out > n_out - ((u.rows - 1) * C + nact);
    int *st = status + (blob_ok ? u.blob : 0);
    if (bad) {
        if (lane == 0) atomicOr(st, 8);
        return;
    }
    const bool active = lane < nact;
    const int c = 32 * cg + lane;
    const int err = vbq2_decode_group(words, u.start, u.end, 0, sh_cum + (active ? lane : 0) * Q,
                                      sh_idx + (active ? lane : 0) * (kRansBuckets + 1), P, Q, nact, u.rows, C,
                                      u.out + lane, code_points + (size_t)(active ? c : 0) * Q, qidx, zhat);
    if (err && lane == 0) atomicOr(st, err);
}

// ---- the shared-table layout (vbq_rans_shared_*): one table per plane, symbols as one flat sequence ----------------
//
// Symbol k of a plane sits at row k / 32, lane k % 32; a group is a segment of seg_rows rows (seg_rows per plane), coded
// by one warp.  Only the plane's last row can be partial.  The table is staged once per CTA (8 KiB at N = 10), so many
// small CTAs share an SM and hide the dependent state chain of each warp.

constexpr int kSharedWarps = 4;

struct SharedShape {
    int n_planes, P, Q;
    long long n, rows;                             // symbols per plane, rows = ceil(n / 32)
    long long seg[VBQ_RANS_SHARED_MAX_PLANES];     // seg_rows of each plane
    long long gbase[VBQ_RANS_SHARED_MAX_PLANES + 1];   // the call's first group of each plane; [n_planes] = all groups
    long long sbase[VBQ_RANS_SHARED_MAX_PLANES + 1];   // first encoder scratch word of each plane
    long long max_groups;                          // of any plane
};

int shared_shape(const char *fn, int n_planes, long long n, const long long *seg_rows, int N, int prob_bits,
                 SharedShape *s) {
    if (n_planes < 1 || n_planes > VBQ_RANS_SHARED_MAX_PLANES || n < 0)
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "%s: n_planes=%d (1..%d) n=%lld", fn, n_planes, VBQ_RANS_SHARED_MAX_PLANES, n);
    if (!seg_rows) return vbq_fail(VBQ_ERR_NULL_POINTER, "%s: seg_rows is NULL", fn);
    if (N < 0 || N > 10) return vbq_fail(VBQ_ERR_BAD_DEPTH, "%s: N=%d (the coder holds N <= 10)", fn, N);
    const int Q = (1 << (N + 1)) - 1;
    if (prob_bits < 12 || prob_bits > 16 || Q > (1 << prob_bits))
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "%s: prob_bits=%d (12..16 with Q=%d <= 2^prob_bits)", fn, prob_bits, Q);
    s->n_planes = n_planes; s->P = prob_bits; s->Q = Q; s->n = n; s->rows = n / 32 + (n % 32 != 0);
    s->gbase[0] = 0; s->sbase[0] = 0; s->max_groups = 0;
    for (int p = 0; p < n_planes; ++p) {
        if (seg_rows[p] < 1) return vbq_fail(VBQ_ERR_BAD_SHAPE, "%s: seg_rows[%d]=%lld", fn, p, seg_rows[p]);
        // a segment longer than the plane is the whole plane: clamp before the scratch is sized from it
        const long long seg = min(seg_rows[p], max(s->rows, 1ll));
        const long long G = (s->rows + seg - 1) / seg;
        // worst-case words of the plane: a word per symbol, two per lane and group, its offset table
        if ((double)n + 66.0 * (double)G >= 4294967296.0 || (double)s->gbase[p] + G >= 2147483647.0)
            return vbq_fail(VBQ_ERR_BAD_SHAPE, "%s: a plane of %lld symbols in segments of %lld rows exceeds the 32-bit "
                            "offset table", fn, n, seg);
        s->seg[p] = seg;
        s->gbase[p + 1] = s->gbase[p] + G;
        s->sbase[p + 1] = s->sbase[p] + G * 32 * (seg + 2);
        s->max_groups = max(s->max_groups, G);
    }
    return VBQ_OK;
}

// Lanes of row r of a plane that hold a symbol.
__device__ __forceinline__ int shared_row_lanes(const SharedShape &s, long long r) {
    return r == s.rows - 1 ? (int)(s.n - 32 * (s.rows - 1)) : 32;
}

__device__ __forceinline__ void load_plane_cum(unsigned *sh_cum, const unsigned *__restrict__ cum, int plane, int Q) {
    const unsigned *src = cum + (size_t)plane * (Q + 1);
    for (int i = threadIdx.x; i <= Q; i += blockDim.x) sh_cum[i] = __ldg(src + i);
}

// One warp per group: rows last to first, lanes high to low, words written back to front into the group's scratch
// region [base, base + 32 (seg + 2)).  Status: 1 for a symbol outside [0, Q), 2 for a symbol of frequency 0.
__global__ void __launch_bounds__(kSharedWarps * 32) vbq_rans_shared_encode_kernel(const int *__restrict__ qidx,
                                                                                  const unsigned *__restrict__ cum,
                                                                                  SharedShape s,
                                                                                  unsigned short *__restrict__ scratch,
                                                                                  long long *__restrict__ sizes,
                                                                                  int *__restrict__ status) {
    extern __shared__ unsigned sh_tab[];   // [Q + 1]
    const int plane = blockIdx.y;
    const long long G = s.gbase[plane + 1] - s.gbase[plane];
    if ((long long)blockIdx.x * kSharedWarps >= G) return;   // CTA-uniform
    load_plane_cum(sh_tab, cum, plane, s.Q);
    __syncthreads();
    const long long g = (long long)blockIdx.x * kSharedWarps + (threadIdx.x >> 5);
    if (g >= G) return;
    const int lane = threadIdx.x & 31;
    const long long seg = s.seg[plane];
    const long long r0 = g * seg;
    const long long len = min(seg, s.rows - r0);
    const int *src = qidx + (long long)plane * s.n + r0 * 32 + lane;
    const unsigned top = 1u << s.P;
    const int fshift = 32 - s.P;
    const long long base = s.sbase[plane] + g * 32 * (seg + 2);
    long long pos = base + 32 * (seg + 2);
    const long long end = pos;
    unsigned x = kRansL;
    int bad = 0;
    const unsigned lt = lanemask_lt();

    int cur[kEncBlock], nxt[kEncBlock];
#pragma unroll
    for (int k = 0; k < kEncBlock; ++k) {
        const long long t = len - 1 - k;
        cur[k] = (t >= 0 && lane < shared_row_lanes(s, r0 + t)) ? __ldg(src + t * 32) : 0;
    }
    for (long long t0 = len - 1; t0 >= 0; t0 -= kEncBlock) {
#pragma unroll
        for (int k = 0; k < kEncBlock; ++k) {
            const long long t = t0 - kEncBlock - k;
            nxt[k] = (t >= 0 && lane < shared_row_lanes(s, r0 + t)) ? __ldg(src + t * 32) : 0;
        }
#pragma unroll
        for (int k = 0; k < kEncBlock; ++k) {
            if (t0 - k < 0) break;                         // warp-uniform
            const bool active = lane < shared_row_lanes(s, r0 + t0 - k);
            const int sym = cur[k];
            unsigned lo = 0, f = top;                      // f = 2^P leaves the state unchanged
            if (active) {
                if (sym < 0 || sym >= s.Q) {
                    bad |= 1;
                } else {
                    lo = sh_tab[sym];
                    f = sh_tab[sym + 1] - lo;
                    if (f == 0) { bad |= 2; lo = 0; f = top; }
                }
            }
            const bool emit = active && (unsigned long long)x >= ((unsigned long long)f << fshift);
            const unsigned mask = __ballot_sync(0xffffffffu, emit);
            pos -= __popc(mask);
            if (emit) {
                scratch[pos + __popc(mask & lt)] = (unsigned short)(x & 0xffffu);
                x >>= 16;
            }
            if (active) x = ((x / f) << s.P) + (x % f) + lo;
        }
#pragma unroll
        for (int k = 0; k < kEncBlock; ++k) cur[k] = nxt[k];
    }
    const int nact = shared_row_lanes(s, r0);
    pos -= 2 * nact;
    if (lane < nact) {
        scratch[pos + 2 * lane] = (unsigned short)(x & 0xffffu);
        scratch[pos + 2 * lane + 1] = (unsigned short)(x >> 16);
    }
    if (lane == 0) sizes[s.gbase[plane] + g] = end - pos;
    bad = __reduce_or_sync(0xffffffffu, bad);
    if (bad && lane == 0) atomicOr(status, bad);
}

// One CTA: the offset tables of every plane, each group's destination and the payload size in bytes.  (The minimum of
// one CTA per SM lets ptxas use more than 32 registers, which keeps the plane loop free of spills.)
__global__ void __launch_bounds__(1024, 1) vbq_rans_shared_scan_kernel(const long long *__restrict__ sizes,
                                                                   long long *__restrict__ dst, SharedShape s,
                                                                   unsigned short *__restrict__ out,
                                                                   long long *__restrict__ out_bytes) {
    __shared__ long long sh_warp[32];
    long long plane_start = 0;
    for (int p = 0; p < s.n_planes; ++p)
        plane_start = scan_plane(sizes + s.gbase[p], dst + s.gbase[p], s.gbase[p + 1] - s.gbase[p], plane_start, out,
                                 sh_warp);
    if (threadIdx.x == 0) *out_bytes = 2 * plane_start;
}

// One CTA per group of the call: move its words from the end of its scratch region to their place in the payload.
__global__ void vbq_rans_shared_compact_kernel(const unsigned short *__restrict__ scratch,
                                               const long long *__restrict__ sizes, const long long *__restrict__ dst,
                                               SharedShape s, unsigned short *__restrict__ out) {
    const long long gid = blockIdx.x;
    int p = 0;
    while (s.gbase[p + 1] <= gid) ++p;
    const long long g = gid - s.gbase[p];
    const long long end = s.sbase[p] + (g + 1) * 32 * (s.seg[p] + 2);
    const long long n = sizes[gid];
    const unsigned short *src = scratch + end - n;
    unsigned short *d = out + dst[gid];
    for (long long i = threadIdx.x; i < n; i += blockDim.x) d[i] = src[i];
}

// Shared memory of the shared-table decoders: the plane's cum table [Q + 1] and the coarse index
// idx[b] = the largest s < Q with cum[s] <= b << (P - 8), b = 0..256, which brackets the decoded symbol of a slot in
// bucket b between idx[b] and idx[b + 1].  Every thread of the CTA takes part (two barriers).
__device__ __forceinline__ void stage_shared_table(unsigned *sh_tab, unsigned short *sh_idx,
                                                   const unsigned *__restrict__ cum, int plane, const SharedShape &s) {
    load_plane_cum(sh_tab, cum, plane, s.Q);
    __syncthreads();
    const int bshift = s.P - 8;
    for (int b = threadIdx.x; b <= kRansBuckets; b += blockDim.x) {
        const unsigned v = (unsigned)b << bshift;
        int lo = 0, hi = s.Q - 1;
        while (lo < hi) {
            const int mid = (lo + hi + 1) >> 1;
            if (sh_tab[mid] <= v) lo = mid; else hi = mid - 1;
        }
        sh_idx[b] = (unsigned short)lo;
    }
    __syncthreads();
}

// A warp's decoder of one group in the shared-table layout is the lanes' states x, the group's next word pos and its
// end, and a window of the next 128 words in registers (w0..w3, one word per lane each; wbase <= pos < wbase + 32).
// The helpers take them as references rather than as one struct: with a struct ptxas adds register moves to every row
// of the unrolled decode loop.

// (Re)load the window at pos: after the initial states, or at a checkpoint.
__device__ __forceinline__ void shared_load_window(const unsigned short *__restrict__ words, long long pos,
                                                   long long end, int lane, long long &wbase, unsigned &w0,
                                                   unsigned &w1, unsigned &w2, unsigned &w3) {
    wbase = pos;
    w0 = ld_word(words, wbase + lane, end);
    w1 = ld_word(words, wbase + 32 + lane, end);
    w2 = ld_word(words, wbase + 64 + lane, end);
    w3 = ld_word(words, wbase + 96 + lane, end);
}

// Row r of the plane in the shared-table decoder (the DECODER rule of include/vbq_b200.h): coarse index, binary
// search, state update and renormalisation of the lanes that hold a symbol on this row, then the window moves on.
// Returns false on every lane if the group ran out of words (the state is then undefined), else the lane's symbol is
// in `sym`.
__device__ __forceinline__ bool shared_decode_row(unsigned &x, long long &pos, long long &wbase, long long end,
                                                  unsigned &w0, unsigned &w1, unsigned &w2, unsigned &w3,
                                                  const SharedShape &s, long long r, const unsigned *sh_tab,
                                                  const unsigned short *sh_idx,
                                                  const unsigned short *__restrict__ words, int lane, unsigned lt,
                                                  int &sym) {
    const int bshift = s.P - 8;
    const unsigned top = 1u << s.P;
    const bool active = lane < shared_row_lanes(s, r);
    const unsigned slot = x & (top - 1);
    int lo = sh_idx[slot >> bshift], hi = sh_idx[(slot >> bshift) + 1];
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (sh_tab[mid] <= slot) lo = mid; else hi = mid - 1;
    }
    const unsigned c0 = sh_tab[lo];
    const unsigned f = sh_tab[lo + 1] - c0;
    x = active ? f * (x >> s.P) + slot - c0 : x;   // a select: ptxas would branch around the table loads for an if
    const bool need = active && x < kRansL;
    const unsigned mask = __ballot_sync(0xffffffffu, need);
    const int n = __popc(mask);
    if (pos + n > end) return false;
    const int rel = (int)(pos - wbase) + __popc(mask & lt);   // < 64 for the lanes that read
    const unsigned a = __shfl_sync(0xffffffffu, w0, rel & 31), b = __shfl_sync(0xffffffffu, w1, rel & 31);
    if (need) x = (x << 16) | (rel < 32 ? a : b);
    pos += n;
    if (pos - wbase >= 32) {
        w0 = w1; w1 = w2; w2 = w3;
        wbase += 32;
        w3 = ld_word(words, wbase + 96 + lane, end);
    }
    sym = lo;
    return true;
}

// Same CTA layout as the encoder; shared memory as stage_shared_table.  Deferred z_hat stores as in
// vbq_rans_decode_kernel.
__global__ void __launch_bounds__(kSharedWarps * 32) vbq_rans_shared_decode_kernel(
        const unsigned short *__restrict__ words, long long n_words, const long long *__restrict__ bounds,
        const unsigned *__restrict__ cum, SharedShape s, const float *__restrict__ code_points,
        int *__restrict__ qidx, float *__restrict__ zhat, int *__restrict__ status) {
    extern __shared__ unsigned sh_tab[];   // [Q + 1] then [kRansBuckets + 1] uint16
    unsigned short *sh_idx = (unsigned short *)(sh_tab + s.Q + 1);
    const int plane = blockIdx.y;
    const long long G = s.gbase[plane + 1] - s.gbase[plane];
    if ((long long)blockIdx.x * kSharedWarps >= G) return;   // CTA-uniform
    stage_shared_table(sh_tab, sh_idx, cum, plane, s);

    const long long g = (long long)blockIdx.x * kSharedWarps + (threadIdx.x >> 5);
    if (g >= G) return;
    const int lane = threadIdx.x & 31;
    const long long seg = s.seg[plane];
    const long long r0 = g * seg;
    const long long len = min(seg, s.rows - r0);
    const int nact = shared_row_lanes(s, r0);
    const long long gid = s.gbase[plane] + g;
    long long start = bounds[2 * gid], end = bounds[2 * gid + 1];
    int err = 0;
    if (start < 0 || end > n_words || end - start < 2ll * nact) { err = 4; end = start = 0; }
    const long long out0 = (long long)plane * s.n + r0 * 32 + lane;
    const unsigned lt = lanemask_lt();

    unsigned x = kRansL;
    if (!err && lane < nact)
        x = (unsigned)__ldg(words + start + 2 * lane) | ((unsigned)__ldg(words + start + 2 * lane + 1) << 16);
    if (__any_sync(0xffffffffu, lane < nact && x < kRansL)) err |= 4;
    long long pos = start + 2 * nact, wbase;
    unsigned w0, w1, w2, w3;
    shared_load_window(words, pos, end, lane, wbase, w0, w1, w2, w3);

    float zprev[kDecBlock];
    long long tprev = -1;
    for (long long t0 = 0; t0 < len && !err; t0 += kDecBlock) {
        int sy[kDecBlock];
#pragma unroll
        for (int k = 0; k < kDecBlock; ++k) {
            sy[k] = 0;
            if (t0 + k >= len) break;                      // warp-uniform
            if (!shared_decode_row(x, pos, wbase, end, w0, w1, w2, w3, s, r0 + t0 + k, sh_tab, sh_idx, words, lane, lt,
                                   sy[k])) { err |= 1; break; }
        }
        if (zhat && tprev >= 0) {
#pragma unroll
            for (int k = 0; k < kDecBlock; ++k) zhat[out0 + (tprev + k) * 32] = zprev[k];   // a full block, full rows
        }
        if (err) break;
#pragma unroll
        for (int k = 0; k < kDecBlock; ++k) {
            if (t0 + k < len && lane < shared_row_lanes(s, r0 + t0 + k)) {
                if (qidx) qidx[out0 + (t0 + k) * 32] = sy[k];
                if (zhat) zprev[k] = __ldg(code_points + sy[k]);
            }
        }
        tprev = t0;
    }
    if (zhat && tprev >= 0 && !err) {
#pragma unroll
        for (int k = 0; k < kDecBlock; ++k)
            if (tprev + k < len && lane < shared_row_lanes(s, r0 + tprev + k)) zhat[out0 + (tprev + k) * 32] = zprev[k];
    }
    if (!err && (__any_sync(0xffffffffu, lane < nact && x != kRansL) || pos != end)) err |= 2;
    if (err && lane == 0) atomicOr(status, err);
}

// ---- decoder checkpoints and row lookups (vbq_rans_shared_checkpoints / _decode_rows) -------------------------------
//
// A checkpoint is the warp's word offset from its group's start and the 32 lane states just before row j K of a segment
// (j >= 1); segment g's checkpoints are entries g (seg - 1) / K + j - 1 of the index (K clamped to seg on the host).

// Decode one plane exactly as vbq_rans_shared_decode_kernel (same bounds, status bits and final integrity rule), write
// no symbols, and record every checkpoint.
__global__ void __launch_bounds__(kSharedWarps * 32) vbq_rans_shared_checkpoints_kernel(
        const unsigned short *__restrict__ words, long long n_words, const long long *__restrict__ bounds,
        const unsigned *__restrict__ cum, SharedShape s, long long K, unsigned *__restrict__ cp_offsets,
        unsigned *__restrict__ cp_states, int *__restrict__ status) {
    extern __shared__ unsigned sh_tab[];   // [Q + 1] then [kRansBuckets + 1] uint16
    unsigned short *sh_idx = (unsigned short *)(sh_tab + s.Q + 1);
    const long long G = s.gbase[1];
    if ((long long)blockIdx.x * kSharedWarps >= G) return;   // CTA-uniform
    stage_shared_table(sh_tab, sh_idx, cum, 0, s);

    const long long g = (long long)blockIdx.x * kSharedWarps + (threadIdx.x >> 5);
    if (g >= G) return;
    const int lane = threadIdx.x & 31;
    const long long seg = s.seg[0];
    const long long r0 = g * seg;
    const long long len = min(seg, s.rows - r0);
    const int nact = shared_row_lanes(s, r0);
    long long start = bounds[2 * g], end = bounds[2 * g + 1];
    int err = 0;
    if (start < 0 || end > n_words || end - start < 2ll * nact) { err = 4; end = start = 0; }
    const unsigned lt = lanemask_lt();

    unsigned x = kRansL;
    if (!err && lane < nact)
        x = (unsigned)__ldg(words + start + 2 * lane) | ((unsigned)__ldg(words + start + 2 * lane + 1) << 16);
    if (__any_sync(0xffffffffu, lane < nact && x < kRansL)) err |= 4;
    long long pos = start + 2 * nact, wbase;
    unsigned w0, w1, w2, w3;
    shared_load_window(words, pos, end, lane, wbase, w0, w1, w2, w3);

    long long c = g * ((seg - 1) / K);   // the next checkpoint's entry
    long long next = K;                  // and its row in the segment
    for (long long t = 0; t < len && !err; ++t) {
        if (t == next) {
            if (lane == 0) cp_offsets[c] = (unsigned)(pos - start);
            cp_states[32 * c + lane] = x;
            ++c;
            next += K;
        }
        int sym;
        if (!shared_decode_row(x, pos, wbase, end, w0, w1, w2, w3, s, r0 + t, sh_tab, sh_idx, words, lane, lt, sym)) {
            err |= 1;
            break;
        }
    }
    if (!err && (__any_sync(0xffffffffu, lane < nact && x != kRansL) || pos != end)) err |= 2;
    if (err && lane == 0) atomicOr(status, err);
}

// One warp per work item: check every field, restore the checkpoint (or read the segment's initial states), decode
// rows up to last_row and write each symbol t = 32 r + lane whose embedding row t / D is in the item's slice of rows to
// out[u][t - D rows[u]].  Status: 8 for a bad item (nothing written), 4 for a bad group range or restored state, 1 for
// a group that ran out of words.  A z_hat store is deferred by one row, so its code-point load never stalls the state
// chain.
__global__ void __launch_bounds__(kSharedWarps * 32) vbq_rans_shared_decode_rows_kernel(
        const unsigned short *__restrict__ words, long long n_words, const long long *__restrict__ bounds,
        const unsigned *__restrict__ cum, SharedShape s, long long K, const unsigned *__restrict__ cp_offsets,
        const unsigned *__restrict__ cp_states, const vbq_rans_lookup_item *__restrict__ items, long long n_items,
        const long long *__restrict__ rows, long long n_req, long long D, const float *__restrict__ code_points,
        int *__restrict__ qidx, float *__restrict__ zhat, int *__restrict__ status) {
    extern __shared__ unsigned sh_tab[];   // [Q + 1] then [kRansBuckets + 1] uint16
    unsigned short *sh_idx = (unsigned short *)(sh_tab + s.Q + 1);
    if ((long long)blockIdx.x * kSharedWarps >= n_items) return;   // CTA-uniform
    stage_shared_table(sh_tab, sh_idx, cum, 0, s);

    const long long it = (long long)blockIdx.x * kSharedWarps + (threadIdx.x >> 5);
    if (it >= n_items) return;
    const int lane = threadIdx.x & 31;
    const long long G = s.gbase[1], seg = s.seg[0], V = s.n / D;
    const vbq_rans_lookup_item w = items[it];
    bool bad = w.segment < 0 || w.segment >= G;
    long long r0 = 0, len = 0, first = 0;
    if (!bad) {
        r0 = w.segment * seg;
        len = min(seg, s.rows - r0);
        bad = w.checkpoint < 0 || w.checkpoint > (len - 1) / K;
    }
    if (!bad) {
        first = r0 + w.checkpoint * K;
        bad = w.last_row < first || w.last_row >= min(first + K, r0 + len);
    }
    if (!bad) bad = w.lo < 0 || w.hi < w.lo || w.hi > n_req;
    for (long long i = w.lo + lane; !bad && i < w.hi; i += 32) {
        const long long r = rows[i];
        bad = r < 0 || r >= V || (i > w.lo && rows[i - 1] >= r);
    }
    if (__any_sync(0xffffffffu, bad)) {
        if (lane == 0) atomicOr(status, 8);
        return;
    }

    const int nact = shared_row_lanes(s, r0);
    long long start = bounds[2 * w.segment], end = bounds[2 * w.segment + 1];
    int err = 0;
    if (start < 0 || end > n_words || end - start < 2ll * nact) { err = 4; end = start = 0; }
    const unsigned lt = lanemask_lt();
    unsigned x = kRansL;
    long long pos, wbase;
    if (w.checkpoint == 0) {
        if (!err && lane < nact)
            x = (unsigned)__ldg(words + start + 2 * lane) | ((unsigned)__ldg(words + start + 2 * lane + 1) << 16);
        pos = start + 2 * nact;
    } else {
        const long long c = w.segment * ((seg - 1) / K) + w.checkpoint - 1;
        x = __ldg(cp_states + 32 * c + lane);
        pos = start + __ldg(cp_offsets + c);
    }
    if (__any_sync(0xffffffffu, lane < nact && x < kRansL)) err |= 4;
    unsigned w0, w1, w2, w3;
    shared_load_window(words, pos, end, lane, wbase, w0, w1, w2, w3);

    // this lane's symbol on the current row: embedding row e, offset o in it; u = the first slice entry with rows[u] >= e
    const unsigned long long t0 = 32ull * first + lane;
    long long e = (long long)(t0 / (unsigned long long)D), o = (long long)t0 - e * D;
    const long long de = 32 / D, dof = 32 % D;
    long long u = w.lo;
    long long ru = u < w.hi ? rows[u] : LLONG_MAX;
    long long pend = -1;                 // output element of the deferred store
    int qpend = 0;
    float zpend = 0.f;
    for (long long r = first; r <= w.last_row && !err; ++r) {
        const bool active = lane < shared_row_lanes(s, r);
        int sym;
        if (!shared_decode_row(x, pos, wbase, end, w0, w1, w2, w3, s, r, sh_tab, sh_idx, words, lane, lt, sym)) {
            err |= 1;
            break;
        }
        if (pend >= 0) {
            if (qidx) qidx[pend] = qpend;
            if (zhat) zhat[pend] = zpend;
        }
        pend = -1;
        if (active) {
            while (ru < e) ru = ++u < w.hi ? rows[u] : LLONG_MAX;
            if (ru == e) {
                pend = u * D + o;
                qpend = sym;
                if (zhat) zpend = __ldg(code_points + sym);
            }
        }
        e += de;
        o += dof;
        if (o >= D) { o -= D; ++e; }
    }
    if (!err && pend >= 0) {
        if (qidx) qidx[pend] = qpend;
        if (zhat) zhat[pend] = zpend;
    }
    if (err && lane == 0) atomicOr(status, err);
}

// ---- query scores against one shared-table plane (vbq_rans_shared_row_scores) --------------------------------------
//
// Warp w owns checkpoint intervals [w ipw, (w + 1) ipw), numbered segment C1 + j (C1 = (seg - 1) / K + 1 slots per
// segment), and scores every embedding row of [row_begin, row_end) whose first coder row lies in them, decoding past its
// last interval (and into later segments) until that row's last symbol.  Each decoded coder row is staged in the warp's
// 32-float buffer; lane l serves queries l and l + 32 and walks the 32 symbols in d order, so the sums follow the
// numerics contract of include/vbq_b200.h exactly.  The four accumulators of a (query, row) pair need no data movement:
// at position i of a coder row, register i & 3 holds the class of the current d (d advances with i, and 32 is a multiple
// of 4), and a row end resets all four.

constexpr int kScoreWarps = 16;
constexpr int kScoreMaxQueries = 64;                  // two per lane
constexpr long long kScoreTargetWarps = 16384;        // ipw is the fewest intervals per warp that stays below this
constexpr long long kScoreSmemBudget = 112 * 1024;    // per CTA (100-128 registers already allow one CTA per SM)

__host__ __device__ long long score_stride(long long D) { return D | 1; }   // odd: the 32 lanes' rows start in 32 different banks

struct ScoreSmem {
    long long tab, idx, cp, z, q, total;              // byte offsets of the parts; q takes B queries
};

__host__ __device__ ScoreSmem score_smem(int Q, long long D, long long B) {
    ScoreSmem m;
    m.tab = 0;
    m.idx = m.tab + 4ll * (Q + 1);
    m.cp = m.idx + ((2ll * (kRansBuckets + 1) + 15) & ~15ll);
    m.z = (m.cp + 4ll * Q + 15) & ~15ll;
    m.q = m.z + 4ll * 32 * kScoreWarps;
    m.total = m.q + 4 * B * score_stride(D);
    return m;
}

// dot = (a0 + a1) + (a2 + a3) where accumulator class c sits in a[(sh + c) & 3]; selects, not an indexed array, so the
// four stay in registers.
__device__ __forceinline__ float score_sum4(const float (&a)[4], int sh) {
    const float a0 = sh == 0 ? a[0] : sh == 1 ? a[1] : sh == 2 ? a[2] : a[3];
    const float a1 = sh == 0 ? a[1] : sh == 1 ? a[2] : sh == 2 ? a[3] : a[0];
    const float a2 = sh == 0 ? a[2] : sh == 1 ? a[3] : sh == 2 ? a[0] : a[1];
    const float a3 = sh == 0 ? a[3] : sh == 1 ? a[0] : sh == 2 ? a[1] : a[2];
    return __fadd_rn(__fadd_rn(a0, a1), __fadd_rn(a2, a3));
}

template <int QPL, bool COS>
__global__ void __launch_bounds__(kScoreWarps * 32, 1) vbq_rans_shared_row_scores_kernel(
        const unsigned short *__restrict__ words, long long n_words, const long long *__restrict__ bounds,
        const unsigned *__restrict__ cum, SharedShape s, long long K, const unsigned *__restrict__ cp_offsets,
        const unsigned *__restrict__ cp_states, const float *__restrict__ code_points,
        const float *__restrict__ queries, int B, long long D, long long row_begin, long long row_end,
        long long ipw, long long w_first, float *__restrict__ scores, int *__restrict__ status) {
    extern __shared__ __align__(16) unsigned char sh_raw[];
    const ScoreSmem m = score_smem(s.Q, D, B);
    unsigned *sh_tab = (unsigned *)(sh_raw + m.tab);
    unsigned short *sh_idx = (unsigned short *)(sh_raw + m.idx);
    float *sh_cp = (float *)(sh_raw + m.cp);
    float *sh_q = (float *)(sh_raw + m.q);
    const long long qs = score_stride(D);
    for (int i = threadIdx.x; i < s.Q; i += blockDim.x) sh_cp[i] = __ldg(code_points + i);
    for (long long i = threadIdx.x; i < (long long)B * D; i += blockDim.x) {
        const long long b = i / D;
        sh_q[b * qs + (i - b * D)] = __ldg(queries + i);
    }
    stage_shared_table(sh_tab, sh_idx, cum, 0, s);      // its barriers also publish sh_cp and sh_q

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float *sh_z = (float *)(sh_raw + m.z) + 32 * warp;
    const long long S = s.seg[0], G = s.gbase[1], C1 = (S - 1) / K + 1, T = G * C1;
    const long long I0 = (w_first + (long long)blockIdx.x * kScoreWarps + warp) * ipw;
    if (I0 >= T) return;
    const long long I1 = min(I0 + ipw, T);
    const long long ra = min((I0 / C1) * S + (I0 % C1) * K, s.rows);
    const long long rb = min((I1 / C1) * S + (I1 % C1) * K, s.rows);
    const long long e_lo = max((32 * ra + D - 1) / D, row_begin), e_hi = min((32 * rb + D - 1) / D, row_end);
    if (ra >= rb || e_lo >= e_hi) return;               // warp-uniform

    // D < kScoreSmemBudget / 4 here (vbq_rans_shared_score_max_queries), so d and the tile offsets fit 32 bits
    const int Di = (int)D;
    int qb[QPL];                                         // the lane's query rows in sh_q (the last one for lanes past B)
    float qn[QPL];                                       // sqrtf(q . q) for the cosine
#pragma unroll
    for (int k = 0; k < QPL; ++k) {
        qb[k] = min(lane + 32 * k, B - 1) * (int)qs;
        float a[4] = {0.f, 0.f, 0.f, 0.f};
        if (COS) {
            for (int d0 = 0; d0 < Di; d0 += 4) {
#pragma unroll
                for (int u = 0; u < 4; ++u)
                    if (d0 + u < Di) a[u] = __fmaf_rn(sh_q[qb[k] + d0 + u], sh_q[qb[k] + d0 + u], a[u]);
            }
        }
        qn[k] = __fsqrt_rn(score_sum4(a, 0));
    }

    // restore the checkpoint of the interval that holds the first owned row's first coder row
    const long long r_first = e_lo * D / 32, r_stop = (e_hi * D - 1) / 32;
    long long g = r_first / S;
    const long long j = (r_first - g * S) / K;
    const long long r_start = g * S + j * K;
    const unsigned lt = lanemask_lt();
    int err = 0;
    unsigned x = kRansL;
    long long start = bounds[2 * g], end = bounds[2 * g + 1], pos, wbase;
    int nact = shared_row_lanes(s, g * S);
    if (start < 0 || end > n_words || end - start < 2ll * nact) { err = 4; end = start = 0; }
    if (j == 0) {
        if (!err && lane < nact)
            x = (unsigned)__ldg(words + start + 2 * lane) | ((unsigned)__ldg(words + start + 2 * lane + 1) << 16);
        pos = start + 2 * nact;
    } else {
        const long long c = g * ((S - 1) / K) + j - 1;
        x = __ldg(cp_states + 32 * c + lane);
        pos = start + __ldg(cp_offsets + c);
    }
    if (__any_sync(0xffffffffu, lane < nact && x < kRansL)) err |= 4;
    unsigned w0, w1, w2, w3;
    shared_load_window(words, pos, end, lane, wbase, w0, w1, w2, w3);

    const long long span = row_end - row_begin;
    long long e = 32 * r_start / D;                      // embedding row of the coder row's first symbol
    int qoff = (int)(32 * r_start - e * D);              // its d; symbol i of the row has d = qoff + i until a row end
    int qp[QPL];                                         // sh_q[qp[k] + i] = the lane's q_d of symbol i of the coder row
#pragma unroll
    for (int k = 0; k < QPL; ++k) qp[k] = qb[k] + qoff;
    float acc[QPL][4], zz[4];
#pragma unroll
    for (int k = 0; k < QPL; ++k) acc[k][0] = acc[k][1] = acc[k][2] = acc[k][3] = 0.f;
    zz[0] = zz[1] = zz[2] = zz[3] = 0.f;
    for (long long r = r_start; r <= r_stop && !err; ++r) {
        if (r != r_start && r == g * S + S) {            // the next segment: start its group from its initial states
            ++g;
            nact = shared_row_lanes(s, r);
            start = bounds[2 * g];
            end = bounds[2 * g + 1];
            if (start < 0 || end > n_words || end - start < 2ll * nact) { err = 4; break; }
            x = kRansL;
            if (lane < nact)
                x = (unsigned)__ldg(words + start + 2 * lane) | ((unsigned)__ldg(words + start + 2 * lane + 1) << 16);
            if (__any_sync(0xffffffffu, lane < nact && x < kRansL)) { err |= 4; break; }
            pos = start + 2 * nact;
            shared_load_window(words, pos, end, lane, wbase, w0, w1, w2, w3);
        }
        int sym;
        if (!shared_decode_row(x, pos, wbase, end, w0, w1, w2, w3, s, r, sh_tab, sh_idx, words, lane, lt, sym)) {
            err |= 1;
            break;
        }
        __syncwarp();                                    // the previous row's reads of sh_z are done
        sh_z[lane] = lane < shared_row_lanes(s, r) ? sh_cp[sym] : 0.f;
        __syncwarp();
        unsigned ends = 0;                               // positions whose symbol is the last of its embedding row
        for (int p = Di - 1 - qoff; p < 32; p += Di) ends |= 1u << p;
#pragma unroll
        for (int i4 = 0; i4 < 32; i4 += 4) {
            const float4 z4 = *(const float4 *)(sh_z + i4);
            const float zv[4] = {z4.x, z4.y, z4.z, z4.w};
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = i4 + u;
                const float z = zv[u];
#pragma unroll
                for (int k = 0; k < QPL; ++k) acc[k][u] = __fmaf_rn(z, sh_q[qp[k] + i], acc[k][u]);
                if (COS) zz[u] = __fmaf_rn(z, z, zz[u]);
                if (ends & (1u << i)) {                  // warp-uniform
                    const int sh = (i + 1 - Di) & 3;   // accumulator class c lives in register (sh + c) & 3
                    if (e >= e_lo && e < e_hi) {
                        const float zn = COS ? __fsqrt_rn(score_sum4(zz, sh)) : 0.f;
#pragma unroll
                        for (int k = 0; k < QPL; ++k) {
                            float v = score_sum4(acc[k], sh);
                            if (COS) {
                                const float den = __fmul_rn(zn, qn[k]);
                                v = den > 0.f ? __fdiv_rn(v, den) : 0.f;
                            }
                            if (lane + 32 * k < B) scores[(long long)(lane + 32 * k) * span + (e - row_begin)] = v;
                        }
                    }
#pragma unroll
                    for (int k = 0; k < QPL; ++k) {
                        acc[k][0] = acc[k][1] = acc[k][2] = acc[k][3] = 0.f;
                        qp[k] = qb[k] - (i + 1);
                    }
                    zz[0] = zz[1] = zz[2] = zz[3] = 0.f;
                    ++e;
                    qoff = -(i + 1);
                }
            }
        }
        qoff += 32;
#pragma unroll
        for (int k = 0; k < QPL; ++k) qp[k] += 32;
    }
    if (err && lane == 0) atomicOr(status, err);
}

}  // namespace

extern "C" long long vbq_rans_workspace_bytes(int n_planes, int items, long long item_rows, int C, long long seg_rows) {
    RansShape s;
    if (rans_shape("vbq_rans_workspace_bytes", n_planes, items, item_rows, C, seg_rows, 0, 16, &s) != VBQ_OK) return -1;
    return 2 * align256(8ll * n_planes * s.G) + align256(2ll * n_planes * rans_plane_scratch_words(s));
}

extern "C" long long vbq_rans_payload_bound(int n_planes, int items, long long item_rows, int C, long long seg_rows) {
    RansShape s;
    if (rans_shape("vbq_rans_payload_bound", n_planes, items, item_rows, C, seg_rows, 0, 16, &s) != VBQ_OK) return -1;
    return 2ll * n_planes * (2 * s.G + rans_plane_scratch_words(s));
}

extern "C" int vbq_rans_encode(const int *d_qidx, int n_planes, int items, long long item_rows, int C,
                               long long seg_rows, int N, int prob_bits, const unsigned short *d_cum,
                               unsigned short *d_payload, long long payload_bytes, long long *d_payload_size,
                               int *d_status, void *d_workspace, long long workspace_bytes, void *stream) {
    RansShape s;
    RETURN_IF(rans_shape("vbq_rans_encode", n_planes, items, item_rows, C, seg_rows, N, prob_bits, &s));
    if (!d_cum || !d_payload || !d_payload_size || !d_status || (s.G > 0 && (!d_qidx || !d_workspace)))
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_rans_encode: null pointer");
    if (payload_bytes < vbq_rans_payload_bound(n_planes, items, item_rows, C, seg_rows))
        return vbq_fail(VBQ_ERR_WORKSPACE, "vbq_rans_encode: payload capacity %lld < vbq_rans_payload_bound %lld",
                        payload_bytes, vbq_rans_payload_bound(n_planes, items, item_rows, C, seg_rows));
    const long long need = vbq_rans_workspace_bytes(n_planes, items, item_rows, C, seg_rows);
    if (s.G > 0 && workspace_bytes < need)
        return vbq_fail(VBQ_ERR_WORKSPACE, "vbq_rans_encode: workspace %lld < %lld bytes", workspace_bytes, need);
    if (((uintptr_t)d_payload & 1) || ((uintptr_t)d_cum & 1) || ((uintptr_t)d_workspace & 7) || ((uintptr_t)d_qidx & 3))
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_rans_encode: misaligned pointer");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int), st));
    if (s.G == 0) {
        CUDA_TRY(cudaMemsetAsync(d_payload_size, 0, sizeof(long long), st));
        return VBQ_OK;
    }
    int dev = 0, sms = 0;
    RETURN_IF(vbq_current_device(&dev, &sms));
    char *ws = (char *)d_workspace;
    long long *sizes = (long long *)ws;
    long long *dst = (long long *)(ws + align256(8ll * n_planes * s.G));
    unsigned short *scratch = (unsigned short *)(ws + 2 * align256(8ll * n_planes * s.G));
    const long long units = (long long)s.items * s.n_segs;
    const dim3 grid((unsigned)((units + kRansWarps - 1) / kRansWarps), s.CG, n_planes);
    const size_t smem = (size_t)32 * s.Q * sizeof(unsigned short);
    VBQ_ENSURE_MAX_SMEM(vbq_rans_encode_kernel, dev);
    vbq_rans_encode_kernel<<<grid, kRansWarps * 32, smem, st>>>(d_qidx, d_cum, s, scratch, sizes, d_status);
    CUDA_TRY(cudaGetLastError());
    vbq_rans_scan_kernel<<<1, 1024, 0, st>>>(sizes, dst, n_planes, s.G, d_payload, d_payload_size);
    CUDA_TRY(cudaGetLastError());
    vbq_rans_compact_kernel<<<(unsigned)(n_planes * s.G), 256, 0, st>>>(scratch, sizes, dst, s, d_payload);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

extern "C" int vbq_rans_decode(const unsigned short *d_payload, long long payload_words,
                               const long long *d_group_bounds, int n_planes, int items, long long item_rows, int C,
                               long long seg_rows, int N, int prob_bits, const unsigned short *d_cum,
                               const float *d_code_points, int *d_qidx, float *d_zhat, int *d_status, void *stream) {
    RansShape s;
    RETURN_IF(rans_shape("vbq_rans_decode", n_planes, items, item_rows, C, seg_rows, N, prob_bits, &s));
    if (payload_words < 0) return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_rans_decode: payload_words=%lld", payload_words);
    if (!d_cum || !d_status || (d_zhat && !d_code_points) || (s.G > 0 && (!d_payload || !d_group_bounds)))
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_rans_decode: null pointer");
    if (((uintptr_t)d_payload & 1) || ((uintptr_t)d_cum & 1) || ((uintptr_t)d_group_bounds & 7) ||
        ((uintptr_t)d_qidx & 3) || ((uintptr_t)d_zhat & 3) || ((uintptr_t)d_code_points & 3))
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_rans_decode: misaligned pointer");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int), st));
    if (s.G == 0) return VBQ_OK;
    int dev = 0, sms = 0;
    RETURN_IF(vbq_current_device(&dev, &sms));
    const long long units = (long long)s.items * s.n_segs;
    const dim3 grid((unsigned)((units + kRansWarps - 1) / kRansWarps), s.CG, n_planes);
    const size_t smem = (size_t)32 * (s.Q + kRansBuckets + 1) * sizeof(unsigned short);
    VBQ_ENSURE_MAX_SMEM(vbq_rans_decode_kernel, dev);
    vbq_rans_decode_kernel<<<grid, kRansWarps * 32, smem, st>>>(d_payload, payload_words, d_group_bounds, d_cum, s,
                                                                d_code_points, d_qidx, d_zhat, d_status);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

extern "C" int vbq_rans_decode_batch(const unsigned short *d_payload, long long payload_words,
                                     const unsigned short *d_cum, const int *d_prob_bits, int n_tables, int C, int N,
                                     const vbq_rans_batch_unit *d_units, long long n_units,
                                     const vbq_rans_batch_cta *d_ctas, long long n_ctas, int n_blobs,
                                     const float *d_code_points, long long n_out, int *d_qidx, float *d_zhat,
                                     int *d_status, void *stream) {
    if (N < 0 || N > 10) return vbq_fail(VBQ_ERR_BAD_DEPTH, "vbq_rans_decode_batch: N=%d (the coder holds N <= 10)", N);
    if (payload_words < 0 || n_tables < 0 || C < 1 || C > 32 * 65535 || n_units < 0 || n_ctas < 0 ||
        n_ctas > 2147483647ll || n_blobs < 0 || n_out < 0 || (n_ctas > 0 && (n_units < 1 || n_blobs < 1 || n_tables < 1)))
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_rans_decode_batch: payload_words=%lld n_tables=%d C=%d n_units=%lld "
                        "n_ctas=%lld n_blobs=%d n_out=%lld", payload_words, n_tables, C, n_units, n_ctas, n_blobs, n_out);
    const bool work = n_ctas > 0;
    if ((n_blobs > 0 && !d_status) || (d_zhat && !d_code_points) ||
        (work && (!d_payload || !d_cum || !d_prob_bits || !d_units || !d_ctas)))
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_rans_decode_batch: null pointer");
    if (((uintptr_t)d_payload & 1) || ((uintptr_t)d_cum & 1) || ((uintptr_t)d_prob_bits & 3) ||
        ((uintptr_t)d_units & 7) || ((uintptr_t)d_ctas & 7) || ((uintptr_t)d_code_points & 3) ||
        ((uintptr_t)d_qidx & 3) || ((uintptr_t)d_zhat & 3) || ((uintptr_t)d_status & 3))
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_rans_decode_batch: misaligned pointer");
    cudaStream_t st = (cudaStream_t)stream;
    if (n_blobs > 0) CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int) * (size_t)n_blobs, st));
    if (!work) return VBQ_OK;
    int dev = 0, sms = 0;
    RETURN_IF(vbq_current_device(&dev, &sms));
    const int Q = (1 << (N + 1)) - 1;
    const size_t smem = (size_t)32 * (Q + kRansBuckets + 1) * sizeof(unsigned short);
    VBQ_ENSURE_MAX_SMEM(vbq_rans_decode_batch_kernel, dev);
    vbq_rans_decode_batch_kernel<<<(unsigned)n_ctas, kRansWarps * 32, smem, st>>>(
        d_payload, payload_words, d_cum, d_prob_bits, n_tables, C, Q, d_units, n_units, d_ctas, n_blobs,
        d_code_points, n_out, d_qidx, d_zhat, d_status);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

extern "C" long long vbq_rans_encode_batch_workspace_bytes(long long n_groups, long long scratch_words) {
    if (n_groups < 0 || n_groups > 2147483647ll || scratch_words < 0 || scratch_words > (1ll << 60)) return -1;
    return 3 * align256(8 * n_groups) + align256(2 * scratch_words);
}

extern "C" int vbq_rans_encode_batch(const int *d_in, long long n_in, const unsigned short *d_cum,
                                     const int *d_prob_bits, int n_tables, int C, int N,
                                     const vbq_rans_encode_unit *d_units, long long n_units,
                                     const vbq_rans_batch_cta *d_ctas, long long n_ctas,
                                     const long long *d_blob_groups, int n_blobs, long long n_groups,
                                     unsigned short *d_payload, long long payload_words, long long *d_blob_starts,
                                     int *d_status, void *d_workspace, long long workspace_bytes, void *stream) {
    if (N < 0 || N > 10) return vbq_fail(VBQ_ERR_BAD_DEPTH, "vbq_rans_encode_batch: N=%d (the coder holds N <= 10)", N);
    if (n_in < 0 || n_tables < 0 || C < 1 || C > 32 * 65535 || n_units < 0 || n_ctas < 0 || n_ctas > 2147483647ll ||
        n_blobs < 0 || n_groups < 0 || n_groups > 2147483647ll || payload_words < 0 || workspace_bytes < 0 ||
        (n_groups > 0 && n_blobs < 1) || (n_ctas > 0 && (n_units < 1 || n_tables < 1 || n_groups < 1)))
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_rans_encode_batch: n_in=%lld n_tables=%d C=%d n_units=%lld n_ctas=%lld "
                        "n_blobs=%d n_groups=%lld payload_words=%lld workspace_bytes=%lld", n_in, n_tables, C, n_units,
                        n_ctas, n_blobs, n_groups, payload_words, workspace_bytes);
    const bool work = n_ctas > 0, groups = n_groups > 0;
    if (!d_blob_starts || (n_blobs > 0 && !d_status) || (groups && (!d_blob_groups || !d_payload || !d_workspace)) ||
        (work && (!d_in || !d_cum || !d_prob_bits || !d_units || !d_ctas)))
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_rans_encode_batch: null pointer");
    if (((uintptr_t)d_in & 3) || ((uintptr_t)d_cum & 1) || ((uintptr_t)d_prob_bits & 3) || ((uintptr_t)d_units & 7) ||
        ((uintptr_t)d_ctas & 7) || ((uintptr_t)d_blob_groups & 7) || ((uintptr_t)d_payload & 1) ||
        ((uintptr_t)d_blob_starts & 7) || ((uintptr_t)d_status & 3) || ((uintptr_t)d_workspace & 7))
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_rans_encode_batch: misaligned pointer");
    const long long index_bytes = 3 * align256(8 * n_groups);
    if (groups && workspace_bytes < index_bytes)
        return vbq_fail(VBQ_ERR_WORKSPACE, "vbq_rans_encode_batch: workspace %lld < %lld bytes for %lld groups",
                        workspace_bytes, index_bytes, n_groups);
    cudaStream_t st = (cudaStream_t)stream;
    if (n_blobs > 0) CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int) * (size_t)n_blobs, st));
    if (!groups) {
        CUDA_TRY(cudaMemsetAsync(d_blob_starts, 0, sizeof(long long) * ((size_t)n_blobs + 1), st));
        return VBQ_OK;
    }
    char *ws = (char *)d_workspace;
    long long *sizes = (long long *)ws;
    long long *ends = (long long *)(ws + align256(8 * n_groups));
    long long *dst = (long long *)(ws + 2 * align256(8 * n_groups));
    unsigned short *scratch = (unsigned short *)(ws + index_bytes);
    const long long scratch_words = (workspace_bytes - index_bytes) / 2;
    CUDA_TRY(cudaMemsetAsync(sizes, 0, 8 * (size_t)n_groups, st));
    if (work) {
        int dev = 0, sms = 0;
        RETURN_IF(vbq_current_device(&dev, &sms));
        const int Q = (1 << (N + 1)) - 1;
        const size_t smem = (size_t)32 * Q * sizeof(unsigned short);
        VBQ_ENSURE_MAX_SMEM(vbq_rans_encode_batch_kernel, dev);
        vbq_rans_encode_batch_kernel<<<(unsigned)n_ctas, kRansWarps * 32, smem, st>>>(
            d_in, n_in, d_cum, d_prob_bits, n_tables, C, Q, d_units, n_units, d_ctas, n_blobs, n_groups, scratch,
            scratch_words, sizes, ends, d_status);
        CUDA_TRY(cudaGetLastError());
    }
    vbq_rans_encode_batch_scan_kernel<<<1, 1024, 0, st>>>(sizes, dst, n_groups, d_blob_groups, n_blobs, d_payload,
                                                          payload_words, d_blob_starts, d_status);
    CUDA_TRY(cudaGetLastError());
    vbq_rans_encode_batch_compact_kernel<<<(unsigned)n_groups, 256, 0, st>>>(scratch, sizes, ends, dst, d_payload,
                                                                             payload_words);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

extern "C" long long vbq_rans_shared_workspace_bytes(int n_planes, long long n, const long long *seg_rows) {
    SharedShape s;
    if (shared_shape("vbq_rans_shared_workspace_bytes", n_planes, n, seg_rows, 0, 16, &s) != VBQ_OK) return -1;
    const long long G = s.gbase[n_planes];
    return 2 * align256(8 * G) + align256(2 * s.sbase[n_planes]);
}

extern "C" long long vbq_rans_shared_payload_bound(int n_planes, long long n, const long long *seg_rows) {
    SharedShape s;
    if (shared_shape("vbq_rans_shared_payload_bound", n_planes, n, seg_rows, 0, 16, &s) != VBQ_OK) return -1;
    long long words = 0;
    for (int p = 0; p < n_planes; ++p) {
        const long long G = s.gbase[p + 1] - s.gbase[p];
        const long long lanes = G ? 32 * (G - 1) + min(32ll, n - 32 * (G - 1) * s.seg[p]) : 0;
        words += 2 * G + n + 2 * lanes;
    }
    return 2 * words;
}

extern "C" int vbq_rans_shared_encode(const int *d_qidx, int n_planes, long long n, const long long *seg_rows, int N,
                                      int prob_bits, const unsigned *d_cum, unsigned short *d_payload,
                                      long long payload_bytes, long long *d_payload_size, int *d_status,
                                      void *d_workspace, long long workspace_bytes, void *stream) {
    SharedShape s;
    RETURN_IF(shared_shape("vbq_rans_shared_encode", n_planes, n, seg_rows, N, prob_bits, &s));
    const long long G = s.gbase[n_planes];
    if (!d_cum || !d_payload || !d_payload_size || !d_status || (G > 0 && (!d_qidx || !d_workspace)))
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_rans_shared_encode: null pointer");
    const long long bound = vbq_rans_shared_payload_bound(n_planes, n, seg_rows);
    if (payload_bytes < bound)
        return vbq_fail(VBQ_ERR_WORKSPACE, "vbq_rans_shared_encode: payload capacity %lld < "
                        "vbq_rans_shared_payload_bound %lld", payload_bytes, bound);
    const long long need = vbq_rans_shared_workspace_bytes(n_planes, n, seg_rows);
    if (G > 0 && workspace_bytes < need)
        return vbq_fail(VBQ_ERR_WORKSPACE, "vbq_rans_shared_encode: workspace %lld < %lld bytes", workspace_bytes, need);
    if (((uintptr_t)d_payload & 1) || ((uintptr_t)d_cum & 3) || ((uintptr_t)d_workspace & 7) ||
        ((uintptr_t)d_qidx & 3) || ((uintptr_t)d_payload_size & 7) || ((uintptr_t)d_status & 3))
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_rans_shared_encode: misaligned pointer");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int), st));
    if (G == 0) {
        CUDA_TRY(cudaMemsetAsync(d_payload_size, 0, sizeof(long long), st));
        return VBQ_OK;
    }
    char *ws = (char *)d_workspace;
    long long *sizes = (long long *)ws;
    long long *dst = (long long *)(ws + align256(8 * G));
    unsigned short *scratch = (unsigned short *)(ws + 2 * align256(8 * G));
    const dim3 grid((unsigned)((s.max_groups + kSharedWarps - 1) / kSharedWarps), n_planes);
    const size_t smem = (size_t)(s.Q + 1) * sizeof(unsigned);
    vbq_rans_shared_encode_kernel<<<grid, kSharedWarps * 32, smem, st>>>(d_qidx, d_cum, s, scratch, sizes, d_status);
    CUDA_TRY(cudaGetLastError());
    vbq_rans_shared_scan_kernel<<<1, 1024, 0, st>>>(sizes, dst, s, d_payload, d_payload_size);
    CUDA_TRY(cudaGetLastError());
    vbq_rans_shared_compact_kernel<<<(unsigned)G, 256, 0, st>>>(scratch, sizes, dst, s, d_payload);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

extern "C" int vbq_rans_shared_decode(const unsigned short *d_payload, long long payload_words,
                                      const long long *d_group_bounds, int n_planes, long long n,
                                      const long long *seg_rows, int N, int prob_bits, const unsigned *d_cum,
                                      const float *d_code_points, int *d_qidx, float *d_zhat, int *d_status,
                                      void *stream) {
    SharedShape s;
    RETURN_IF(shared_shape("vbq_rans_shared_decode", n_planes, n, seg_rows, N, prob_bits, &s));
    if (payload_words < 0)
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_rans_shared_decode: payload_words=%lld", payload_words);
    const long long G = s.gbase[n_planes];
    if (!d_cum || !d_status || (d_zhat && !d_code_points) || (G > 0 && (!d_payload || !d_group_bounds)))
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_rans_shared_decode: null pointer");
    if (((uintptr_t)d_payload & 1) || ((uintptr_t)d_cum & 3) || ((uintptr_t)d_group_bounds & 7) ||
        ((uintptr_t)d_qidx & 3) || ((uintptr_t)d_zhat & 3) || ((uintptr_t)d_code_points & 3) || ((uintptr_t)d_status & 3))
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_rans_shared_decode: misaligned pointer");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int), st));
    if (G == 0) return VBQ_OK;
    const dim3 grid((unsigned)((s.max_groups + kSharedWarps - 1) / kSharedWarps), n_planes);
    const size_t smem = (size_t)(s.Q + 1) * sizeof(unsigned) + (kRansBuckets + 1) * sizeof(unsigned short);
    vbq_rans_shared_decode_kernel<<<grid, kSharedWarps * 32, smem, st>>>(d_payload, payload_words, d_group_bounds, d_cum,
                                                                       s, d_code_points, d_qidx, d_zhat, d_status);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

namespace {

// shared_shape of one plane, plus K >= 1 clamped to the segment length (a longer interval holds no checkpoint).
int lookup_shape(const char *fn, long long n, long long seg_rows, int N, int prob_bits, long long K, SharedShape *s,
                 long long *k) {
    if (K < 1) return vbq_fail(VBQ_ERR_BAD_SHAPE, "%s: checkpoint_rows=%lld (>= 1)", fn, K);
    RETURN_IF(shared_shape(fn, 1, n, &seg_rows, N, prob_bits, s));
    *k = min(K, s->seg[0]);
    return VBQ_OK;
}

long long lookup_checkpoints(const SharedShape &s, long long k) {
    const long long G = s.gbase[1];
    if (G == 0) return 0;
    return (G - 1) * ((s.seg[0] - 1) / k) + (s.rows - (G - 1) * s.seg[0] - 1) / k;
}

}  // namespace

extern "C" long long vbq_rans_shared_checkpoint_count(long long n, long long seg_rows, long long checkpoint_rows) {
    SharedShape s;
    long long k;
    if (lookup_shape("vbq_rans_shared_checkpoint_count", n, seg_rows, 0, 16, checkpoint_rows, &s, &k) != VBQ_OK)
        return -1;
    return lookup_checkpoints(s, k);
}

extern "C" int vbq_rans_shared_checkpoints(const unsigned short *d_payload, long long payload_words,
                                           const long long *d_group_bounds, long long n, long long seg_rows, int N,
                                           int prob_bits, const unsigned *d_cum, long long checkpoint_rows,
                                           unsigned *d_offsets, unsigned *d_states, int *d_status, void *stream) {
    SharedShape s;
    long long k;
    RETURN_IF(lookup_shape("vbq_rans_shared_checkpoints", n, seg_rows, N, prob_bits, checkpoint_rows, &s, &k));
    if (payload_words < 0)
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_rans_shared_checkpoints: payload_words=%lld", payload_words);
    const long long G = s.gbase[1], M = lookup_checkpoints(s, k);
    if (!d_cum || !d_status || (G > 0 && (!d_payload || !d_group_bounds)) || (M > 0 && (!d_offsets || !d_states)))
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_rans_shared_checkpoints: null pointer");
    if (((uintptr_t)d_payload & 1) || ((uintptr_t)d_cum & 3) || ((uintptr_t)d_group_bounds & 7) ||
        ((uintptr_t)d_offsets & 3) || ((uintptr_t)d_states & 3) || ((uintptr_t)d_status & 3))
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_rans_shared_checkpoints: misaligned pointer");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int), st));
    if (G == 0) return VBQ_OK;
    const size_t smem = (size_t)(s.Q + 1) * sizeof(unsigned) + (kRansBuckets + 1) * sizeof(unsigned short);
    vbq_rans_shared_checkpoints_kernel<<<(unsigned)((G + kSharedWarps - 1) / kSharedWarps), kSharedWarps * 32, smem,
                                         st>>>(d_payload, payload_words, d_group_bounds, d_cum, s, k, d_offsets,
                                               d_states, d_status);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

extern "C" int vbq_rans_shared_decode_rows(const unsigned short *d_payload, long long payload_words,
                                           const long long *d_group_bounds, long long n, long long seg_rows, int N,
                                           int prob_bits, const unsigned *d_cum, long long checkpoint_rows,
                                           const unsigned *d_offsets, const unsigned *d_states,
                                           const vbq_rans_lookup_item *d_items, long long n_items,
                                           const long long *d_rows, long long n_req, long long row_size,
                                           const float *d_code_points, int *d_qidx, float *d_zhat, int *d_status,
                                           void *stream) {
    SharedShape s;
    long long k;
    RETURN_IF(lookup_shape("vbq_rans_shared_decode_rows", n, seg_rows, N, prob_bits, checkpoint_rows, &s, &k));
    if (payload_words < 0 || row_size < 1 || n % row_size != 0 || n_items < 0 ||
        n_items > 2147483647ll * kSharedWarps || n_req < 0 || n_req > n / row_size)
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_rans_shared_decode_rows: payload_words=%lld row_size=%lld n=%lld "
                        "n_items=%lld n_req=%lld", payload_words, row_size, n, n_items, n_req);
    const long long G = s.gbase[1], M = lookup_checkpoints(s, k);
    if (!d_cum || !d_status || (d_zhat && !d_code_points) ||
        (n_items > 0 && (!d_payload || !d_group_bounds || !d_items || (G > 0 && M > 0 && (!d_offsets || !d_states)))) ||
        (n_req > 0 && !d_rows))
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_rans_shared_decode_rows: null pointer");
    if (((uintptr_t)d_payload & 1) || ((uintptr_t)d_cum & 3) || ((uintptr_t)d_group_bounds & 7) ||
        ((uintptr_t)d_offsets & 3) || ((uintptr_t)d_states & 3) || ((uintptr_t)d_items & 7) ||
        ((uintptr_t)d_rows & 7) || ((uintptr_t)d_code_points & 3) || ((uintptr_t)d_qidx & 3) ||
        ((uintptr_t)d_zhat & 3) || ((uintptr_t)d_status & 3))
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_rans_shared_decode_rows: misaligned pointer");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int), st));
    if (n_items == 0) return VBQ_OK;
    const size_t smem = (size_t)(s.Q + 1) * sizeof(unsigned) + (kRansBuckets + 1) * sizeof(unsigned short);
    vbq_rans_shared_decode_rows_kernel<<<(unsigned)((n_items + kSharedWarps - 1) / kSharedWarps), kSharedWarps * 32,
                                         smem, st>>>(d_payload, payload_words, d_group_bounds, d_cum, s, k, d_offsets,
                                                     d_states, d_items, n_items, d_rows, n_req, row_size,
                                                     d_code_points, d_qidx, d_zhat, d_status);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

extern "C" int vbq_rans_shared_score_max_queries(long long row_size) {
    if (row_size < 1) return 0;
    const long long fixed = score_smem(2047, row_size, 0).total;      // the largest table: N = 10
    const long long per = 4 * score_stride(row_size);
    return (int)max(0ll, min((long long)kScoreMaxQueries, (kScoreSmemBudget - fixed) / per));
}

extern "C" int vbq_rans_shared_row_scores(const unsigned short *d_payload, long long payload_words,
                                          const long long *d_group_bounds, long long n, long long seg_rows, int N,
                                          int prob_bits, const unsigned *d_cum, long long checkpoint_rows,
                                          const unsigned *d_offsets, const unsigned *d_states, long long row_size,
                                          long long row_begin, long long row_end, const float *d_queries,
                                          int n_queries, int metric, const float *d_code_points, float *d_scores,
                                          int *d_status, void *stream) {
    SharedShape s;
    long long k;
    RETURN_IF(lookup_shape("vbq_rans_shared_row_scores", n, seg_rows, N, prob_bits, checkpoint_rows, &s, &k));
    const long long V = row_size >= 1 ? n / row_size : 0;
    if (payload_words < 0 || row_size < 1 || n % row_size != 0 || row_begin < 0 || row_end < row_begin ||
        row_end > V || n_queries < 0 || n_queries > vbq_rans_shared_score_max_queries(row_size) ||
        (metric != VBQ_SCORE_DOT && metric != VBQ_SCORE_COSINE))
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_rans_shared_row_scores: payload_words=%lld row_size=%lld n=%lld rows "
                        "[%lld, %lld) n_queries=%d (max %d) metric=%d", payload_words, row_size, n, row_begin, row_end,
                        n_queries, vbq_rans_shared_score_max_queries(row_size), metric);
    const long long G = s.gbase[1], M = lookup_checkpoints(s, k);
    const bool work = row_end > row_begin && n_queries > 0;
    if (!d_cum || !d_status ||
        (work && (!d_payload || !d_group_bounds || !d_queries || !d_code_points || !d_scores ||
                  (G > 0 && M > 0 && (!d_offsets || !d_states)))))
        return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_rans_shared_row_scores: null pointer");
    if (((uintptr_t)d_payload & 1) || ((uintptr_t)d_cum & 3) || ((uintptr_t)d_group_bounds & 7) ||
        ((uintptr_t)d_offsets & 3) || ((uintptr_t)d_states & 3) || ((uintptr_t)d_queries & 3) ||
        ((uintptr_t)d_code_points & 3) || ((uintptr_t)d_scores & 3) || ((uintptr_t)d_status & 3))
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_rans_shared_row_scores: misaligned pointer");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(d_status, 0, sizeof(int), st));
    if (!work) return VBQ_OK;
    int dev = 0, sms = 0;
    RETURN_IF(vbq_current_device(&dev, &sms));
    // the intervals that hold the first coder rows of row_begin and row_end - 1, and the fewest intervals per warp
    // that keep the launch at most kScoreTargetWarps warps
    const long long S = s.seg[0], C1 = (S - 1) / k + 1;
    auto interval = [&](long long r) { return (r / S) * C1 + (r % S) / k; };
    const long long Ia = interval(row_begin * row_size / 32), Ib = interval((row_end - 1) * row_size / 32);
    const long long ipw = max(1ll, (Ib - Ia + kScoreTargetWarps) / kScoreTargetWarps);
    const long long w_first = Ia / ipw, warps = Ib / ipw - w_first + 1;
    const size_t smem = (size_t)score_smem(s.Q, row_size, n_queries).total;
    const unsigned grid = (unsigned)((warps + kScoreWarps - 1) / kScoreWarps);
#define VBQ_SCORE_LAUNCH(QPL, COS)                                                                                    \
    do {                                                                                                              \
        VBQ_ENSURE_MAX_SMEM((vbq_rans_shared_row_scores_kernel<QPL, COS>), dev);                                      \
        vbq_rans_shared_row_scores_kernel<QPL, COS><<<grid, kScoreWarps * 32, smem, st>>>(                            \
            d_payload, payload_words, d_group_bounds, d_cum, s, k, d_offsets, d_states, d_code_points, d_queries,     \
            n_queries, row_size, row_begin, row_end, ipw, w_first, d_scores, d_status);                               \
    } while (0)
    const bool cosine = metric == VBQ_SCORE_COSINE;
    if (n_queries <= 32) {
        if (cosine) VBQ_SCORE_LAUNCH(1, true); else VBQ_SCORE_LAUNCH(1, false);
    } else {
        if (cosine) VBQ_SCORE_LAUNCH(2, true); else VBQ_SCORE_LAUNCH(2, false);
    }
#undef VBQ_SCORE_LAUNCH
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}
