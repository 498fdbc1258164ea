// image_metrics.cu — exact SSE and the per-level SSIM / contrast-structure means of the TF-models MultiScaleSSIM
// (vbq_image_metrics), for M reconstructions of each of N same-shaped uint8 images.
//
// Pyramid.  The reference's step between levels, ndimage.convolve(im, ones((2, 2)) / 4, mode='reflect')[::2, ::2], is
// the mean of each 2 x 2 block with the last row or column repeated when a size is odd.  Level k holds multiples of
// 4^-k below 256, at most 16 significant bits for k <= 4, so float32 holds every level exactly and the block sum is
// exact in any order.  The originals' levels are built once and shared by their M reconstructions.
//
// Moments.  The 2-D Gaussian window is the outer product of a normalised 1-D window g (s = min(11, h, w) taps,
// sigma = 1.5 s / 11, the half-offset of _FSpecialGauss for even s), so each level is one launch over (tile, pair)
// whose CTA stages the halo of a 32 x 32 output tile of both images in shared memory (rows x flattened w * C columns,
// taps C apart), runs the horizontal and then the vertical 1-D pass of the five moments x, y, x^2, y^2, xy in float64
// (x^2, y^2 and xy are exact there) and forms ssim and cs at every valid position.  Taps past s are 0 and the halo
// past the image is 0, so every level runs the same 11-tap loops and the extra terms add exact zeros.
//
// Sums.  Each CTA writes one (ssim, cs) partial pair, and at level 0 also the exact integer SSE of the image elements
// it owns (its tile, extended to the image edge on the last tile row and column: the staged halo covers that).  A
// second kernel adds each (pair, level)'s partials in a fixed order, so there are no float atomics and two runs give
// the same bits.
#include <climits>

#include "common.h"

namespace {

constexpr int kLevels = 5;
constexpr int kTaps = 11;
constexpr int kHalo = kTaps - 1;
constexpr int kTileRows = 32;                   // output rows per CTA
constexpr int kTileCols = 32;                   // output columns (flattened w * C) per CTA
constexpr int kRowsPerThread = 8;               // the vertical pass keeps 5 x 8 accumulators per thread
constexpr int kThreads = kTileCols * kTileRows / kRowsPerThread;
constexpr int kMaxChannels = 4;
constexpr int kInRows = kTileRows + kHalo;
constexpr int kReduceThreads = 256;
constexpr double kC1 = (0.01 * 255.0) * (0.01 * 255.0);
constexpr double kC2 = (0.03 * 255.0) * (0.03 * 255.0);

struct SsimLevel {
    double g[kTaps];              // the 1-D window, 0 past s
    int h, w, C;                  // the level's image
    int ho, woc;                  // valid positions: ho rows x woc = (w - s + 1) C flattened columns
    int tiles_x, tiles;           // tiles per pair (tiles_x along the flattened columns)
};

struct LevelShape {
    int h, w, s;
};

void level_shapes(int H, int W, LevelShape *L) {
    for (int k = 0; k < kLevels; ++k) {
        L[k].h = k ? (L[k - 1].h + 1) / 2 : H;
        L[k].w = k ? (L[k - 1].w + 1) / 2 : W;
        L[k].s = min(kTaps, min(L[k].h, L[k].w));
    }
}

long long level_tiles(const LevelShape &L, int C, int *tiles_x) {
    const long long ty = (L.h - L.s + 1 + kTileRows - 1) / kTileRows;
    const long long tx = ((long long)(L.w - L.s + 1) * C + kTileCols - 1) / kTileCols;
    if (tiles_x) *tiles_x = (int)tx;
    return ty * tx;
}

size_t stage_bytes(int C) { return (size_t)2 * kInRows * (kTileCols + kHalo * C) * sizeof(float); }

size_t ssim_smem_bytes(int C) {
    return ((stage_bytes(C) + 15) & ~(size_t)15) + (size_t)5 * kInRows * kTileCols * sizeof(double);
}

// Workspace: the pyramid levels 1..4 (originals, then reconstructions, float32), then per level the (ssim, cs) partials
// of every (pair, tile), then the level-0 SSE partials.
struct Layout {
    LevelShape L[kLevels];
    long long img_elems[kLevels];                 // elements of one image at each level
    long long pyr_off[kLevels];                   // byte offsets of levels 1..4 (entry 0 unused)
    long long tiles[kLevels];
    long long part_off[kLevels];                  // byte offsets of the (pairs, tiles) double2 partials
    long long sse_off;
    long long bytes;
};

long long align256(long long b) { return (b + 255) & ~255ll; }

bool make_layout(long long N, long long M, int H, int W, int C, Layout *lay) {
    if (N < 0 || M < 0 || H < 1 || W < 1 || C < 1 || C > kMaxChannels) return false;
    level_shapes(H, W, lay->L);
    const long long pairs = N * M;
    if ((M > 0 && N > INT_MAX / M) || (long long)H * W * C >= (1ll << 31)) return false;
    const long long images = N + pairs;
    if (images > (1ll << 60) / ((long long)H * W * C)) return false;
    long long b = 0;
    for (int k = 0; k < kLevels; ++k) {
        lay->img_elems[k] = (long long)lay->L[k].h * lay->L[k].w * C;
        lay->tiles[k] = level_tiles(lay->L[k], C, nullptr);
        if (pairs > 0 && lay->tiles[k] > INT_MAX / pairs) return false;
        if (k) {
            lay->pyr_off[k] = b;
            b = align256(b + images * lay->img_elems[k] * (long long)sizeof(float));
        }
    }
    for (int k = 0; k < kLevels; ++k) {
        lay->part_off[k] = b;
        b = align256(b + pairs * lay->tiles[k] * 2 * (long long)sizeof(double));
    }
    lay->sse_off = b;
    lay->bytes = align256(b + pairs * lay->tiles[0] * (long long)sizeof(unsigned long long));
    lay->pyr_off[0] = 0;
    return true;
}

template <typename T>
__global__ void __launch_bounds__(256) vbq_image_pyramid_kernel(const T *__restrict__ in, float *__restrict__ out,
                                                                long long n_img, int h, int w, int C) {
    const int h2 = (h + 1) / 2, w2 = (w + 1) / 2;
    const long long per = (long long)h2 * w2 * C, total = n_img * per;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
         e += (long long)gridDim.x * blockDim.x) {
        const long long img = e / per;
        long long r = e - img * per;
        const int c = (int)(r % C);
        r /= C;
        const int j = (int)(r % w2), i = (int)(r / w2);
        const int i1 = min(2 * i + 1, h - 1), j1 = min(2 * j + 1, w - 1);
        const T *src = in + img * ((long long)h * w * C);
        const float a = (float)src[((long long)(2 * i) * w + 2 * j) * C + c];
        const float b = (float)src[((long long)(2 * i) * w + j1) * C + c];
        const float d = (float)src[((long long)i1 * w + 2 * j) * C + c];
        const float f = (float)src[((long long)i1 * w + j1) * C + c];
        out[e] = 0.25f * ((a + b) + (d + f));     // exact (see the header)
    }
}

template <typename T>
__device__ __forceinline__ T block_sum(T v, T *red) {   // fixed-order sum over the CTA; the result on thread 0
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    const int warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int k = 1; k < n_warps; ++k) v += red[k];
    return v;
}

// One CTA = one 32 x 32 tile of valid positions of one (reconstruction, original) pair.  T is uint8 at level 0 (which
// also sums the SSE) and float above.
template <typename T, bool SSE>
__global__ void __launch_bounds__(kThreads) vbq_ssim_level_kernel(
        const T *__restrict__ x, const T *__restrict__ y, int n_img, const SsimLevel L,
        double2 *__restrict__ part, unsigned long long *__restrict__ sse_part) {
    extern __shared__ __align__(16) unsigned char smem[];
    __shared__ double s_red[kThreads / 32];
    __shared__ unsigned long long s_red_u[kThreads / 32];
    const int C = L.C, cols_in = kTileCols + kHalo * C;
    float *sx = (float *)smem, *sy = sx + kInRows * cols_in;
    double *hb = (double *)(smem + ((2 * kInRows * cols_in * sizeof(float) + 15) & ~(size_t)15));
    constexpr int plane = kInRows * kTileCols;

    const long long pr = blockIdx.x / L.tiles;
    const int tile = (int)(blockIdx.x - pr * L.tiles);
    const int ty = tile / L.tiles_x, tx = tile - ty * L.tiles_x;
    const int r0 = ty * kTileRows, c0 = tx * kTileCols, wc = L.w * C;
    const long long img = (long long)L.h * wc;
    const T *xi = x + (pr % n_img) * img, *yi = y + pr * img;

    // stage the halo; at level 0 also the SSE of the owned elements (outside the image both are 0)
    const int own_r = ty == L.tiles / L.tiles_x - 1 ? kInRows : kTileRows;
    const int own_c = tx == L.tiles_x - 1 ? cols_in : kTileCols;
    unsigned long long e = 0;
    for (int k = threadIdx.x; k < kInRows * cols_in; k += kThreads) {
        const int r = k / cols_in, c = k - r * cols_in, gr = r0 + r, gc = c0 + c;
        float a = 0.f, b = 0.f;
        if (gr < L.h && gc < wc) {
            a = (float)xi[(long long)gr * wc + gc];
            b = (float)yi[(long long)gr * wc + gc];
        }
        sx[k] = a;
        sy[k] = b;
        if (SSE && r < own_r && c < own_c) {
            const int d = (int)a - (int)b;
            e += (unsigned long long)(d * d);
        }
    }
    __syncthreads();

    // horizontal pass: the five moments of every staged row at the tile's 32 output columns
    for (int k = threadIdx.x; k < plane; k += kThreads) {
        const int r = k / kTileCols, p = k - r * kTileCols;
        const float *px = sx + r * cols_in + p, *py = sy + r * cols_in + p;
        double m0 = 0.0, m1 = 0.0, m2 = 0.0, m3 = 0.0, m4 = 0.0;
#pragma unroll
        for (int t = 0; t < kTaps; ++t) {
            const double a = px[t * C], b = py[t * C], g = L.g[t];
            m0 = __fma_rn(g, a, m0);
            m1 = __fma_rn(g, b, m1);
            m2 = __fma_rn(g, __dmul_rn(a, a), m2);
            m3 = __fma_rn(g, __dmul_rn(b, b), m3);
            m4 = __fma_rn(g, __dmul_rn(a, b), m4);
        }
        hb[k] = m0;
        hb[plane + k] = m1;
        hb[2 * plane + k] = m2;
        hb[3 * plane + k] = m3;
        hb[4 * plane + k] = m4;
    }
    __syncthreads();

    // vertical pass: thread (p, i0) owns output rows i0 .. i0 + 7 of column p; taps in increasing order per output
    const int p = threadIdx.x % kTileCols, i0 = (threadIdx.x / kTileCols) * kRowsPerThread;
    double acc[5][kRowsPerThread];
#pragma unroll
    for (int q = 0; q < 5; ++q)
#pragma unroll
        for (int i = 0; i < kRowsPerThread; ++i) acc[q][i] = 0.0;
#pragma unroll
    for (int r = 0; r < kRowsPerThread + kHalo; ++r) {
        double v[5];
#pragma unroll
        for (int q = 0; q < 5; ++q) v[q] = hb[q * plane + (i0 + r) * kTileCols + p];
#pragma unroll
        for (int i = 0; i < kRowsPerThread; ++i) {
            const int t = r - i;
            if (t >= 0 && t < kTaps) {
#pragma unroll
                for (int q = 0; q < 5; ++q) acc[q][i] = __fma_rn(L.g[t], v[q], acc[q][i]);
            }
        }
    }

    // ssim and cs with the reference's operations in its order (identical images give exactly 1 at every position)
    double ss = 0.0, cc = 0.0;
    const bool col_ok = c0 + p < L.woc;
#pragma unroll
    for (int i = 0; i < kRowsPerThread; ++i) {
        if (col_ok && r0 + i0 + i < L.ho) {
            const double mu1 = acc[0][i], mu2 = acc[1][i];
            const double mu11 = __dmul_rn(mu1, mu1), mu22 = __dmul_rn(mu2, mu2), mu12 = __dmul_rn(mu1, mu2);
            const double s11 = __dsub_rn(acc[2][i], mu11), s22 = __dsub_rn(acc[3][i], mu22);
            const double s12 = __dsub_rn(acc[4][i], mu12);
            const double v1 = __dadd_rn(__dmul_rn(2.0, s12), kC2), v2 = __dadd_rn(__dadd_rn(s11, s22), kC2);
            const double n1 = __dadd_rn(__dmul_rn(2.0, mu12), kC1), d1 = __dadd_rn(__dadd_rn(mu11, mu22), kC1);
            ss = __dadd_rn(ss, __ddiv_rn(__dmul_rn(n1, v1), __dmul_rn(d1, v2)));
            cc = __dadd_rn(cc, __ddiv_rn(v1, v2));
        }
    }
    ss = block_sum(ss, s_red);
    cc = block_sum(cc, s_red);
    if (SSE) e = block_sum(e, s_red_u);
    if (threadIdx.x == 0) {
        part[blockIdx.x] = make_double2(ss, cc);
        if (SSE) sse_part[blockIdx.x] = e;
    }
}

struct ReduceArgs {
    long long part_off[kLevels];      // in double2 entries from the level-0 partials
    long long tiles[kLevels];
    double count[kLevels];            // valid positions x channels
};

// Block (pair, level): the level's partials of the pair in a fixed order, divided by the position count.
__global__ void __launch_bounds__(kReduceThreads) vbq_ssim_reduce_kernel(
        const double2 *__restrict__ part, const unsigned long long *__restrict__ sse_part, const ReduceArgs A,
        long long *__restrict__ sse, double *__restrict__ ssim, double *__restrict__ cs) {
    __shared__ double s_red[kReduceThreads / 32];
    __shared__ unsigned long long s_red_u[kReduceThreads / 32];
    const long long pr = blockIdx.x / kLevels;
    const int k = (int)(blockIdx.x - pr * kLevels);
    const long long n = A.tiles[k];
    const double2 *src = part + A.part_off[k] + pr * n;
    double ss = 0.0, cc = 0.0;
    unsigned long long e = 0;
    for (long long t = threadIdx.x; t < n; t += kReduceThreads) {
        const double2 v = src[t];
        ss += v.x;
        cc += v.y;
        if (k == 0) e += sse_part[pr * n + t];
    }
    ss = block_sum(ss, s_red);
    cc = block_sum(cc, s_red);
    e = block_sum(e, s_red_u);
    if (threadIdx.x == 0) {
        ssim[pr * kLevels + k] = ss / A.count[k];
        cs[pr * kLevels + k] = cc / A.count[k];
        if (k == 0) sse[pr] = (long long)e;
    }
}

SsimLevel level_params(const LevelShape &S, int C) {
    SsimLevel L;
    const double sigma = S.s * 1.5 / 11.0;           // _FSpecialGauss(size, sigma) with sigma = size * 1.5 / 11
    const int radius = S.s / 2;
    const double offset = S.s % 2 == 0 ? 0.5 : 0.0;
    double sum = 0.0;
    for (int t = 0; t < kTaps; ++t) {
        const double u = t - radius + offset;
        L.g[t] = t < S.s ? exp(-(u * u) / (2.0 * sigma * sigma)) : 0.0;
        sum += L.g[t];
    }
    for (int t = 0; t < kTaps; ++t) L.g[t] /= sum;
    L.h = S.h;
    L.w = S.w;
    L.C = C;
    L.ho = S.h - S.s + 1;
    L.woc = (S.w - S.s + 1) * C;
    L.tiles = (int)level_tiles(S, C, &L.tiles_x);
    return L;
}

template <typename T>
int launch_pyramid(const T *in, float *out, long long n_img, int h, int w, int C, cudaStream_t st) {
    const long long total = n_img * ((h + 1) / 2) * (long long)((w + 1) / 2) * C;
    if (total == 0) return VBQ_OK;
    const long long blocks = min((total + 255) / 256, 148ll * 16);
    vbq_image_pyramid_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(in, out, n_img, h, w, C);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

template <typename T, bool SSE>
int launch_level(const T *x, const T *y, long long N, long long pairs, const SsimLevel &L, double2 *part,
                 unsigned long long *sse_part, cudaStream_t st) {
    const size_t smem = ssim_smem_bytes(L.C);
    int dev = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    VBQ_ENSURE_MAX_SMEM((vbq_ssim_level_kernel<T, SSE>), dev);
    vbq_ssim_level_kernel<T, SSE><<<(unsigned)(pairs * L.tiles), kThreads, smem, st>>>(x, y, (int)N, L, part,
                                                                                        sse_part);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}

}  // namespace

extern "C" long long vbq_image_metrics_workspace_bytes(long long N, long long M, int H, int W, int C) {
    Layout lay;
    return make_layout(N, M, H, W, C, &lay) ? lay.bytes : -1;
}

extern "C" int vbq_image_metrics(const unsigned char *d_x, const unsigned char *d_y, long long N, long long M, int H,
                                 int W, int C, void *d_workspace, long long workspace_bytes, long long *d_sse,
                                 double *d_ssim, double *d_cs, void *stream) {
    Layout lay;
    if (!make_layout(N, M, H, W, C, &lay))
        return vbq_fail(VBQ_ERR_BAD_SHAPE, "vbq_image_metrics: N=%lld M=%lld H=%d W=%d C=%d (1 <= C <= %d, H W C < 2^31)", N, M, H,
                        W, C, kMaxChannels);
    const long long pairs = N * M;
    if (pairs == 0) return VBQ_OK;
    if (!d_x || !d_y || !d_sse || !d_ssim || !d_cs) return vbq_fail(VBQ_ERR_NULL_POINTER, "vbq_image_metrics: null pointer");
    if (((uintptr_t)d_sse & 7) || ((uintptr_t)d_ssim & 7) || ((uintptr_t)d_cs & 7) || ((uintptr_t)d_workspace & 15))
        return vbq_fail(VBQ_ERR_MISALIGNED, "vbq_image_metrics: misaligned pointer");
    if (!d_workspace || workspace_bytes < lay.bytes)
        return vbq_fail(VBQ_ERR_WORKSPACE, "vbq_image_metrics: workspace of %lld bytes, %lld needed", workspace_bytes,
                        lay.bytes);
    cudaStream_t st = (cudaStream_t)stream;
    char *ws = (char *)d_workspace;
    double2 *part0 = (double2 *)(ws + lay.part_off[0]);
    unsigned long long *sse_part = (unsigned long long *)(ws + lay.sse_off);
    ReduceArgs A;
    for (int k = 0; k < kLevels; ++k) {
        const SsimLevel L = level_params(lay.L[k], C);
        double2 *part = (double2 *)(ws + lay.part_off[k]);
        A.part_off[k] = (lay.part_off[k] - lay.part_off[0]) / (long long)sizeof(double2);
        A.tiles[k] = lay.tiles[k];
        A.count[k] = (double)L.ho * L.woc;
        if (k == 0) {
            RETURN_IF((launch_level<unsigned char, true>(d_x, d_y, N, pairs, L, part, sse_part, st)));
        } else {
            const float *px = (const float *)(ws + lay.pyr_off[k]), *py = px + N * lay.img_elems[k];
            RETURN_IF((launch_level<float, false>(px, py, N, pairs, L, part, nullptr, st)));
        }
        if (k + 1 < kLevels) {                       // the next level of the originals, then of the reconstructions
            float *ox = (float *)(ws + lay.pyr_off[k + 1]), *oy = ox + N * lay.img_elems[k + 1];
            const LevelShape &S = lay.L[k];
            if (k == 0) {
                RETURN_IF(launch_pyramid(d_x, ox, N, S.h, S.w, C, st));
                RETURN_IF(launch_pyramid(d_y, oy, pairs, S.h, S.w, C, st));
            } else {
                const float *ix = (const float *)(ws + lay.pyr_off[k]);
                RETURN_IF(launch_pyramid(ix, ox, N + pairs, S.h, S.w, C, st));
            }
        }
    }
    vbq_ssim_reduce_kernel<<<(unsigned)(pairs * kLevels), kReduceThreads, 0, st>>>(part0, sse_part, A, d_sse, d_ssim,
                                                                                   d_cs);
    CUDA_TRY(cudaGetLastError());
    return VBQ_OK;
}
