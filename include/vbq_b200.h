/*
 * vbq_b200 — C ABI of the B200-native VBQ rate-distortion quantization path.
 *
 * The reference (mandt-lab/vbq) has no FFI layer: its boundary is the Python surface of
 * img-compression/quantizer.py, learned_prior.py, vae_models.py, utils.py and one notebook cell.  Each entry
 * point below names the reference interface it replaces (paths relative to the reference root).  All pointers
 * prefixed d_ are DEVICE pointers owned by the caller; the library never allocates, keeps no global state and
 * orders all work on the given stream (a cudaStream_t passed as void*, NULL = legacy default stream).  Every
 * function returns a VBQ_* status (0 = ok) and never throws; vbq_last_error() gives the thread's last message.
 *
 * Data layout
 *   latents        (rows, C) float32, channel-last, row-major  — quantizer.py:196-197 reshape(-1, C)
 *   code points    (C, Q) float32, Q = 2^(N+1)-1, HEAP order: entry h = 2^n-1+i is F_c^-1((i+1/2)2^-n)
 *                  — quantizer.py:30-36 `all_code_points`; the notebook's `codepoints` (ipynb:383-390) is one row
 *   packed table   ceil(C/16) groups x 2069 entries x 16 channels, the shared-memory image of a 16-channel group:
 *                  bit depths 0..10, each stored as [pad, 2^n points, pad] so bracket ends need no clamping;
 *                  followed by ceil(C/16) "walk trees" of 40992 floats (the same code points in heap order, scaled by
 *                  2^24, bit depths 1..7 twice: the shared-memory image of vbq_bisect_tma_kernel); made by
 *                  vbq_pack_code_points, vbq_packed_table_floats(C, N) floats in all
 *   prior params   (C, 43) float32: for layer k=0..3: matrix (d_{k+1} x d_k row-major), bias (d_{k+1}),
 *                  factor (d_{k+1}, k<3), dims (1,3,3,3,1), already softplus/tanh-transformed
 *                  — learned_prior.py:30-58 `_matrices`, `_biases`, `_factors`
 *   penalties      (n_lambda, pen_channels, N+1) float32 = fl(float32(lambda) * float32(len[c][n])),
 *                  pen_channels = 1 (raw lengths len = n, quantizer.py:166-169) or C (corrected lengths
 *                  n + R_lambda[c][n], quantizer.py:170-180); utils.py:393-396 forms exactly this product
 *   sorted index   q = (2i+1) 2^(N-n) - 1, the rank of code point (n,i) among the channel's Q ascending code
 *                  points — what quantizer.py:135,223 compute by searchsorted(code_points_by_channel, z_hat)
 */
#ifndef VBQ_B200_H
#define VBQ_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define VBQ_VERSION 100

enum {
    VBQ_OK = 0,
    VBQ_ERR_NULL_POINTER = 1,
    VBQ_ERR_BAD_SHAPE = 2,     /* rows < 0, C < 1, n_lambda < 1, pen_channels not in {1, C} */
    VBQ_ERR_BAD_DEPTH = 3,     /* N outside [0, VBQ_MAX_DEPTH] */
    VBQ_ERR_BAD_FLAGS = 4,
    VBQ_ERR_WORKSPACE = 5,     /* workspace missing or too small */
    VBQ_ERR_CUDA = 6,          /* a CUDA runtime call failed; see vbq_last_error() */
    VBQ_ERR_MISALIGNED = 7
};

#define VBQ_MAX_DEPTH 20
#define VBQ_PRIOR_PARAMS 43
#define VBQ_GROUP 16             /* channels interleaved per shared-memory group */
#define VBQ_SMEM_LEVELS 11       /* bit depths 0..10 of a group live in shared memory */
#define VBQ_TOTALS 4             /* per lambda: sum raw depth n, sum code length, sum entropy-model bits, sum (z_hat-mu)^2/(2 sigma^2) */

/* flags of vbq_quantize */
#define VBQ_FLAG_LOGVAR   1u     /* d_sigma holds log-variances; sigma = sqrt(exp(logvar)) (quantizer.py:193-198) */
#define VBQ_FLAG_NO_PRUNE 2u     /* visit every bit depth even when deeper levels provably cannot win */
#define VBQ_FLAG_RESERVE_SM 64u       /* launch one CTA fewer than there are SMs, so that a concurrent kernel on another
                                         stream (e.g. the NCCL all-reduce of the previous call's totals) finds a free SM */
#define VBQ_FLAG_WORKSPACE_ZEROED 256u /* the caller guarantees that the first 256 bytes per 64 lambdas of d_workspace (the
                                         ticket counters) are zero: true after a cudaMemset at allocation and after every
                                         completed call, which leaves them zero again.  Saves the per-call memset node
                                         (about 5 us of stream time on a B200). */
#define VBQ_FLAG_TABLE_STABLE 1024u     /* the caller vouches that d_packed was completely written before the PREVIOUS operation
                                         on `stream` was enqueued (e.g. it synchronized after vbq_pack_code_points): the search
                                         kernel then fetches its code points while the stream's previous kernel still drains
                                         (programmatic dependent launch) instead of after it */
#define VBQ_FLAG_NEIGHBOUR_EVERY_DEPTH 2048u /* arbitrary penalties (vbq_bisect_tma_kernel both-ends variant, vbq_both_sweep_kernel): score the second
                                          bracket end at every depth, not only where the penalties allow it to win (same
                                          results; diagnostics and tests) */
#define VBQ_FLAG_NO_TMA 512u           /* single lambda: stage the latents with per-warp cp.async (vbq_bisect_kernel) instead
                                         of the TMA pipeline (vbq_bisect_tma_kernel); same results, for comparison */
#define VBQ_FLAG_BRACKET_WALK 128u     /* single lambda: use the nearer-bracket-end walk (strict mode) even where the
                                         certified bisection kernel applies (same results; for comparison) */
#define VBQ_FLAG_REFERENCE_WALK 32u   /* score both bracket ends of every depth (the slower, literal formulation; same results) */
#define VBQ_FLAG_NO_SWEEP 16u         /* walk the tree once per lambda instead of once for all lambdas */
#define VBQ_FLAG_ACCUMULATE_TOTALS 8u /* add this call's sums to d_totals instead of overwriting them */
#define VBQ_FLAG_FAST     4u     /* score with d*d*(0.5/sigma^2) + pen on the nearer bracket end only (not bit-faithful
                                    to utils.py:318-320 rounding; differs only inside float32 rounding ties) */

int vbq_version(void);
const char *vbq_status_string(int status);
const char *vbq_last_error(void);

/* ---- prior models -------------------------------------------------------------------------------------- */

/* BMSHJ2018Prior.cdf (learned_prior.py:109-148): d_x, d_cdf (rows, C) float32 channel-last. */
int vbq_learned_cdf(const float *d_params, int C, const float *d_x, long long rows, float *d_cdf, void *stream);

/* BMSHJ2018Prior.inverse_cdf (learned_prior.py:173-218): d_xi (rows, C) float64 in (0,1) -> d_z (rows, C)
 * float32.  Solves logits_c(z) = logit(xi) in float64 by bracketed Newton and rounds to float32, so the
 * result is a pure function of (channel parameters, xi). */
int vbq_learned_inverse_cdf(const float *d_params, int C, const double *d_xi, long long rows, float *d_z,
                            void *stream);

/* StandardGaussianPrior / FactoredGaussianPrior.inverse_cdf (vae_models.py:23-25, :40-43) and the notebook's
 * norm.ppf(xi, scale=empirical_std) (ipynb:385): d_z = mean[c] + std[c] * ndtri(xi), float64.
 * d_mean / d_std may be NULL (0 / 1). */
int vbq_gaussian_inverse_cdf(const double *d_mean, const double *d_std, int C, const double *d_xi,
                             long long rows, double *d_z, void *stream);

/* ---- code-point tables (ChannelwisePriorCDFQuantizer.build_code_points, quantizer.py:25-63) ------------ */

int vbq_build_code_points_learned(const float *d_params, int C, int N, float *d_table, void *stream);
int vbq_build_code_points_gaussian(const double *d_mean, const double *d_std, int C, int N, float *d_table,
                                   void *stream);
long long vbq_packed_table_floats(int C, int N);
int vbq_pack_code_points(const float *d_table, int C, int N, float *d_packed, void *stream);

/* ---- the hot path -------------------------------------------------------------------------------------- */

long long vbq_quantize_workspace_bytes(int n_lambda);

/* Replaces ChannelwisePriorCDFQuantizer.get_all_N_bit_intervals + compress_batch_channel_latents
 * (quantizer.py:65-80, :156-188), utils.curry_normal_logpdf + utils.batch_quantize_indep_dims
 * (utils.py:307-327, :363-423) and the sorted-index / entropy-model gather of compress_latents
 * (quantizer.py:223-228) for n_lambda rate-distortion trade-offs at once.  For every coordinate it finds the
 * bracketing code points of mu at each bit depth and returns the first maximiser (candidate order left_0..left_N,
 * right_1..right_N) of  -0.5*((z-mu)/sigma)^2 - penalty[lambda][c][n]  in float32 arithmetic.
 *
 * Outputs (any may be NULL), each (n_lambda, rows, C):
 *   d_zhat      float32  chosen code point                       (Z_hat_dict[lamb])
 *   d_qidx      int32    its sorted quantile index               (I / qidx, quantizer.py:135,223)
 *   d_level     int32    its bit depth n                         (raw_num_bits in raw-length mode)
 *   d_bits      float32  d_length[lambda][c][n] (n if d_length is NULL)  (num_bits_dict[lamb])
 *   d_em_bits   float32  d_entropy_model[lambda][c][q]           (num_bits, quantizer.py:226-228)
 * d_totals (n_lambda, VBQ_TOTALS) float64 receives the per-lambda sums (deterministic reduction order).
 * d_length has the shape of d_penalty; d_entropy_model is (n_lambda, C, Q) float32.
 * While the call runs, an entropy-model output plane may temporarily hold integer heap indices (em_gather_kernel replaces
 * them before the call's work on the stream completes); code lengths above 512 bits and entropy-model entries above 512
 * bits per coordinate are outside the exact range of the integer sums of the multi-lambda kernels (lengths fall back to a
 * float32 sum, entropy-model sums saturate). */
int vbq_quantize(const float *d_mu, const float *d_sigma, long long rows, int C,
                 const float *d_table, const float *d_packed, int N,
                 const float *d_penalty, const float *d_length, int n_lambda, int pen_channels,
                 const float *d_entropy_model,
                 float *d_zhat, int *d_qidx, int *d_level, float *d_bits, float *d_em_bits,
                 double *d_totals, void *d_workspace, long long workspace_bytes,
                 unsigned flags, void *stream);

/* vbq_quantize with an additional HOST copy of the penalties (same shape and values as d_penalty; may be NULL).  The
 * reference forms lambda * code_length on the host (utils.py:393-396), so its caller always has them; when they do
 * not depend on the channel (raw code lengths, quantizer.py:166-169) and n_lambda == 1 the search kernel takes them
 * as launch constants instead of spending a register per bit depth on them.  Results are identical. */
int vbq_quantize_hp(const float *d_mu, const float *d_sigma, long long rows, int C,
                    const float *d_table, const float *d_packed, int N,
                    const float *d_penalty, const float *h_penalty, const float *d_length, int n_lambda,
                    int pen_channels, const float *d_entropy_model,
                    float *d_zhat, int *d_qidx, int *d_level, float *d_bits, float *d_em_bits,
                    double *d_totals, void *d_workspace, long long workspace_bytes,
                    unsigned flags, void *stream);

/* ---- the exchange step of the data-parallel path (SURVEY 8e; the sums are consumed by utils.py:546-553) ------------ */

/* One context per rank (one process per GPU).  It owns this rank's INBOX in device memory; the 64-byte handle of
 * vbq_peer_ctx_handle travels to the other ranks of the node by any means (e.g. torch.distributed.all_gather), and
 * vbq_peer_ctx_connect(handles = world x 64 bytes, in rank order) maps their inboxes (cudaIpc, NVLink peer access). */
typedef struct vbq_peer_ctx vbq_peer_ctx;
int vbq_peer_ctx_create(int rank, int world, int n_lambda_max, vbq_peer_ctx **out);
int vbq_peer_ctx_handle(vbq_peer_ctx *ctx, unsigned char *handle64);
int vbq_peer_ctx_connect(vbq_peer_ctx *ctx, const unsigned char *handles);
int vbq_peer_ctx_destroy(vbq_peer_ctx *ctx);

/* The sums of the call with sequence number `seq` (>= 1, chosen by the caller: the same on every rank for the same call,
 * increasing by one per call) are DELIVERED by writing them into every rank's inbox (peer stores over NVLink + a
 * system-scope release of the sequence number) and COLLECTED by waiting, on the device, for every rank's entry and adding
 * the entries in rank order (deterministic) into d_totals (n_lambda, VBQ_TOTALS).  At most 8 calls may be delivered but
 * not yet collected.  vbq_peer_push / vbq_peer_collect are one-CTA kernels.  vbq_quantize_peer is vbq_quantize_hp that
 * also delivers the COMPLETED totals of an earlier call (`d_push_totals`, sequence number push_seq; 0 / NULL = none) and
 * collects a still earlier one (collect_seq -> d_collected; 0 / NULL = none): with n_lambda == 1 an idle lane of the
 * search kernel does both while the search runs, so a sequence of calls exchanges its totals once per call without any
 * other stream operation and without a collective library. */
int vbq_peer_push(vbq_peer_ctx *ctx, unsigned long long seq, int n_lambda, const double *d_totals, void *stream);
int vbq_peer_collect(vbq_peer_ctx *ctx, unsigned long long seq, int n_lambda, double *d_totals, void *stream);
int vbq_quantize_peer(const float *d_mu, const float *d_sigma, long long rows, int C,
                      const float *d_table, const float *d_packed, int N,
                      const float *d_penalty, const float *h_penalty, const float *d_length, int n_lambda,
                      int pen_channels, const float *d_entropy_model,
                      float *d_zhat, int *d_qidx, int *d_level, float *d_bits, float *d_em_bits,
                      double *d_totals, void *d_workspace, long long workspace_bytes,
                      unsigned flags, void *stream, vbq_peer_ctx *peer, unsigned long long push_seq,
                      const double *d_push_totals, unsigned long long collect_seq, double *d_collected);

/* ---- the hot path for host-resident latents ---------------------------------------------------------------- */

/* output selection bits of vbq_host_ctx_create */
#define VBQ_OUT_ZHAT    1u
#define VBQ_OUT_QIDX    2u
#define VBQ_OUT_LEVEL   4u
#define VBQ_OUT_BITS    8u
#define VBQ_OUT_EM_BITS 16u
#define VBQ_OUT_TOTALS  32u

/* A context owns three device staging slots of `chunk_rows` rows (inputs plus the selected outputs for n_lambda
 * trade-offs), three streams and the totals workspace.  It is the only object of this library that allocates;
 * one context serves one calling thread at a time. */
typedef struct vbq_host_ctx vbq_host_ctx;
int vbq_host_ctx_create(int C, int N, int n_lambda, long long chunk_rows, unsigned outputs, vbq_host_ctx **out);
int vbq_host_ctx_destroy(vbq_host_ctx *ctx);

/* vbq_quantize for HOST arrays (pinned memory recommended): the reference's host-side call
 * compress_batch_channel_latents(batch_means, batch_stds, lambs) on NumPy inputs (quantizer.py:156-188).
 * h_mu / h_sigma are (rows, C); outputs are (n_lambda, rows, C) host arrays (NULL to skip; must have been
 * selected at context creation); h_totals is (n_lambda, VBQ_TOTALS).  Tables, penalties and entropy models are
 * device pointers as in vbq_quantize.  Rows are processed in chunks whose upload, kernel and download overlap on
 * three streams of the context; the call returns when all results are in host memory.  The d_* tables must be
 * complete when the call is made (it does not order itself after other streams). */
int vbq_quantize_host(vbq_host_ctx *ctx, const float *h_mu, const float *h_sigma, long long rows,
                      const float *d_table, const float *d_packed, const float *d_penalty, const float *d_length,
                      int pen_channels, const float *d_entropy_model,
                      float *h_zhat, int *h_qidx, int *h_level, float *h_bits, float *h_em_bits, double *h_totals,
                      unsigned flags);

/* ---- word embeddings: the notebook's float64 search (ipynb:429-443) ------------------------------------------- */

/* compress_coordinates for one shared prior: d_mu, d_sigma (n) float32, d_codepoints (Q) float64 heap order
 * (ipynb:383-390), d_lengths (N+1) float64 code length of each bit depth, N <= 12.  Minimises
 * (c-mu)^2 + (2 beta) sigma^2 len(c) with the notebook's float64 roundings, first minimum in heap order.
 * pen_f32 != 0: (2 beta) sigma^2 is formed in float32 first (NumPy 1.17, or a Python-float beta under NumPy 2).
 * Outputs (n), any may be NULL: the optimum cast to float32, its heap index, its bit depth. */
int vbq_compress_coordinates_f64(const float *d_mu, const float *d_sigma, long long n, const double *d_codepoints,
                                 int N, const double *d_lengths, double beta, int pen_f32, float *d_optima,
                                 int *d_heap_index, int *d_level, void *stream);

/* ---- after the search: symbols for an external entropy coder (SURVEY 8 f4) ------------------------------------- */

/* The reference counts its sorted quantile indices per channel (quantizer.py:135-146, np.bincount in a Python loop)
 * and reports ideal code lengths (ipynb:452-455); it has no wire format.  vbq_symbol_histogram adds, for every
 * channel c and symbol s < Q = 2^(N+1)-1, the number of rows with d_qidx[r][c] == s to d_counts (C, Q) uint64
 * (the caller zeroes it; N <= 10).  vbq_pack_indices writes n symbols as a bit stream of N+1 bits per symbol
 * (symbol k = bits [k(N+1), (k+1)(N+1)), least significant bit first, in little-endian 32-bit words;
 * vbq_packed_index_words(n, N) words); vbq_unpack_indices is its inverse. */
long long vbq_packed_index_words(long long n, int N);
int vbq_pack_indices(const int *d_qidx, long long n, int N, unsigned *d_words, void *stream);
int vbq_unpack_indices(const unsigned *d_words, long long n, int N, int *d_qidx, void *stream);
int vbq_symbol_histogram(const int *d_qidx, long long rows, int C, int N, unsigned long long *d_counts,
                         void *stream);

/* ---- entropy coding of the sorted quantile indices: interleaved rANS (DESIGN.md §10) ------------------------------ */

/* A PLANE is (items, item_rows, C) int32 symbols q in [0, Q), Q = 2^(N+1)-1, N <= 10, coded with one frequency table per
 * (plane, channel) whose entries are >= 1 and sum to 2^prob_bits (12 <= prob_bits <= 16, Q <= 2^prob_bits).  Tables are
 * passed as d_cum (n_planes, C, Q) uint16: cum[s] = f[0] + ... + f[s-1], with an implicit cum[Q] = 2^prob_bits.
 * A GROUP is (item, segment of seg_rows rows, 32-channel group g); lane j of group g codes channel 32g+j over the
 * segment's rows in increasing order.  The coder has a 32-bit state in [2^16, 2^32) and emits 16-bit words, at most one
 * per symbol and lane.  The DECODER defines the format: read the active lanes' initial states (two words each, low half
 * first); for each row and each active lane in increasing order: slot = x & (2^P-1), s the symbol with
 * cum[s] <= slot < cum[s]+f[s], x = f[s] (x >> P) + slot - cum[s], and if x < 2^16 then x = (x << 16) | the group's
 * next word.  After the last row every state is 2^16 and every word of the group has been read.
 * PAYLOAD (uint16 words): per plane, the group end offset table (one uint32 per group as two words, low half first, in
 * words from the start of the plane's group data; groups in (item, segment, channel group) order), then the groups
 * (states, then words).  The planes' payloads follow each other.
 *
 * vbq_rans_workspace_bytes / vbq_rans_payload_bound: the encoder's workspace and the worst-case payload in bytes for a
 * shape (every lane emitting a word per row); -1 for a bad shape.
 * vbq_rans_encode codes n_planes planes (d_qidx (n_planes, items, item_rows, C)) in one launch into d_payload (at least
 * vbq_rans_payload_bound bytes) and leaves the payload size in bytes in the device scalar *d_payload_size; no host
 * synchronisation.  *d_status (device int) becomes nonzero (1) if a symbol was outside [0, Q).
 * vbq_rans_decode reads groups of d_payload (payload_words words) at the word ranges d_group_bounds
 * (n_planes * groups, 2) int64 [start, end), which the caller takes from the offset tables, and writes any of d_qidx
 * (int32) and d_zhat (float32 = d_code_points[c][q], the caller's (C, Q) ascending code points) of shape
 * (n_planes, items, item_rows, C).  A group never reads outside its range; *d_status (device int) receives 1 if a
 * group ran out of words, 2 if a final state differs from 2^16 or words are left over, 4 if a range or initial state
 * is invalid (0 = every group decoded and passed the integrity check).
 * Status codes: VBQ_ERR_BAD_DEPTH for N > 10, VBQ_ERR_BAD_SHAPE for a bad shape or prob_bits. */
long long vbq_rans_workspace_bytes(int n_planes, int items, long long item_rows, int C, long long seg_rows);
long long vbq_rans_payload_bound(int n_planes, int items, long long item_rows, int C, long long seg_rows);
int vbq_rans_encode(const int *d_qidx, int n_planes, int items, long long item_rows, int C, long long seg_rows, int N,
                    int prob_bits, const unsigned short *d_cum, unsigned short *d_payload, long long payload_bytes,
                    long long *d_payload_size, int *d_status, void *d_workspace, long long workspace_bytes,
                    void *stream);
int vbq_rans_decode(const unsigned short *d_payload, long long payload_words, const long long *d_group_bounds,
                    int n_planes, int items, long long item_rows, int C, long long seg_rows, int N, int prob_bits,
                    const unsigned short *d_cum, const float *d_code_points, int *d_qidx, float *d_zhat, int *d_status,
                    void *stream);

/* ---- many VBQ2 streams in one launch: the work-list decoder (DESIGN.md §8h) ------------------------------------
 *
 * vbq_rans_decode_batch decodes any set of groups of the layout above, from any number of streams (blobs) that share C
 * and N but may differ in table, prob_bits, seg_rows, item_rows, n_planes and items.  Each group is a UNIT.  Inputs:
 *   d_payload    (payload_words,) uint16: the streams' payloads back to back;
 *   d_cum        (n_tables, C, Q) uint16 cum tables as for vbq_rans_decode, and d_prob_bits (n_tables,) int32 device
 *                array with each table's prob_bits;
 *   d_units      (n_units,) vbq_rans_batch_unit;
 *   d_ctas       (n_ctas,) vbq_rans_batch_cta: CTA i decodes units [first, first + count), 1 <= count <= 8, which must
 *                all have the descriptor's (table, cg): the CTA stages that table set once;
 *   d_status     (n_blobs,) int32, zeroed by the call: bits 1, 2 and 4 of vbq_rans_decode for the groups of each blob,
 *                and bit 8 for a bad unit.
 * A unit decodes rows r = 0 .. rows - 1 of lanes j < nact = min(32, C - 32 cg) from its word range [start, end) and
 * writes symbol (r, j) to element out + r C + j of d_qidx (int32) and/or d_zhat (float32 d_code_points[32 cg + j][q],
 * the (C, Q) ascending code points), both flat of n_out elements; per row, the decoder is that of vbq_rans_decode.
 * Units and descriptors come from the caller's memory, so the kernel checks each before it acts: a range inside the
 * payload that holds at least the 2 nact state words, table and cg in range and equal to the descriptor's, rows >= 1,
 * 0 <= out and out + (rows - 1) C + nact <= n_out, 0 <= blob < n_blobs, and the table's prob_bits valid.  A bad unit
 * sets bit 8 of its blob (of blob 0 if the blob id itself, or the descriptor, is bad) and writes nothing.  Units
 * whose output ranges overlap write in an undefined order.
 * Status codes: VBQ_ERR_BAD_DEPTH for N > 10, VBQ_ERR_BAD_SHAPE for a bad count or C. */
typedef struct {
    long long start, end;   /* word range [start, end) of the group in d_payload: states, then words */
    long long out;          /* output element of row 0, lane 0 */
    long long rows;         /* rows of the segment */
    long long table, cg;    /* table id in d_cum, 32-channel group */
    long long blob;         /* the d_status entry this unit reports to */
} vbq_rans_batch_unit;      /* 56 bytes: an (n_units, 7) int64 array */

typedef struct {
    long long first, count; /* units [first, first + count) */
    long long table, cg;    /* shared by all of them */
} vbq_rans_batch_cta;       /* 32 bytes: an (n_ctas, 4) int64 array */

int vbq_rans_decode_batch(const unsigned short *d_payload, long long payload_words, const unsigned short *d_cum,
                          const int *d_prob_bits, int n_tables, int C, int N, const vbq_rans_batch_unit *d_units,
                          long long n_units, const vbq_rans_batch_cta *d_ctas, long long n_ctas, int n_blobs,
                          const float *d_code_points, long long n_out, int *d_qidx, float *d_zhat, int *d_status,
                          void *stream);

/* ---- many images in one launch: the work-list encoder (DESIGN.md §8i) --------------------------------------------
 *
 * vbq_rans_encode_batch codes any set of groups of the layout above, from any number of images that share C and N but
 * may differ in rows, table, prob_bits and seg_rows, into n_blobs BLOBS back to back in d_payload.  Each blob is one
 * plane of one item: exactly the payload vbq_rans_encode writes for that item alone (its group end offset table, then
 * its groups).  Each group is a UNIT.  Inputs:
 *   d_in         (n_in,) int32 symbols; a unit codes rows r = 0 .. rows - 1 of lanes j < nact = min(32, C - 32 cg),
 *                symbol (r, j) at element in + r C + j;
 *   d_cum, d_prob_bits, n_tables: as for vbq_rans_decode_batch;
 *   d_units      (n_units,) vbq_rans_encode_unit;
 *   d_ctas       (n_ctas,) vbq_rans_batch_cta: CTA i codes units [first, first + count), 1 <= count <= 8, which must all
 *                have the descriptor's (table, cg): the CTA stages that table set once;
 *   d_blob_groups (n_blobs + 1,) int64: the first group of each blob in blob-major group order, [n_blobs] = n_groups;
 *   d_workspace  vbq_rans_encode_batch_workspace_bytes(n_groups, scratch_words) bytes: three int64 arrays of n_groups
 *                entries, then the scratch, in which unit u writes at most nact (rows + 2) words from word u.scratch on
 *                (the Python planner gives every unit its own range).
 * Outputs (no host synchronisation):
 *   d_payload    (payload_words,) uint16: blob b occupies words [d_blob_starts[b], d_blob_starts[b + 1]);
 *                2 n_groups + scratch_words words always suffice;
 *   d_blob_starts (n_blobs + 1,) int64, [n_blobs] = the payload size in words;
 *   d_status     (n_blobs,) int32, zeroed by the call: bit 1 if a symbol of the blob's groups lies outside [0, Q), bit 8
 *                for a bad unit or descriptor (of blob 0 if no valid blob id names the fault, as in
 *                vbq_rans_decode_batch), and bit 8 of blob 0 if d_blob_groups does not run from 0 to n_groups without
 *                decreasing (then every blob start is 0 and nothing is moved to the payload).
 * Units and descriptors come from the caller's memory, so the kernel checks each before it acts: 0 <= in and
 * in + (rows - 1) C + nact <= n_in, rows >= 1, table and cg in range and equal to the descriptor's, the table's
 * prob_bits valid, 0 <= group < n_groups, 0 <= blob < n_blobs, and 0 <= scratch with scratch + nact (rows + 2) inside
 * the workspace's scratch.  A bad unit writes no scratch and leaves its group's size 0.  Every write of the scan and the
 * compaction stays inside d_payload and the workspace whatever the units say; units that name one group twice, or
 * whose scratch ranges overlap, give an unspecified payload but no access out of bounds.  A blob's group data must stay
 * below 2^32 words (its offset table is 32-bit); the caller checks this from the worst case, nact (rows + 2) words per
 * group.  The scan is one CTA of 1,024 threads that walks the groups 1,024 at a time, so its time grows linearly with
 * n_groups (n_groups < 2^31).
 * Status codes: VBQ_ERR_BAD_DEPTH for N > 10, VBQ_ERR_BAD_SHAPE for a bad count or C, VBQ_ERR_WORKSPACE for a workspace
 * smaller than the three index arrays. */
typedef struct {
    long long in;           /* element of row 0, lane 0 in d_in */
    long long rows;         /* rows of the segment */
    long long table, cg;    /* table id in d_cum, 32-channel group */
    long long group;        /* the group's index in blob-major order */
    long long scratch;      /* first word of the unit's scratch range */
    long long blob;         /* the d_status entry this unit reports to */
} vbq_rans_encode_unit;     /* 56 bytes: an (n_units, 7) int64 array */

long long vbq_rans_encode_batch_workspace_bytes(long long n_groups, long long scratch_words);
int vbq_rans_encode_batch(const int *d_in, long long n_in, const unsigned short *d_cum, const int *d_prob_bits,
                          int n_tables, int C, int N, const vbq_rans_encode_unit *d_units, long long n_units,
                          const vbq_rans_batch_cta *d_ctas, long long n_ctas, const long long *d_blob_groups,
                          int n_blobs, long long n_groups, unsigned short *d_payload, long long payload_words,
                          long long *d_blob_starts, int *d_status, void *d_workspace, long long workspace_bytes,
                          void *stream);

/* ---- entropy coding with one shared table per plane: word embeddings (DESIGN.md §8d) ------------------------------
 *
 * All coordinates of an embedding matrix share one prior and one empirical model, so the channel axis of the layout
 * above has no meaning.  This layout codes a plane as one flat sequence with ONE table:
 *   PLANE   n int32 symbols q in [0, Q), Q = 2^(N+1)-1, N <= 10.  Symbol k sits at row k / 32, lane k % 32; a GROUP is
 *           a segment of seg_rows rows (seg_rows chosen per plane).  The lanes of a group that hold at least one symbol
 *           carry a state; on the plane's last row only the lanes with k < n take part.
 *   TABLES  d_cum (n_planes, Q+1) uint32 with cum[0] = 0, cum[s+1] - cum[s] = f[s] and cum[Q] = 2^prob_bits
 *           (12 <= prob_bits <= 16, Q <= 2^prob_bits).  Frequencies may be 0, and one symbol may hold all of 2^prob_bits
 *           (its symbols then cost nothing and the group is only its states).
 *   DECODER the decoded symbol is the largest s with cum[s] <= slot, which skips zero-frequency symbols wherever they
 *           sit.  State, renormalisation, word order, the per-plane group end offset table, the payload layout and the
 *           integrity rule (final state 2^16, every word read, every read inside the group's own range) are those of
 *           vbq_rans_decode, with groups in segment order.
 *
 * seg_rows is a HOST array of n_planes entries (1 <= n_planes <= VBQ_RANS_SHARED_MAX_PLANES), each >= 1; a value
 * above the plane's row count means one segment and is treated as that row count (the stream is the same).
 * vbq_rans_shared_workspace_bytes / vbq_rans_shared_payload_bound: the encoder's workspace and the worst-case payload in
 * bytes; -1 for a bad shape.  vbq_rans_shared_encode codes d_qidx (n_planes, n) in one launch into d_payload (at least
 * vbq_rans_shared_payload_bound bytes) and leaves the payload size in bytes in *d_payload_size, without host
 * synchronisation; *d_status gets bit 1 for a symbol outside [0, Q) and bit 2 for a symbol of frequency 0.
 * vbq_rans_shared_decode takes the group word ranges d_group_bounds (all groups of the call, 2) int64 [start, end) from
 * the offset tables and writes any of d_qidx (int32) and d_zhat (float32 d_code_points[q], a (Q,) ascending table) of
 * shape (n_planes, n); *d_status as for vbq_rans_decode. */
#define VBQ_RANS_SHARED_MAX_PLANES 64
long long vbq_rans_shared_workspace_bytes(int n_planes, long long n, const long long *seg_rows);
long long vbq_rans_shared_payload_bound(int n_planes, long long n, const long long *seg_rows);
int vbq_rans_shared_encode(const int *d_qidx, int n_planes, long long n, const long long *seg_rows, int N, int prob_bits,
                           const unsigned *d_cum, unsigned short *d_payload, long long payload_bytes,
                           long long *d_payload_size, int *d_status, void *d_workspace, long long workspace_bytes,
                           void *stream);
int vbq_rans_shared_decode(const unsigned short *d_payload, long long payload_words, const long long *d_group_bounds,
                           int n_planes, long long n, const long long *seg_rows, int N, int prob_bits,
                           const unsigned *d_cum, const float *d_code_points, int *d_qidx, float *d_zhat, int *d_status,
                           void *stream);

/* ---- row access into one shared-table plane: decoder checkpoints (DESIGN.md §8e) ---------------------------------
 *
 * A decoder's state at any row is fully determined by the stream, so one full pass can record it every K rows and a
 * later decode can start there.  Both functions take ONE plane (n symbols, seg_rows, N, prob_bits, d_cum (Q+1) uint32,
 * d_group_bounds (groups, 2) int64 word ranges into d_payload) as vbq_rans_shared_decode does, and checkpoint_rows
 * K >= 1; a K of at least the (clamped) segment length is treated as that length and records no checkpoint.
 *
 * CHECKPOINT INDEX (normative).  In segment g (rows r0 = g seg_rows .. r0 + len - 1), checkpoint j = 1 .. (len - 1) / K
 * is the decoder just before row r0 + j K: the word position of the next unread word as a uint32 offset from the
 * group's start word (its range start in d_group_bounds), and the 32 lane states as uint32 (a lane without a symbol in
 * the segment keeps 2^16).  It is entry c = g ((seg_rows - 1) / K) + j - 1 of d_offsets (M,) and d_states (M, 32), so
 * every full segment has (seg_rows - 1) / K entries and only the last segment may have fewer.  The segment start
 * (j = 0) is not stored: its states are the group's first words.  M = vbq_rans_shared_checkpoint_count(n, seg_rows, K);
 * the index takes 132 M bytes.
 *
 * vbq_rans_shared_checkpoints decodes the plane exactly as vbq_rans_shared_decode (same bounds, same status bits 1, 2
 * and 4, the same final integrity rule), writes no symbols and writes the index.
 *
 * vbq_rans_shared_decode_rows gathers embedding rows.  The plane is (n / row_size, row_size) symbols (row_size = D =
 * prod(shape[1:]) >= 1, dividing n); d_rows (n_req,) int64 are sorted, unique embedding rows.  One warp runs each of
 * the n_items WORK ITEMS of d_items: it restores checkpoint `checkpoint` of segment `segment` (0 = the segment's
 * start), decodes coder rows up to `last_row` (inside that checkpoint's interval [r0 + j K, min(r0 + (j+1) K, r0 +
 * len))) and writes every decoded symbol t (row t / 32, lane t % 32) whose embedding row t / D equals d_rows[u] for a u
 * in [lo, hi) to element (u, t - D d_rows[u]) of d_qidx (int32) and/or d_zhat (float32 d_code_points[q]), both
 * (n_req, D).  Items that cover disjoint coder rows write disjoint elements.  The kernel checks every field of every
 * item (segment and checkpoint in range, last_row inside the interval, 0 <= lo <= hi <= n_req, d_rows[lo..hi) strictly
 * increasing and below n / D): a bad item sets status bit 8 and writes nothing.  A partial decode cannot apply the
 * final-state rule, so only bits 1 (ran out of words) and 4 (bad group range or restored state below 2^16) remain.
 * Status codes: VBQ_ERR_BAD_SHAPE also for K < 1, row_size < 1 or not dividing n, n_req < 0 or above n / row_size. */
typedef struct {
    long long segment;      /* group of the plane */
    long long checkpoint;   /* j: 0 = the segment's start, else index entry segment ((seg_rows - 1) / K) + j - 1 */
    long long last_row;     /* the last coder row to decode, inside the checkpoint's interval */
    long long lo, hi;       /* the slice [lo, hi) of d_rows this item writes */
} vbq_rans_lookup_item;     /* 40 bytes: an (n_items, 5) int64 array */

long long vbq_rans_shared_checkpoint_count(long long n, long long seg_rows, long long checkpoint_rows);
int vbq_rans_shared_checkpoints(const unsigned short *d_payload, long long payload_words,
                                const long long *d_group_bounds, long long n, long long seg_rows, int N, int prob_bits,
                                const unsigned *d_cum, long long checkpoint_rows, unsigned *d_offsets,
                                unsigned *d_states, int *d_status, void *stream);
int vbq_rans_shared_decode_rows(const unsigned short *d_payload, long long payload_words,
                                const long long *d_group_bounds, long long n, long long seg_rows, int N, int prob_bits,
                                const unsigned *d_cum, long long checkpoint_rows, const unsigned *d_offsets,
                                const unsigned *d_states, const vbq_rans_lookup_item *d_items, long long n_items,
                                const long long *d_rows, long long n_req, long long row_size,
                                const float *d_code_points, int *d_qidx, float *d_zhat, int *d_status, void *stream);

/* ---- query scores against one shared-table plane (DESIGN.md §8f) ------------------------------------------------
 *
 * vbq_rans_shared_row_scores decodes the embedding rows [row_begin, row_end) of one plane (arguments as for
 * vbq_rans_shared_decode_rows; the plane is (n / row_size, row_size)) from the checkpoint index and writes
 * d_scores (n_queries, row_end - row_begin) float32: the dot product (metric VBQ_SCORE_DOT) or the cosine
 * (VBQ_SCORE_COSINE) of every query row of d_queries (n_queries, row_size) float32 with every embedding row.  The
 * matrix is never written.  1 <= n_queries <= vbq_rans_shared_score_max_queries(row_size) (the launch's query tile
 * sits in shared memory; 0 means no query of that length fits), or 0 for no work.
 *
 * NUMERICS (normative).  For query b and row e with D = row_size, z_d = d_code_points[symbol (e, d)], q_d =
 * queries[b, d], in IEEE float32 with round-to-nearest and no flush-to-zero (the kernel uses __fmaf_rn, __fadd_rn,
 * __fsqrt_rn, __fmul_rn and __fdiv_rn, so no contraction or build flag changes a bit):
 *     a0 = a1 = a2 = a3 = +0;  for d = 0 .. D-1: a[d % 4] = fmaf(z_d, q_d, a[d % 4]);  dot = (a0 + a1) + (a2 + a3)
 *     cosine: zz and qq by the same rule from z.z and q.q;  den = sqrtf(zz) * sqrtf(qq);
 *             cosine = den > 0 ? dot / den : 0
 * A score depends only on (b, e): not on the row range, the number of queries in the launch, the checkpoint interval
 * or the split of the work.
 *
 * WORK SPLIT.  With C1 = (seg_rows - 1) / K + 1 interval slots per segment, interval segment C1 + j holds coder rows
 * [segment seg_rows + j K, min(segment seg_rows + (j + 1) K, (segment + 1) seg_rows, rows)).  Warp w owns intervals
 * [w ipw, (w + 1) ipw) (ipw chosen by the function from the shape) and scores every row e of the range whose first coder
 * row floor(e D / 32) lies in them: it restores the checkpoint of the interval of its first such row and decodes, across
 * a segment boundary from the next group's initial states, up to the coder row of its last row's last symbol.  Every
 * row is scored whole by one warp; there are no partial sums across warps.
 *
 * Status: bit 1 = a group ran out of words, bit 4 = a bad group range or a restored state below 2^16 (as for
 * vbq_rans_shared_decode_rows); every word read stays inside its group's range.  VBQ_ERR_BAD_SHAPE also for a bad row
 * range, row_size not dividing n, too many queries or an unknown metric. */
#define VBQ_SCORE_DOT 0
#define VBQ_SCORE_COSINE 1
int vbq_rans_shared_score_max_queries(long long row_size);
int vbq_rans_shared_row_scores(const unsigned short *d_payload, long long payload_words,
                               const long long *d_group_bounds, long long n, long long seg_rows, int N, int prob_bits,
                               const unsigned *d_cum, long long checkpoint_rows, const unsigned *d_offsets,
                               const unsigned *d_states, long long row_size, long long row_begin, long long row_end,
                               const float *d_queries, int n_queries, int metric, const float *d_code_points,
                               float *d_scores, int *d_status, void *stream);

/* ---- exact target ranks against dense float32 rows (DESIGN.md §8g) ---------------------------------------------
 *
 * SCORES follow the numerics above (four accumulators a[d % 4] = fmaf(z_d, q_d, a[d % 4]) in d order, dot = (a0 + a1)
 * + (a2 + a3), cosine = dot / (sqrtf(zz) * sqrtf(qq)) when that product is > 0, else 0; _rn intrinsics throughout),
 * so a score here equals vbq_rans_shared_row_scores on the same float32 rows bit for bit.
 * ORDER is that of CompressedEmbedding.topk: the key of a score is the order-preserving map of its float32 bits, with
 * -0.0 equal to +0.0 and NaN lowest; row j BEATS target t of query i iff key(s_ij) > key(s_it), or the keys are equal
 * and j < t (ids are global row ids).  The RANK of t is 1 + the number of rows that beat it (minus any the caller
 * excludes); the target never beats itself.
 *
 * vbq_score_ranks ADDS to d_counts[i] (n_queries,) int64 the number of rows of the block d_rows (n_rows, row_size)
 * float32, whose first row has global id row_offset, that beat target d_targets[i] (n_queries,) int64 of query i of
 * d_queries (n_queries, row_size) float32, given d_thresholds[i] = s_it (float32, e.g. from vbq_pair_scores).  No
 * score is written; the counts are integers, so they do not depend on the tiling, the block split or the launch order.
 * Any n_rows >= 0, row_size >= 1 and 0 <= n_queries <= INT_MAX - 64.
 * vbq_pair_scores writes d_scores[p] = the score of query d_pair_queries[p] with row d_pair_rows[p] of d_rows, for
 * n_pairs pairs (both index arrays int64; a pair with an index out of range gets NaN).
 * Status codes: VBQ_ERR_BAD_SHAPE for a bad size or an unknown metric (VBQ_SCORE_DOT / VBQ_SCORE_COSINE). */
int vbq_score_ranks(const float *d_rows, long long n_rows, long long row_size, long long row_offset,
                    const float *d_queries, long long n_queries, int metric, const float *d_thresholds,
                    const long long *d_targets, long long *d_counts, void *stream);
int vbq_pair_scores(const float *d_rows, long long n_rows, long long row_size, const float *d_queries,
                    long long n_queries, const long long *d_pair_rows, const long long *d_pair_queries,
                    long long n_pairs, int metric, float *d_scores, void *stream);

/* ---- image quality: exact SSE and MS-SSIM levels (DESIGN.md §8j) -------------------------------------------------
 *
 * d_x (N, H, W, C) uint8 are N originals and d_y (M, N, H, W, C) uint8 are M reconstructions of each (1 <= C <= 4).
 * For every pair (m, n), vbq_image_metrics writes d_sse[m, n] (M, N) int64 = the exact sum over H W C of
 * (x - y)^2, and d_ssim[m, n, k] / d_cs[m, n, k] (M, N, 5) float64 = the means of ssim and cs at pyramid level k of
 * TF models' MultiScaleSSIM with max_val 255 (k1 = 0.01, k2 = 0.03): level k + 1 is the 2 x 2 mean of level k with
 * the last row or column repeated at an odd size; at each level the window is _FSpecialGauss(s, 1.5 s / 11) with
 * s = min(11, h, w), the moments are filtered over the valid positions, and the means run over all valid positions
 * and all channels.  The moments are computed in float64 with a separable window (agreeing with the reference's FFT
 * filtering to about 1e-14 relative); the sums over positions run in a fixed order, so two calls give the same bits.
 * MS-SSIM = prod_k<4 cs[k]^w[k] * ssim[4]^w[4] and PSNR are left to the caller.
 * d_workspace: vbq_image_metrics_workspace_bytes(N, M, H, W, C) bytes, 16-byte aligned (-1 for a bad shape).
 * N = 0 or M = 0 is no work.  Status codes: VBQ_ERR_BAD_SHAPE for a bad size, VBQ_ERR_WORKSPACE for a workspace
 * missing or too small. */
long long vbq_image_metrics_workspace_bytes(long long N, long long M, int H, int W, int C);
int vbq_image_metrics(const unsigned char *d_x, const unsigned char *d_y, long long N, long long M, int H, int W,
                      int C, void *d_workspace, long long workspace_bytes, long long *d_sse, double *d_ssim,
                      double *d_cs, void *stream);

/* ---- stand-alone operator forms------------------------------------------------------------------------------- */

/* ChannelwisePriorCDFQuantizer.get_all_N_bit_intervals (quantizer.py:65-80): d_mu (rows, C) -> d_left, d_right
 * (C, N+1, rows): at every bit depth the largest code point below mu and the smallest one >= mu, with the edge
 * semantics of the reference's padded search grids. */
int vbq_intervals(const float *d_mu, long long rows, int C, const float *d_table, int N, float *d_left,
                  float *d_right, void *stream);

/* utils.batch_quantize_indep_dims (utils.py:363-423) on explicit candidates: d_P (M, BK) float32 code points,
 * d_L (M, BK) or (n_lambda, M, BK) code lengths (int32, or float32 when l_is_float), scores
 * fun_P - fl(lambda*L) with fun_P = d_funP (M, BK) if given, else -0.5*((P-loc)/scale)^2 (utils.py:318-320) from
 * d_loc, d_scale (BK).  Outputs (n_lambda, BK): chosen code point, its code length (dtype of d_L), optional index. */
int vbq_argmax_candidates(const float *d_P, const void *d_L, int l_is_float, int l_per_lambda, const float *d_funP,
                          const float *d_loc, const float *d_scale, const float *d_lambs, int n_lambda, int M,
                          long long BK, float *d_zhat, void *d_bits, int *d_index, void *stream);

/* Self-test helper: out[i] = the kernel's division a[i]/b[i] (reciprocal + FMA correction) so that tests can
 * compare it with IEEE division bit for bit. */
int vbq_selftest_divide(const float *d_a, const float *d_b, long long n, float *d_out, void *stream);

/* Self-test helper: out[i] = the sigma every search kernel derives from a log-variance input lv[i] under
 * VBQ_FLAG_LOGVAR (sqrt(exp(lv)) with CUDA's expf and sqrtf), so that tests can hand the oracle the kernels' sigma. */
int vbq_selftest_sigma_from_logvar(const float *d_lv, long long n, float *d_out, void *stream);

/* Self-test helper (host only): out[b] .. out[b+1] is the range of 4-row x 16-channel tiles, in (channel group, row)
 * order, that CTA b of a `grid`-CTA launch of the bisection kernels processes; out has grid+1 entries. */
int vbq_selftest_span_cuts(long long rows, int C, int grid, long long *out);

#ifdef __cplusplus
}
#endif
#endif /* VBQ_B200_H */
