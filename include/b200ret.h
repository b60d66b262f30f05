/*
 * b200ret.h — C-ABI of libb200ret.so: the B200 (sm_100a) implementation of the two hot paths of
 * ArseneAmoya/image-retrieval-wavelet.  Plain pointers and sizes only; no torch / ATen types.
 *
 * All paths below are relative to /root/reference (the upstream project).
 *
 * Conventions
 *   - every function returns B200_OK (0) or a negative B200_ERR_* code; b200_error_string() names the code and
 *     b200_last_cuda_error() gives the CUDA runtime message of the calling thread's last B200_ERR_CUDA.
 *   - "device pointer" arguments must point to memory of the current CUDA device; work is enqueued on `stream`
 *     (a cudaStream_t passed as void*; NULL = legacy default stream) and is stream-ordered: no hidden
 *     synchronisation, no hidden allocation.  Scratch memory is caller-provided and sized by the matching
 *     *_workspace_bytes() query.
 *   - the library keeps no global mutable state besides per-function CUDA attributes; entry points are re-entrant.
 *   - the *_host entry points take HOST buffers, do their own H2D/D2H copies and synchronise before returning:
 *     they are what a non-CUDA caller (the reference's DataLoader / evaluator glue) binds directly.
 *
 * Packed formats
 *   codes   uint64 [rows][CW], CW = b200_code_words(B) in {1, 2, 4}; bit (b % 64) of word (b / 64) is set iff
 *           code[row][b] > 0; padding bits / words are 0.
 *   labels  multi-hot: uint64 [rows][LW], LW = b200_label_words(L) in {1, 2, 4}, bit l set iff label[row][l] != 0
 *           scalar   : uint64 [rows][1], a canonical bit pattern of the label value (equal values <=> equal words)
 *   Every packed buffer must have room for `rows` rounded up to a multiple of 2 (16-byte granularity of the
 *   bulk-copy engine); the pack kernels zero the padding row.
 */
#ifndef B200RET_H_
#define B200RET_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_ERR_INVALID_ARG (-1)  /* NULL pointer, negative size, bad enum                            */
#define B200_ERR_UNSUPPORTED (-2)  /* legal request outside the compiled envelope (e.g. B > 256)       */
#define B200_ERR_CUDA (-3)         /* a CUDA runtime call failed; see b200_last_cuda_error()           */
#define B200_ERR_WORKSPACE (-4)    /* workspace NULL or smaller than *_workspace_bytes()               */
#define B200_ERR_ALIGNMENT (-5)    /* pointer not aligned as documented                                */
#define B200_ERR_NO_DEVICE (-6)    /* no sm_100 device / kernel image not loadable                     */

#define B200_LABELS_OVERLAP 0 /* 2-D multi-hot labels: relevant iff the label sets intersect           */
#define B200_LABELS_EQUAL 1   /* 1-D labels: relevant iff equal                                        */

#define B200_MAX_CODE_BITS 256
#define B200_MAX_LABEL_BITS 256
#define B200_SWT_MAX_FILTER 20
#define B200_SWT_MAX_LEVEL 4

typedef void *b200_stream_t;

int b200_version(void);
/* sizeof(b200_map_plan) as this library was built: bindings that mirror the struct check it at load time. */
size_t b200_sizeof_map_plan(void);
const char *b200_error_string(int code);
const char *b200_last_cuda_error(void);
/* Number of kernel launches issued by this library since load (all threads); bench.py's "gpu_launches". */
unsigned long long b200_launch_count(void);

/* words per packed row: 1 (<= 64 bits), 2 (<= 128) or 4 (<= 256) */
static inline int b200_code_words(int bits) { return bits <= 64 ? 1 : (bits <= 128 ? 2 : 4); }
static inline int b200_label_words(int labels) { return labels <= 64 ? 1 : (labels <= 128 ? 2 : 4); }

/* ============================================================================================== HP-SWT
 * Replaces, for a whole batch already on the device, the per-image CPU path
 *   BaseWaveletTransform.__call__        main/transforms/custom_transforms.py:145-157
 *   SWTTransform._apply_wavelet          main/transforms/custom_transforms.py:163-166  (pywt.swt2, coeffs[0])
 * in  : [B][C][H][W] uint8 (scaled by 1/255 as custom_transforms.py:147 does) or float32, device, contiguous
 * out : [B][C][4][H][W] float32, device; band order cA, cH, cV, cD = LL, LH, HL, HH of level `level` only
 * dec_lo / dec_hi : HOST pointers to the F decomposition taps (PyWavelets convention), F even, 2 <= F <= 20
 * H and W must be divisible by 2^level (fix_size, custom_transforms.py:132-139, stays on the host side).
 */
int b200_swt2_fwd(const void *in, int in_is_u8, float *out, int B, int C, int H, int W, const float *dec_lo,
                  const float *dec_hi, int F, int level, b200_stream_t stream);

/* RawStackTransform._apply_wavelet  main/transforms/custom_transforms.py:172-188: `copies` identical planes.
 * out : [B][C][copies][H][W] float32. */
int b200_raw_stack(const void *in, int in_is_u8, float *out, int B, int C, int H, int W, int copies,
                   b200_stream_t stream);

/* Host-buffer form of b200_swt2_fwd (what SWTTransform.__call__ binds for a single PIL image):
 * in_host is HWC-interleaved uint8 [H][W][C] when in_is_hwc_u8 != 0 (np.array(PIL image)), else planar
 * [B][C][H][W] uint8/float32 as above.  out_host: [B][C][4][H][W] float32. */
int b200_swt2_fwd_host(const void *in_host, int in_is_u8, int in_is_hwc, float *out_host, int B, int C, int H, int W,
                       const float *dec_lo, const float *dec_hi, int F, int level);

/* ---- the pixel step in front of the SWT (SURVEY.md §8 f3)
 * BaseWaveletTransform.fix_size, main/transforms/custom_transforms.py:132-139: PIL bicubic resize up to a multiple
 * of 2^level (518 -> 520 for levels 2-3), and the antialiased bilinear PIL resize behind torchvision's Resize in the
 * eval transforms (config/transform/NAME.yaml).  Bit-exact restatement of Pillow's 8-bit resampler (Resample.c:
 * double-precision windowed weights rounded to 22-bit fixed point, horizontal then vertical pass through a uint8
 * intermediate, a pass skipped when its size does not change).
 * in : uint8 [planes][H][W] device;  out : uint8 [planes][Hout][Wout] device;  workspace: device scratch of
 * b200_resize_workspace_bytes() (intermediate plane + weight tables, which are computed on the host per call). */
#define B200_RESIZE_BICUBIC 0
#define B200_RESIZE_BILINEAR 1
size_t b200_resize_workspace_bytes(long long planes, int H, int W, int Hout, int Wout, int filter);
int b200_resize_u8(const uint8_t *in, uint8_t *out, long long planes, int H, int W, int Hout, int Wout, int filter,
                   void *workspace, size_t workspace_bytes, b200_stream_t stream);

/* Resize + crop of a ragged batch of decoded images in one launch: the eval transform Resize(256) -> CenterCrop(224)
 * (config/transform/basic_swt.yaml) applied to every image, bit-identical to torchvision on PIL images.
 * in           : device; image i is HWC-interleaved uint8 [H_i][W_i][C] (row pitch W_i * C bytes) at byte
 *                offsets_host[i] of `in`.  `in` and every offset must be multiples of 4 (B200_ERR_ALIGNMENT).
 * geom_host    : HOST int [n][6] = H, W, RH, RW, top, left per image: the resized size (Pillow's Image.resize with
 *                `filter`, exactly as b200_resize_u8) and the crop origin inside it; 0 <= top <= RH - Hc and
 *                0 <= left <= RW - Wc (B200_ERR_INVALID_ARG otherwise).  The size and crop rules of torchvision stay with
 *                the caller.
 * out          : device uint8 [n][C][Hc][Wc] (planar, the layout b200_swt2_fwd takes);  C in 1..4.
 * workspace    : device scratch of b200_resize_crop_workspace_bytes() (per-image descriptors and the weight tables of the
 *                crop windows, built on the host per call and copied with one H2D copy).
 * B200_ERR_UNSUPPORTED when a window is wider than 64 taps (a reduction of more than ~31x bilinear / ~15x bicubic).
 * n = 0 is a no-op; the workspace query returns 0 for n < 1 and for arguments the call rejects. */
size_t b200_resize_crop_workspace_bytes(int n, const int *geom_host, int C, int Hc, int Wc, int filter);
int b200_resize_crop_u8(const uint8_t *in, const long long *offsets_host, const int *geom_host, int n, int C, int Hc, int Wc,
                        int filter, uint8_t *out, void *workspace, size_t workspace_bytes, b200_stream_t stream);

/* ---- the decimated transform next to the SWT (SURVEY.md §8 f4)
 * DWTTransform._apply_wavelet, main/transforms/custom_transforms.py:196-200: pywt.wavedec2(channel, wavelet, level)
 * in PyWavelets' default 'symmetric' mode, keeping the coarsest level: out [planes][4][H_L][W_L] = (cA, cH, cV, cD),
 * H_l = b200_dwt_out_len(H_{l-1}, F) = floor((H_{l-1} + F - 1) / 2).  in: uint8 (scaled by 1/255) or float32
 * [planes][H][W], device; dec_lo / dec_hi: HOST pointers to the F taps; workspace: b200_dwt2_workspace_bytes(). */
static inline int b200_dwt_out_len(int n, int F, int level) {
    for (int l = 0; l < level; ++l) n = (n + F - 1) / 2;
    return n;
}
size_t b200_dwt2_workspace_bytes(long long planes, int H, int W, int F, int level);
int b200_dwt2_fwd(const void *in, int in_is_u8, float *out, long long planes, int H, int W, const float *dec_lo,
                  const float *dec_hi, int F, int level, void *workspace, size_t workspace_bytes, b200_stream_t stream);

/* ============================================================================================== HP-EVAL
 * sign()/multi-hot -> bit packing of what compute_all_embeddings (main/engine/evaluate.py:26-64) hands over.
 * codes  : float32 [N][B] device.  n_invalid (device int32, caller-zeroed) is incremented by the number of
 *          entries that are not exactly +1 or -1 (sign(0) = 0, raw logits, NaN): such inputs have no Hamming
 *          distance in the sense of accuracy_calculator.py:183-186 and the caller must reject them.
 * labels : float32 [N][L] multi-hot; n_invalid counts entries that are neither 0 nor 1. */
int b200_pack_codes(const float *codes, long long N, int B, uint64_t *packed, int *n_invalid, b200_stream_t stream);
int b200_pack_labels(const float *labels, long long N, int L, uint64_t *packed, int *n_invalid, b200_stream_t stream);
/* 1-D labels (accuracy_calculator.py:37 equality branch): is_int64 = 0: float32 values, 1: int64, 2: float64.  Equal
 * values give equal words across the three (5, 5.0f and 5.0 compare equal, like the reference's promoting `==`). */
int b200_pack_labels_scalar(const void *labels, int is_int64, long long N, uint64_t *packed, int *n_invalid,
                            b200_stream_t stream);

/* per_bit_balance numerator, accuracy_calculator.py:188-194: ones[b] = #{rows with bit b set}, uint32 [B]. */
int b200_bit_counts(const uint64_t *packed_codes, long long N, int B, uint32_t *ones, b200_stream_t stream);

/* Dense utilities for API parity (the fused evaluator never materialises them):
 * calc_hamming_dist, accuracy_calculator.py:183-186 -> dist float32 [Q][N] (exact integers 0..B);
 * label_comparison_fn, accuracy_calculator.py:31-37  -> rel uint8 [Q][N]. */
int b200_hamming_dist(const uint64_t *q_codes, const uint64_t *db_codes, int Q, long long N, int B, float *dist,
                      b200_stream_t stream);
int b200_label_relevance(const uint64_t *q_labels, const uint64_t *db_labels, int Q, long long N, int LW, int label_mode,
                         uint8_t *rel, b200_stream_t stream);

/* calculate_maphashing, accuracy_calculator.py:203-231, for one database shard.
 *
 * Ranking is ascending (Hamming distance, global database index) — torch.argsort's tie order made
 * deterministic.  AP_q = mean over the relevant items among the first k ranks of (hit ordinal / rank);
 * queries without a hit get AP 0 and still count in the mean (accuracy_calculator.py:226-231).
 *
 * The evaluation is a counting sort in three stream-ordered stages so that a sharded database only has to
 * exchange per-query histograms (b200_hamming_hist -> all-gather of totals -> b200_hamming_scan ->
 * b200_hamming_ap -> b200_ap_reduce -> all-gather -> b200_ap_finalize).  b200_hamming_map runs all of them for
 * the single-shard case.
 *
 * q_codes [Q][CW], q_labels [Q][LW], db_codes [N][CW], db_labels [N][LW]: packed, device.
 * k : ranks that count (0 < k; values > total database size mean "all", like topk=None).
 */
typedef struct b200_map_plan {
    int Q;             /* queries                                                         */
    long long N;       /* database rows in THIS shard                                     */
    long long N_total; /* rows over all shards (== N when unsharded)                      */
    int B;             /* code bits, 1..256                                               */
    int LW;            /* label words, 1..4                                               */
    int label_mode;    /* B200_LABELS_OVERLAP / B200_LABELS_EQUAL                         */
    long long k;       /* top-k, already clamped to [1, N_total]                          */
    /* filled by b200_map_plan_init: launch geometry + workspace carve-up */
    int bins, T, groups, Qpad, S, seg_len, wide, tile;
    int stash;         /* 1: stage A keeps (distance, relevance) of every (row, query) pair in the workspace and
                          stage B ranks from that stash instead of scoring again.  Chosen when 4k <= N_total,
                          B <= 254 and the stash takes less than 24576 MB; B200_MAP_STASH=0/1 forces it off / on */
    size_t off_hist, off_tot, off_dstar, off_psum, off_phits, off_stash_d, off_stash_r, workspace_bytes;
    /* Select mode (single shard, 8k <= N_total, B <= 254; B200_MAP_SELECT=0/1 forces): the top k are a small part of the
     * database, so instead of counting every (row, query) pair into per-distance histograms, a sampled histogram
     * (every sel_stride-th 32-row group) gives each query a distance bound that covers its top k with 5-sigma margin;
     * ONE pass over the database keeps only the rows within the bound as compact per-(query, segment) candidate lists
     * (chunks of sel_chunk entries from a pool), and one warp per query then counting-sorts its own list (exact: a
     * query whose list turns out shorter than k is redone with the bound lifted; a pool overflow hands the whole
     * problem to the three-stage path above, whose kernels are otherwise gated off).  b200_hamming_map and
     * b200_hamming_topk take this path by themselves; the staged API (hist / scan / ap) never does.
     * The one pass has two forms, and the plan alone decides which.  Tensor-core form (when the queries come in groups of
     * 128, the hit masks fit 4 GB and the e4m3 codes 8 GB): the +-1 codes are expanded to e4m3 bytes and a tcgen05 fp8 GEMM
     * (dot = B - 2 distance, exact) writes one hit bit per (row, query) — off_smp_codes then points at the e4m3 copies and
     * the masks, otherwise off_smp_codes == workspace_bytes — and a SIMT kernel scores only the hit rows again and appends
     * them.  SIMT form: XOR + POPC of every pair in the same kernel that appends. */
    int select, sel_stride, sel_S, sel_seg_len, sel_chunk, sel_maxc, smp_S, smp_seg_len, sel_T;
    long long smp_rows, sel_pool_chunks;
    size_t off_sel_flags, off_sel_bound, off_sel_count, off_sel_table, off_sel_pool, off_smp_codes, off_smp_hist;
} b200_map_plan;

/* Chooses the launch geometry for the current device and sizes the workspace.  n_shards/shard are only
 * recorded by the caller; pass N_total = N for a single shard. */
int b200_map_plan_init(b200_map_plan *plan, int Q, long long N, long long N_total, int B, int LW, int label_mode,
                       long long k);

/* Stage A: per-(segment, distance, query) counts of (all, relevant) rows -> workspace; and the shard totals
 * tot[bins][Qpad] as uint32 pairs (all, rel) at workspace + plan->off_tot (what a sharded run all-gathers). */
int b200_hamming_hist(const b200_map_plan *plan, const uint64_t *q_codes, const uint64_t *q_labels,
                      const uint64_t *db_codes, const uint64_t *db_labels, void *workspace, b200_stream_t stream);
/* Stage S: turns counts into rank / hit-ordinal bases.  tot_all_shards = NULL (single shard) or device
 * uint32 [n_shards][bins][Qpad][2] gathered from every shard's off_tot block, shard = this shard's position
 * in global index order. */
int b200_hamming_scan(const b200_map_plan *plan, void *workspace, const uint32_t *tot_all_shards, int n_shards,
                      int shard, b200_stream_t stream);
/* Stage B: per-(segment, query) partial sum of (ordinal / rank) [double] and hit counts [uint32] -> workspace.
 * Optionally materialises this shard's part of the ranked list: for every row whose global rank r <= k,
 * rank_idx[q][r-1] = index_base + row, rank_dist[q][r-1] = distance (either may be NULL).  rank_idx/rank_dist
 * have row stride k. */
int b200_hamming_ap(const b200_map_plan *plan, const uint64_t *q_codes, const uint64_t *q_labels,
                    const uint64_t *db_codes, const uint64_t *db_labels, void *workspace, uint32_t *rank_idx,
                    uint16_t *rank_dist, long long index_base, b200_stream_t stream);
/* Per-query reduction of this shard's stage-B partials over its segments: sum_q uint64 [Q] (sum of hit-ordinal / rank
 * as exact 2^-40 fixed point — integer, hence independent of the segment / shard decomposition), hits_q uint32 [Q]:
 * the two small vectors a sharded run all-gathers. */
int b200_ap_reduce(const b200_map_plan *plan, void *workspace, uint64_t *sum_q, uint32_t *hits_q, b200_stream_t stream);
/* AP_q = (sum over parts of sums[p*stride + q]) / 2^40 / (sum over parts of hits[p*stride + q]); AP_q = 0 without a
 * hit.  ap double [Q], tsum uint32 [Q] (may be NULL), map_out[0] = mean AP (may be NULL). */
int b200_ap_finalize(const uint64_t *sums, const uint32_t *hits, int n_parts, long long stride, int Q, double *ap,
                     uint32_t *tsum, double *map_out, b200_stream_t stream);

/* All stages for an unsharded database. */
int b200_hamming_map(const b200_map_plan *plan, const uint64_t *q_codes, const uint64_t *q_labels,
                     const uint64_t *db_codes, const uint64_t *db_labels, void *workspace, double *ap, uint32_t *tsum,
                     double *map_out, b200_stream_t stream);

/* b200_hamming_map without its rarely needed tail, for callers that read a result back anyway (a CUDA-graph step): runs
 * the select pipeline's first round only (or the three stages for a non-select plan) and sets the device word *status
 * (caller-zeroed) to 1 when that was not enough — a query's candidate list came out short or the pool overflowed; the
 * caller then repeats the evaluation with b200_hamming_map.  ap / tsum of the other queries are final either way. */
int b200_hamming_map_try(const b200_map_plan *plan, const uint64_t *q_codes, const uint64_t *q_labels,
                         const uint64_t *db_codes, const uint64_t *db_labels, void *workspace, double *ap, uint32_t *tsum,
                         uint32_t *status, b200_stream_t stream);
/* Last kernel of such a step: out2[0] = mean of ap[0..Q) (accuracy_calculator.py:231, same fixed-shape tree as
 * b200_mean_f64), out2[1] = 1.0 when any of the n_status uint32 words at status + r * status_stride is non-zero. */
int b200_map_final(const double *ap, int Q, const void *status, int n_status, long long status_stride, double *out2,
                   b200_stream_t stream);

/* b200_hamming_map with a CUDA event behind every stage (synchronises): ms_out[i] / names_out[i] (static strings) for
 * i < *n_stages <= max_stages — "sample_hist", "bound", ["expand", "filter",] "select", "rank", ... for a select plan, "hist", "scan", "ap",
 * "finalize" for the three stages.  bench.py's per-kernel roofline numbers come from here. */
int b200_hamming_map_stage_ms(const b200_map_plan *plan, const uint64_t *q_codes, const uint64_t *q_labels,
                              const uint64_t *db_codes, const uint64_t *db_labels, void *workspace, double *ap, uint32_t *tsum,
                              int max_stages, float *ms_out, const char **names_out, int *n_stages, b200_stream_t stream);

/* Diagnostics of the select pipeline after a b200_hamming_map / b200_hamming_topk call on `workspace` (synchronises the
 * stream): out[0] = pool chunks used, out[1] = 1 when the pipeline gave up and the three-stage path produced the result,
 * out[2] = queries redone with the bound lifted, out[3] = estimated candidates per query (from the sample).
 * Returns B200_ERR_INVALID_ARG when the plan is not a select plan. */
int b200_map_select_status(const b200_map_plan *plan, const void *workspace, uint32_t *out4, b200_stream_t stream);

/* Fused top-k: the ranked list itself (hamming "knn", get_knn.py:9-24 with distance_metric="hamming", and
 * get_accuracy(return_indices=True), accuracy_calculator.py:347-348).  idx uint32 [Q][k], dist uint16 [Q][k]. */
int b200_hamming_topk(const b200_map_plan *plan, const uint64_t *q_codes, const uint64_t *db_codes, void *workspace,
                      uint32_t *idx, uint16_t *dist, b200_stream_t stream);

/* Relevance + AP over a ranked list (calculate_map, accuracy_calculator.py:156-167, and the list-merge
 * form of the sharded evaluator).  idx: int64 [Q][k] (is_int64) or uint32 [Q][k]; rows with idx < 0 /
 * 0xFFFFFFFF are padding.  query_mask (uint8 [Q], may be NULL) selects the queries that enter the mean.
 * ap double [Q], hits uint32 [Q], map_out[0] = mean over selected queries. */
int b200_ranked_ap(const void *idx, int is_int64, int Q, long long k, const uint64_t *q_labels,
                   const uint64_t *db_labels, int LW, int label_mode, const uint8_t *query_mask, double *ap,
                   uint32_t *hits, double *map_out, b200_stream_t stream);

/* k-way merge of n_shards per-shard ranked lists (each sorted by (dist, idx), shards in ascending index
 * order) into the global top-k: the "all-gather then merge" step of the sharded evaluator.
 * in_idx uint32 [n_shards][Q][k], in_dist uint16 [n_shards][Q][k] (0xFFFF = padding) -> out_idx/out_dist [Q][k]. */
int b200_merge_topk(const uint32_t *in_idx, const uint16_t *in_dist, int n_shards, int Q, long long k, int B,
                    uint32_t *out_idx, uint16_t *out_dist, b200_stream_t stream);

/* ---- other Hamming metrics on the same scan (SURVEY.md §8 f2)
 * Counts within every Hamming radius: after b200_hamming_hist on `workspace`,
 *   cum[d][q] = (#database rows, #relevant database rows) of query q with distance <= d, uint32 [B+1][Q][2].
 * All DSCH pr_curve (main/engine/DSCH/_utils.py:467-492) and get_precision_recall_by_Hamming_Radius
 * (_utils.py:577-594) need; replaces their [Q][N] float distance / relevance matrices. */
int b200_hamming_radius_counts(const b200_map_plan *plan, const void *workspace, uint32_t *cum, b200_stream_t stream);

/* Relevance along a ranked list as a running hit count: cum[q][p] = #relevant among ranks 1..p+1 of query q
 * (gnd[argsort(hamm)] -> cumsum of calculate_pr_rc_hashing, main/engine/accuracy_calculator.py:247-254; DSCH
 * p_topK, _utils.py:495-512, reads cum[q][K-1]).  idx uint32 [Q][k] (0xFFFFFFFF = padding), cum uint32 [Q][k]. */
int b200_ranked_cumhits(const uint32_t *idx, int Q, long long k, const uint64_t *q_labels, const uint64_t *db_labels,
                        int LW, int label_mode, uint32_t *cum, b200_stream_t stream);
/* Tail of calculate_pr_rc_hashing (accuracy_calculator.py:255-265): over the queries with query_mask[q] != 0
 * (NULL: all) that have a relevant row (cum[q][k-1] > 0),
 *   prec_sum[p] += float32(cum[q][p] / (p+1)),  rec_sum[p] += float32(cum[q][p] / cum[q][k-1]),  n_used[0] += 1.
 * Accumulates INTO the caller-zeroed double [k] / uint32 [1] buffers so that queries can be streamed in chunks. */
int b200_curve_accumulate(const uint32_t *cum, int Q, long long k, const uint8_t *query_mask, double *prec_sum,
                          double *rec_sum, uint32_t *n_used, b200_stream_t stream);

/* Continuous-embedding k-NN, get_knn.py:9-24,60-71: top-k by inner product (cosine / "hamming" metrics,
 * largest first) or by L2 distance (smallest first), ties by index.  refs float32 [N][D], queries float32
 * [Q][D] device; idx int64 [Q][k], score float32 [Q][k] (inner product, or L2 distance).  -0.0 equals +0.0 (reported
 * as +0.0); a NaN score or distance ranks after every number for both metrics.  +-inf coordinates: L2 only (the
 * tensor-core scorer's bf16 hi/lo split makes an inner product with them NaN). */
size_t b200_knn_workspace_bytes(int Q, long long N, int D, int k);
int b200_knn_topk(const float *refs, const float *queries, int Q, long long N, int D, int k, int metric_l2,
                  int64_t *idx, float *score, void *workspace, size_t workspace_bytes, b200_stream_t stream);

/* mean of ap[0..Q) over the queries with query_mask[q] != 0 (NULL: all) -> out[0]; one CTA, fixed-shape tree
 * (bit-reproducible).  The last line of calculate_maphashing, accuracy_calculator.py:231. */
int b200_mean_f64(const double *ap, const uint8_t *query_mask, int Q, double *out, b200_stream_t stream);

/* ============================================================================================== multi-GPU exchange
 * One process per GPU on one box; replaces the host-side merge of faiss' sharded index (main/engine/get_knn.py:41-44).
 * Every rank creates one region of the same size; the regions are mapped into every peer through CUDA IPC (NVLink /
 * NVSwitch peer access) and laid out identically by the caller.  Producers store straight into every rank's copy
 * (b200_pack_to_ranks, b200_comm_put) and b200_comm_barrier — a stream-ordered kernel: one release store per peer, one
 * acquire spin per peer — replaces the rendezvous of a collective.  All of it is CUDA-graph capturable.
 *   create (collective by convention) -> export my 64-byte handle -> exchange the handles out of band (e.g.
 *   torch.distributed.all_gather) -> open -> use -> destroy. */
#define B200_COMM_MAX_RANKS 16
#define B200_COMM_HANDLE_BYTES 64
typedef struct b200_comm b200_comm;
int b200_comm_create(int rank, int world, size_t bytes, b200_comm **out);
int b200_comm_export(b200_comm *comm, void *handle64);
int b200_comm_open(b200_comm *comm, const void *handles /* world x 64 bytes, rank order */);
void *b200_comm_buffer(b200_comm *comm, int rank); /* device pointer of rank's region as mapped in this process */
size_t b200_comm_bytes(b200_comm *comm);
int b200_comm_world(b200_comm *comm);
int b200_comm_rank(b200_comm *comm);
/* Every store this rank issued to peer regions earlier in `stream` is visible to a peer once the peer's matching
 * barrier returns.  Gives up after ~2 s without a peer (b200_comm_status reports it) instead of hanging the GPU. */
int b200_comm_barrier(b200_comm *comm, b200_stream_t stream);
/* region[r][dst_offset[k] .. +bytes[k]) = src[k][0 .. bytes[k]) for every rank r and segment k < n_segments <= 4, one
 * launch; src / offsets / sizes 16-byte aligned. */
int b200_comm_put(b200_comm *comm, int n_segments, const void *const *src, const size_t *dst_offset, const size_t *bytes,
                  b200_stream_t stream);
/* Last kernel of a multi-GPU evaluation step, one single-CTA launch: b200_comm_put of the segments, b200_comm_barrier,
 * then b200_map_final over the Q float64 values at ap_offset and the world uint32 status words (16 bytes apart) at
 * status_offset of the LOCAL region — the same summation order as b200_map_final, so out2[0] is bit-identical to the
 * single-GPU mean (accuracy_calculator.py:231).  Offsets 16-byte aligned. */
int b200_comm_put_barrier_final(b200_comm *comm, int n_segments, const void *const *src, const size_t *dst_offset,
                                const size_t *bytes, size_t ap_offset, int Q, size_t status_offset, double *out2,
                                b200_stream_t stream);
/* b200_pack_codes (is_codes != 0) / b200_pack_labels of this rank's rows, written at dst_offset of EVERY rank's
 * region: the packed shard is all-gathered by the pack kernel itself. */
int b200_pack_to_ranks(const float *src, int is_codes, long long N, int cols, b200_comm *comm, size_t dst_offset,
                       int *n_invalid, b200_stream_t stream);
int b200_comm_status(b200_comm *comm, int *timed_out); /* synchronous read of the region's status word */
/* device address of that uint32 status word (non-zero: a barrier timed out), for callers that copy it back themselves
 * as part of a captured launch sequence */
const void *b200_comm_status_word(b200_comm *comm);
int b200_comm_destroy(b200_comm *comm);

/* Top-k of every row of a float32 matrix on the device (row stride ldS, a multiple of 4; 16-byte aligned base):
 * idx int64 [Q][k] = column numbers, score float32 [Q][k]; largest != 0: largest first, else smallest first; ties to
 * the smaller column, -0.0 equals +0.0 (reported as +0.0), NaN ranks after every number for either `largest`;
 * any k <= N.  The merge step of the database-sharded k-NN (get_knn.py:41-44: faiss merges its
 * shards on the host): per-shard (score, index) lists concatenated in shard order are such a matrix. */
int b200_select_topk_f32(const float *S, int Q, long long N, long long ldS, int k, int largest, int64_t *idx, float *score,
                         b200_stream_t stream);

/* Host-buffer evaluator: CustomCalculator.calculate_maphashing as the reference calls it (float32 +-1 codes
 * and float32 labels in host memory).  labels: multi-hot [.,L] when label_mode == OVERLAP, [.,1] when EQUAL.
 * Does H2D, pack, the three stages and D2H; ap_out[Q] (may be NULL), *map_out = mean AP.
 * Returns B200_ERR_INVALID_ARG and sets *n_invalid (may be NULL) when codes are not +-1 / labels not 0-1. */
int b200_maphashing_host(const float *q_codes, const float *q_labels, const float *db_codes, const float *db_labels,
                         int Q, long long N, int B, int L, int label_mode, long long k, double *ap_out,
                         uint32_t *tsum_out, double *map_out, int *n_invalid);

/* b200_maphashing_host for a caller that already holds PACKED codes / labels (b200_pack_* layout, Q x CW and N x CW
 * words, no padding row needed) in host memory: 24-48 bytes per row cross PCIe instead of 4 (B + L). */
int b200_maphashing_host_packed(const uint64_t *q_codes, const uint64_t *q_labels, const uint64_t *db_codes,
                                const uint64_t *db_labels, int Q, long long N, int B, int LW, int label_mode, long long k,
                                double *ap_out, uint32_t *tsum_out, double *map_out);

#ifdef __cplusplus
}
#endif
#endif /* B200RET_H_ */
