/* seam_b200.h -- C ABI of the B200-native SEAM Match-RCNN retrieval hot path.
 *
 * The reference (HumaticsLAB/SEAM-Match-RCNN) is pure Python and has no FFI; the boundary
 * it offers is its nn.Module surface and the evaluation scripts' score / rank outputs.
 * Each entry point below names the reference code it replaces (paths relative to the
 * reference root).  The Python host package binds these with ctypes and keeps the
 * reference's module signatures on top (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch tensors' data_ptr());
 *     the library never allocates or frees caller-visible memory.  The handle owns only the
 *     folded weights.
 *   - all calls enqueue work on `stream` (a cudaStream_t passed as void*) and return
 *     without synchronising the host.
 *   - return value: 0 = OK, otherwise a seam_status; text via seam_last_error().
 *   - no CPU fallback exists: without a CUDA device every compute call fails.
 *   - D = 256 channels (models/match_head.py:81), inter channels 128 (models/nlb.py:15-17).
 */
#ifndef SEAM_B200_H_
#define SEAM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct seam_handle seam_handle;

enum seam_status {
  SEAM_OK = 0,
  SEAM_ERR_BAD_ARG = 1,      /* null pointer, negative size, misaligned pointer */
  SEAM_ERR_UNSUPPORTED = 2,  /* outside the envelope: T > 64, k > 32, strides not 16-byte multiples */
  SEAM_ERR_CUDA = 3,         /* a CUDA runtime / driver call failed */
  SEAM_ERR_STATE = 4,        /* weights not loaded, workspace too small */
};

enum { SEAM_D = 256, SEAM_DI = 128, SEAM_MAX_T = 64, SEAM_MAX_K = 32, SEAM_MAX_WORLD = 8 };

/* ABI version of this header: bumped when an existing signature changes, not when an entry point is added. */
int seam_abi_version(void);

/* One handle per device.  Not thread-safe; distinct handles are independent. */
int seam_create(seam_handle** out, int device);
void seam_destroy(seam_handle* h);
const char* seam_last_error(const seam_handle* h);
/* Number of kernels this handle has launched since creation (bench.py's gpu_launches). */
uint64_t seam_launch_count(const seam_handle* h);

/* Diagnostics.  Every blocking wait inside the kernels carries a wall-clock watchdog: instead of hanging
 * the GPU, a protocol error traps the launch after leaving a record {tag, blockIdx.x, threadIdx.x, barrier
 * shared address, parity, 0, 0, 0} in host-mapped memory.  Copies up to max_records records of 8 words into
 * out and returns their number (0 in normal operation); works after the context has been lost. */
int seam_watchdog_read(const seam_handle* h, uint32_t* out, int max_records);

/* Writes the device's nanosecond timer (%globaltimer) to *dst (device memory) when the stream gets there: a one-thread
 * kernel, graph-capturable -- how bench.py times a sharded step BETWEEN graph nodes (CUDA events cannot be recorded
 * inside a replayed graph), after the node that aligns the ranks. */
int seam_device_stamp(seam_handle* h, uint64_t* dst, void* stream);

/* Per-kernel device timing for bench.py's roofline: while enabled, the library brackets each
 * of its named kernels with CUDA events on the launching stream.  seam_profile_read waits
 * for the recorded events of one kernel, returns their summed duration and count, and
 * forgets them. */
enum seam_kernel {
  SEAM_KERNEL_AGGREGATE = 0,    /* K1a aggregate_kernel */
  SEAM_KERNEL_NLB_GEMM = 1,     /* K1b */
  SEAM_KERNEL_PREP_QUERIES = 2,
  SEAM_KERNEL_SCORE = 3,        /* K2 score_topk_kernel (tcgen05) */
  SEAM_KERNEL_RESCORE = 4,      /* K3b */
  SEAM_KERNEL_EXACT = 5,        /* K3c exhaustive path */
  SEAM_KERNEL_PREP_GALLERY = 6,
  SEAM_KERNEL_MERGE = 7,        /* merge_topk_kernel / merge_sharded_kernel */
  SEAM_KERNEL_TOWER = 8,        /* the whole conv tower (layout pass + 4 conv3x3_kernel + pool/linear/BN) */
};
int seam_profile_enable(seam_handle* h, int enable);
int seam_profile_read(seam_handle* h, int kernel, double* total_ms, int* launches);

/* Hot-path weights, fp32, device pointers, in the reference's state_dict layout
 * (TemporalAggregationNLB().state_dict(); SURVEY.md section 8(b)):
 *   newnlb.{theta,phi,g}.weight (128,256,1) / .bias (128)      models/nlb.py:34,51,54
 *   newnlb.W.weight (256,128,1) / .bias (256)                  models/nlb.py:45-49
 *   newnlb.concat_project.0.weight (1,256,1,1)                 models/nlb.py:57-60
 *   attention_scorer.weight (1,256) / .bias (1)                models/match_head.py:86
 *   last.weight (2,256) / .bias (2)                            models/match_head.py:64   */
typedef struct seam_weights {
  const float* theta_w; const float* theta_b;
  const float* phi_w;   const float* phi_b;
  const float* g_w;     const float* g_b;
  const float* W_w;     const float* W_b;
  const float* concat_w;
  const float* att_w;   const float* att_b;
  const float* last_w;  const float* last_b;
} seam_weights;

/* Folds the weights on the device into the collapsed form the kernels use (DESIGN.md "K1
 * algebra").  Replaces nothing at run time in the reference -- it is what
 * nn.Module.load_state_dict (evaluate_movingfashion.py:502-503) becomes. */
int seam_load_weights(seam_handle* h, const seam_weights* w, void* stream);

/* Only `last` (match_predictor.last, models/match_head.py:64): enough for the scorer entry
 * points when no aggregation is needed (per-frame scorers, evaluate_movingfashion.py:94-121). */
int seam_load_scorer(seam_handle* h, const float* last_w, const float* last_b, void* stream);

/* ---- (a) temporal aggregation ------------------------------------------------------
 * Replaces the seq-branch of TemporalAggregationNLB.forward, models/match_head.py:133-154:
 * per-track unpack (first True of the mask row ends the track, row 0 is a dummy),
 * NONLocalBlock1D when T_i > 1 (models/nlb.py:66-101), attention_scorer + softmax over
 * frames + weighted sum.
 *   seq          (1+Tmax, Q, 256) fp32 addressed as seq[t*frame_stride + i*track_stride + c]
 *                (strides in floats, multiples of 4; the reference layout is
 *                frame_stride = Q*256, track_stride = 256)
 *   mask         (Q, 1+Tmax) uint8 (torch.bool), nonzero = padding; may be NULL
 *   lens         (Q) int32 frames per track (overrides mask when non-NULL); may be NULL;
 *                both NULL means every track has Tmax frames
 *   out          (Q, 256) fp32  = x3_1b
 *   att          (Q, Tmax) fp32 attention weights p (zero beyond T_i), or NULL  (getatt=True)
 *   workspace    seam_aggregate_workspace_bytes(Q) bytes, 256-byte aligned              */
size_t seam_aggregate_workspace_bytes(int Q);
int seam_aggregate(seam_handle* h, const float* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                   int64_t frame_stride, int64_t track_stride, float* out, float* att, void* workspace,
                   size_t workspace_bytes, void* stream);
/* seam_aggregate for fp16 tracks: seq (1+Tmax, Q, 256) holds IEEE fp16 bit patterns (the dtype torch.autocast
 * and the reference's host-side feature store, evaluate_movingfashion.py:82-92, produce), strides in fp16
 * elements and multiples of 8 (16 bytes), seq 16-byte aligned; otherwise SEAM_ERR_UNSUPPORTED.  The kernel
 * widens each frame to fp32 as it leaves shared memory (exact) and runs the fp32 arithmetic from there on:
 * out / att are bit-identical to seam_aggregate on the widened tracks, for half the bytes read.  Same outputs
 * (fp32) and workspace as seam_aggregate. */
int seam_aggregate_f16(seam_handle* h, const void* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                       int64_t frame_stride, int64_t track_stride, float* out, float* att, void* workspace,
                       size_t workspace_bytes, void* stream);

/* Full non-local block output (not pooled): NONLocalBlock1D.forward, models/nlb.py:66-101.
 *   x, z  (B, 256, T) fp32 channel-major as in the reference; T <= 64.
 *   workspace  seam_nlb_workspace_bytes(B, T) bytes                                        */
size_t seam_nlb_workspace_bytes(int B, int T);
int seam_nlb_forward(seam_handle* h, const float* x, int B, int T, float* z, void* workspace,
                     size_t workspace_bytes, void* stream);

/* ---- (b)+(c) pair scorer and per-query top-k ----------------------------------------
 * Gallery preparation (once per gallery shard): fp16 copy for the tensor-core pass, the
 * per-item term cg_j = sum_k dw_k g_jk^2 (dw = last.weight[1]-last.weight[0]) and
 * gstat[0] = max_j ||g_j||_2.  g (G,256) fp32 -> g16 (G,256) fp16, cg (G) fp32, gstat (4) fp32. */
int seam_prepare_gallery(seam_handle* h, const float* g, int G, void* g16, float* cg, float* gstat, void* stream);
/* Preparation of an fp16 gallery (the dtype the reference's shop-descriptor store, evaluate_movingfashion.py:82-92, and
 * torch.autocast produce): g16 (G,256) fp16, 256 contiguous halves per row, 16-byte aligned (otherwise
 * SEAM_ERR_UNSUPPORTED), is read only -- it IS the tensor-core operand, and the direct form reads it as the gallery rows,
 * so neither an fp32 copy nor a second fp16 copy exists (516 instead of 1,540 bytes per prepared row).  Writes cg and
 * gstat, bit-identical to seam_prepare_gallery of the widened rows (overflow flag included).  A gallery prepared this
 * way is scored through the _g16 entry points below. */
int seam_prepare_gallery_f16(seam_handle* h, const void* g16, int G, float* cg, float* gstat, void* stream);

/* Fused scorer + top-k.  Replaces, for all queries at once, the per-query loop body
 * evaluate_movingfashion.py:263-269 (evaluate_multiDF2.py:220-226):
 *   sq_diffs = (gallery - q)**2 ; raw = sq_diffs @ W.T + b ; softmax[...,1] ; argsort desc
 * and the module tail models/match_head.py:160-162 without materialising x4 / x5.
 *   q (Q,256) fp32 queries; g (G,256) fp32 gallery shard with its prepared g16 / cg / gstat
 *   out_score  (Q,k) fp32  softmax(x5)[...,1] of the k best, best first
 *   out_margin (Q,k) fp32  l1 - l0 of the same entries (ranking key; does not saturate)
 *   out_idx    (Q,k) int32 gallery row + index_offset, -1 where G < k
 * Ordering: margin descending, ties by lowest index.  Results are those of the fp32
 * direct form; the fp16 tensor-core pass only nominates candidates, every returned entry is
 * re-scored in fp32 and rows whose candidate set cannot be proven complete are re-ranked
 * exhaustively (DESIGN.md "certified top-k").  k <= SEAM_MAX_K.
 *   stats      optional (4) int32: [0] = rows that took the exhaustive path               */
size_t seam_score_workspace_bytes(const seam_handle* h, int Q, int G, int k);
/* Introspection: how seam_score_topk decomposes a (Q,G) problem and lays out its workspace.
 * out[0] query tiles (128 rows), [1] gallery tiles (256 rows), [2] CTAs launched, [3] P = max
 * CTAs sharing one query tile's gallery sweep (each owns 4 candidate sub-lists per row),
 * [4] capacity of a sub-list (a power of two), [5..12] byte offsets of {a16, rq, anorm, thr,
 * rowcnt (Q,P,4), rowbuf (Q,P,4,cap; base rounded up to a multiple of cap*8), counters,
 * fallback_rows} in the workspace, [13] workspace bytes. */
int seam_score_plan(const seam_handle* h, int Q, int G, int64_t* out14);

/* Pure host logic, callable without a device: the work decomposition of the scorer for num_sms persistent
 * CTAs.  The (query tile, gallery tile) grid is linearised query-major; CTA b sweeps tiles
 * [bounds[b], bounds[b+1]) (bounds_len >= CTAs + 1 entries), ranges balanced by cost (tiles + sample tiles
 * + segment starts).  out6 = {query tiles, gallery tiles, CTAs, P, sub-list capacity, sample tiles per
 * sampled segment}.  rank_variant != 0: the decomposition seam_rank_of_target_prepared uses. */
int seam_score_partition(int num_sms, int Q, int G, int rank_variant, int32_t* bounds, int bounds_len, int32_t* out6);
int seam_score_topk(seam_handle* h, const float* q, int Q, const float* g, const void* g16, const float* cg,
                    const float* gstat, int G, int index_offset, int k, float* out_score, float* out_margin,
                    int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes, void* stream);
/* The _g16 entry points take an fp16 gallery: there is no g argument, the gallery IS g16 (prepared by
 * seam_prepare_gallery_f16) -- the tensor-core operand and the rows the fp32 direct form reads, widened exactly.  Results
 * are bit-identical to the fp32 entry on the widened gallery g16.float().  (Given the g16 that seam_prepare_gallery
 * made of an fp32 gallery, they score the rounded rows.)  g16 16-byte aligned with rows of 256 contiguous halves,
 * otherwise SEAM_ERR_UNSUPPORTED; everything else as the fp32 twin.
 * seam_score_topk for an fp16 gallery: */
int seam_score_topk_g16(seam_handle* h, const float* q, int Q, const void* g16, const float* cg, const float* gstat,
                        int G, int index_offset, int k, float* out_score, float* out_margin, int32_t* out_idx,
                        int32_t* stats, void* workspace, size_t workspace_bytes, void* stream);

/* seam_aggregate + seam_score_topk in one call: tracks in, descriptors (q_out (Q,256) = x3_1b) and per-query top-k
 * out -- the whole per-product loop body evaluate_movingfashion.py:252-277 for all products at once; same results as
 * the two calls.  (Writing the scorer's per-query operands from the aggregation kernel's read-back instead of the
 * prepare-queries pass was measured and dropped: the extra registers slowed the aggregation by more than the 6 us the
 * pass costs inside a graph -- DESIGN.md.)  workspace: seam_score_workspace_bytes(h, Q, G, k). */
int seam_search(seam_handle* h, const float* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                int64_t frame_stride, int64_t track_stride, float* q_out, const float* g, const void* g16, const float* cg,
                const float* gstat, int G, int index_offset, int k, float* out_score, float* out_margin, int32_t* out_idx,
                int32_t* stats, void* workspace, size_t workspace_bytes, void* stream);
/* seam_search for fp16 tracks (seq, strides and alignment as seam_aggregate_f16); everything else, q_out
 * included, as seam_search, and bit-identical to it on the widened tracks. */
int seam_search_f16(seam_handle* h, const void* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                    int64_t frame_stride, int64_t track_stride, float* q_out, const float* g, const void* g16,
                    const float* cg, const float* gstat, int G, int index_offset, int k, float* out_score,
                    float* out_margin, int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes,
                    void* stream);
/* seam_search / seam_search_f16 (fp32 / fp16 tracks) for an fp16 gallery (see seam_score_topk_g16). */
int seam_search_g16(seam_handle* h, const float* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                    int64_t frame_stride, int64_t track_stride, float* q_out, const void* g16, const float* cg,
                    const float* gstat, int G, int index_offset, int k, float* out_score, float* out_margin,
                    int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes, void* stream);
int seam_search_f16_g16(seam_handle* h, const void* seq, const uint8_t* mask, const int32_t* lens, int Tmax, int Q,
                        int64_t frame_stride, int64_t track_stride, float* q_out, const void* g16, const float* cg,
                        const float* gstat, int G, int index_offset, int k, float* out_score, float* out_margin,
                        int32_t* out_idx, int32_t* stats, void* workspace, size_t workspace_bytes, void* stream);

/* Dense logits (parity / small problems): x5 (Q,G,2) fp32 = last((q-g)^2).
 * models/match_head.py:160-162 and MatchPredictor.forward :70-74. */
int seam_score_dense(seam_handle* h, const float* q, int Q, const float* g, int G, float* x5, void* stream);

/* Class-1 probabilities softmax(x5)[...,1] as a dense (Q,G) fp32 matrix: compute_distances
 * (evaluate_movingfashion.py:101-106) and, with g = q, compute_selfdist (:115-121, the street x street matrix the
 * tracker thresholds).  Small problems only (the fused entries never materialise it). */
int seam_score_prob(seam_handle* h, const float* q, int Q, const float* g, int G, float* prob, void* stream);

/* "AVG & MAX DISTANCE" fusions of the eval script (evaluate_movingfashion.py:294-316) for all products at once: per
 * product the class-1 probabilities of its frames against every shop item are averaged / maximised over the frames
 * and the rank of the true item in the descending order (ties: lower index first) is returned -- without the
 * (frames x gallery) matrix ever existing, in the fp32 direct form.
 *   frames (N,256) fp32 SORTED BY PRODUCT; start (P+1) int32 CSR offsets into it; target (P) int32 shop row;
 *   rank_avg / rank_max (P) int32; products without frames get G. */
int seam_rank_fused_distances(seam_handle* h, const float* frames, const int32_t* start, int P, const float* g, int G,
                              const int32_t* target, int32_t* rank_avg, int32_t* rank_max, void* stream);

/* Rank of one designated gallery item per query (0 = best), the quantity the eval script
 * reads out of its full argsort: evaluate_movingfashion.py:268-269.
 *   target (Q) int32 gallery row;  out_rank (Q) int32;  out_margin (Q) fp32 optional   */
int seam_rank_of_target(seam_handle* h, const float* q, int Q, const float* g, int G, const int32_t* target,
                        int32_t* out_rank, float* out_margin, void* stream);

/* Same result as seam_rank_of_target (bit for bit: ranks are integers decided in the same fp32 direct
 * form) through the tensor cores, for a PREPARED gallery (seam_prepare_gallery): the tcgen05 pass counts
 * the items whose value exceeds the target's by more than the pass's error bound and nominates the items
 * inside the band, a resolve kernel decides those in fp32, rows it cannot certify are ranked exhaustively
 * (their number is returned in stats[0]).  This is the "rank = position in the full argsort" of
 * evaluate_movingfashion.py:268-269 / evaluate_multiDF2.py:225-226 for every query at once, without a sort.
 *   workspace: seam_rank_workspace_bytes(h, Q, G) bytes, 256-byte aligned; stats (4) int32 optional. */
size_t seam_rank_workspace_bytes(const seam_handle* h, int Q, int G);
int seam_rank_of_target_prepared(seam_handle* h, const float* q, int Q, const float* g, const void* g16,
                                 const float* cg, const float* gstat, int G, const int32_t* target, int32_t* out_rank,
                                 float* out_margin, int32_t* stats, void* workspace, size_t workspace_bytes,
                                 void* stream);
/* seam_rank_of_target_prepared for an fp16 gallery (see seam_score_topk_g16): same ranks and margins as the fp32 entry
 * on the widened gallery, its exhaustive fallback included. */
int seam_rank_of_target_prepared_g16(seam_handle* h, const float* q, int Q, const void* g16, const float* cg,
                                     const float* gstat, int G, const int32_t* target, int32_t* out_rank,
                                     float* out_margin, int32_t* stats, void* workspace, size_t workspace_bytes,
                                     void* stream);

/* Rank of the target over a gallery split into shards (one per GPU), exactly: for global target t,
 *   rank_i = sum over shards s of #{ j in s : (d_ij, j) ranks before (d_it, t) }   (ties by GLOBAL row).
 * Only the shard holding row t can compute d_it, so a sharded rank is three steps per shard:
 *   1. seam_shard_target_margin: out_margin (Q) fp32 = d_it where global row target[i] lies in
 *      [index_offset, index_offset + G), else -inf -- bit for bit the margin seam_rank_of_target[_prepared] reports;
 *   2. all-reduce MAX of the margins over the shards (every shard now holds every d_it);
 *   3. seam_shard_rank_count_prepared: out_count (Q) int32 = this shard's count against target_margin, by the
 *      tensor-core path of seam_rank_of_target_prepared on this shard's PREPARED rows (same workspace:
 *      seam_rank_workspace_bytes(h, Q, G)); queries it cannot certify on this shard are counted exhaustively here
 *      (their number in stats[0]);
 * then an all-reduce SUM of the counts gives the unsharded rank, integer for integer.
 *   target (Q) int32 GLOBAL gallery rows; index_offset >= 0 (else SEAM_ERR_BAD_ARG); target_margin must not be null
 *   (SEAM_ERR_BAD_ARG); Q == 0 is a no-op.  The _g16 forms take an fp16 shard (see seam_score_topk_g16), 16-byte
 *   aligned (else SEAM_ERR_UNSUPPORTED), and give the fp32 forms' results on the widened rows. */
int seam_shard_target_margin(seam_handle* h, const float* q, int Q, const float* g, int G, int index_offset,
                             const int32_t* target, float* out_margin, void* stream);
int seam_shard_target_margin_g16(seam_handle* h, const float* q, int Q, const void* g16, int G, int index_offset,
                                 const int32_t* target, float* out_margin, void* stream);
int seam_shard_rank_count_prepared(seam_handle* h, const float* q, int Q, const float* g, const void* g16,
                                   const float* cg, const float* gstat, int G, int index_offset, const int32_t* target,
                                   const float* target_margin, int32_t* out_count, int32_t* stats, void* workspace,
                                   size_t workspace_bytes, void* stream);
int seam_shard_rank_count_prepared_g16(seam_handle* h, const float* q, int Q, const void* g16, const float* cg,
                                       const float* gstat, int G, int index_offset, const int32_t* target,
                                       const float* target_margin, int32_t* out_count, int32_t* stats,
                                       void* workspace, size_t workspace_bytes, void* stream);

/* Merge N per-shard top-k lists (after the all-gather) into one: lists are (N,Q,k)
 * contiguous; entries with idx < 0 are invalid.  Same ordering contract as seam_score_topk.
 * No reference counterpart (the reference ranks a single gallery).  scores may be NULL: the score is
 * softmax(0, margin)[1], recomputed bit-identically, so shards need only exchange margins and indices. */
int seam_merge_topk(seam_handle* h, const float* scores, const float* margins, const int32_t* idx, int N, int Q,
                    int k, float* out_score, float* out_margin, int32_t* out_idx, void* stream);

/* ---- gallery-sharded search over the GPUs of one box (SURVEY.md section 8(e)) --------------------------
 * One process per GPU; rank r holds gallery rows [r G/N, (r+1) G/N) and OWNS queries [q_lo[r], q_lo[r+1]): it
 * aggregates their tracks and merges their per-shard top-k lists.  The kernels exchange data themselves: the
 * aggregation kernel stores every descriptor into the q_all buffer of every rank, the re-score kernels store a
 * query's list into the list buffer of its owner, the merge stores the merged rows into every rank's final
 * buffers -- plain stores into peer-mapped memory (NVLink / NVSwitch), ordered by flag words (release / acquire
 * at system scope), no collective call, no barrier kernel, no copy (csrc/exchange.cuh).  The reference has no
 * multi-GPU retrieval path; its torch.distributed use (stuffs/utils.py:340) is training-only.
 *
 * All pointers are DEVICE pointers valid on the calling rank; entry [r] of a table addresses rank r's buffer
 * (entry [rank] the local one).  The caller allocates them in peer-mapped memory (torch symmetric memory in the
 * Python host), zero-fills flags / done and sets *step = 1 once; the library advances *step.
 *   q_all        (2, Q, 256) fp32 per rank      descriptors, double-buffered by step parity
 *   list_margin  (2, world, own_max, k) fp32    lists for the queries the rank owns (own_max = largest ownership)
 *   list_idx     (2, world, own_max, k) int32
 *   final_*      (Q, k) per rank, or all NULL: then seam_sharded_merge writes the owner's rows to its out_* only
 *   flags        (3, SEAM_MAX_WORLD) uint32 per rank;  step (1), done (3) uint32, local to the rank            */
typedef struct seam_exchange {
  int32_t world, rank, Q, k, own_max;
  int32_t q_lo[SEAM_MAX_WORLD + 1];
  float* q_all[SEAM_MAX_WORLD];
  float* list_margin[SEAM_MAX_WORLD];
  int32_t* list_idx[SEAM_MAX_WORLD];
  float* final_score[SEAM_MAX_WORLD];
  float* final_margin[SEAM_MAX_WORLD];
  int32_t* final_idx[SEAM_MAX_WORLD];
  uint32_t* flags[SEAM_MAX_WORLD];
  uint32_t* step;
  uint32_t* done;
  /* optional (null: not used): the NVSwitch MULTICAST mapping of q_all -- one store to it lands in every rank's q_all
   * (the switch replicates it), so a rank's descriptors leave its GPU once instead of world - 1 times */
  float* q_all_mc;
  /* the same for the merged rows (all three or none) */
  float* final_score_mc;
  float* final_margin_mc;
  int32_t* final_idx_mc;
} seam_exchange;

/* sizeof(seam_exchange) as this library was built (device-free): a binding checks its own struct layout against it */
size_t seam_exchange_sizeof(void);

/* seam_aggregate for tracks [row0, row0 + Qlocal) of the step's Q queries (a rank may pass its tracks in several
 * calls, e.g. as they arrive from the host): descriptors go to rows row0.. of every rank's q_all; the call with
 * last != 0 tells the other ranks that this rank's descriptors are complete. */
int seam_sharded_aggregate(seam_handle* h, const seam_exchange* x, const float* seq, const uint8_t* mask,
                           const int32_t* lens, int Tmax, int Qlocal, int64_t frame_stride, int64_t track_stride,
                           int row0, int last, float* att, void* stream);
/* seam_sharded_aggregate for fp16 tracks (seq, strides and alignment as seam_aggregate_f16). */
int seam_sharded_aggregate_f16(seam_handle* h, const seam_exchange* x, const void* seq, const uint8_t* mask,
                               const int32_t* lens, int Tmax, int Qlocal, int64_t frame_stride, int64_t track_stride,
                               int row0, int last, float* att, void* stream);
/* seam_score_topk of all Q queries (this rank's q_all, once every rank's descriptors have landed) against the
 * rank's prepared gallery shard; the top-k rows go to the queries' owners.  Workspace as seam_score_topk. */
int seam_sharded_score_topk(seam_handle* h, const seam_exchange* x, const float* g, const void* g16, const float* cg,
                            const float* gstat, int G, int index_offset, int32_t* stats, void* workspace,
                            size_t workspace_bytes, void* stream);
/* seam_sharded_score_topk for an fp16 gallery shard (see seam_score_topk_g16). */
int seam_sharded_score_topk_g16(seam_handle* h, const seam_exchange* x, const void* g16, const float* cg,
                                const float* gstat, int G, int index_offset, int32_t* stats, void* workspace,
                                size_t workspace_bytes, void* stream);
/* Merges the world lists of the queries this rank owns and ends the step.  With final buffers in the exchange every
 * rank holds the complete (Q,k) result when its stream reaches the end of this call; without, out_* (own,k) receive
 * the owner's rows. */
int seam_sharded_merge(seam_handle* h, const seam_exchange* x, float* out_score, float* out_margin, int32_t* out_idx,
                       void* stream);

/* ---- backward of the hot path, for training (SURVEY.md section 8 f4) ---------------------------------------
 * The reference trains through the aggregator with autograd: its losses consume x5 of TemporalAggregationNLB's
 * x-branch (models/match_head.py:339, 429; stuffs/engine.py:158-185).  These entries give the vector-Jacobian
 * products the forward entries need to sit inside an autograd graph (the Python host wraps them in
 * torch.autograd.Function).  The forward kernels run on folded weights; the backward recomputes each track in the
 * reference's un-folded formulation (models/nlb.py:66-101, match_head.py:144-151) and differentiates that.
 *
 * seam_aggregate_backward: dout (Q,256) = d loss / d x3_1b  ->  dseq (1+Tmax,Q,256) contiguous fp32 = d loss / d
 * x3_1_seq (the caller zero-fills it: row 0 and padded frames stay zero) and the parameter gradients, ACCUMULATED
 * into the buffers of `grads` (same shapes as the weights; the caller zero-fills them).  Tracks of at most 16
 * frames (training uses about 10: train_movingfashion.py:165).  `w` holds the un-folded parameters (last_* unused). */
typedef struct seam_weight_grads {
  float* theta_w; float* theta_b;
  float* phi_w;   float* phi_b;
  float* g_w;     float* g_b;
  float* W_w;     float* W_b;
  float* concat_w;
  float* att_w;   float* att_b;
} seam_weight_grads;
int seam_aggregate_backward(seam_handle* h, const seam_weights* w, const float* seq, const uint8_t* mask,
                            const int32_t* lens, int Tmax, int Q, int64_t frame_stride, int64_t track_stride,
                            const float* dout, float* dseq, const seam_weight_grads* grads, void* stream);
/* Backward of seam_score_dense (x5 = last((q - g)^2), models/match_head.py:160-162): dx5 (Q,G,2) -> dq (Q,256),
 * dg (G,256) (overwritten) and dlast_w (2,256), dlast_b (2) (accumulated; the caller zero-fills them). */
int seam_score_dense_backward(seam_handle* h, const float* last_w, const float* q, int Q, const float* g, int G,
                              const float* dx5, float* dq, float* dg, float* dlast_w, float* dlast_b, void* stream);

/* ---- the match head's conv tower: ROI features -> 256-d embedding (SURVEY.md section 8 f3) ---------------
 * Replaces MatchPredictor's conv_seq / pool / linear in eval mode, models/match_head.py:50-62 as called at :67-69
 * and :93-95:   4 x [Conv2d 3x3 valid + ReLU] (256 -> 256 -> 256 -> 256 -> 1024 channels, 14 -> 6 spatial),
 * AvgPool2d(6) + ReLU, Linear(1024,256), BatchNorm1d(256) with its running statistics.
 * The convolutions run as shifted GEMMs on the tensor cores (tcgen05, fp16 operands, fp32 accumulation: the
 * precision class of the TF32 path cuDNN runs for the reference by default); results agree with the fp32 module
 * to ~2e-3 of the output scale (tests state 1e-2).
 *   conv_w[l] (Cout,256,3,3) fp32, conv_b[l] (Cout): conv_seq.{0,2,4,6}.{weight,bias}; lin_w (256,1024), lin_b (256):
 *   linear.0; bn_*: linear.1.{weight,bias,running_mean,running_var}, bn_eps its eps.  The handle keeps its own
 *   reorganised copy.
 *   x (K,256,14,14) fp32 NCHW (the RoIAlign output the reference feeds, models/video_matchrcnn.py roi_features);
 *   out: fp32 rows of 256; ROI i goes to row dst_row[i] (int64; NULL: row i) -- e.g. slot (1+t)*Q + track of the
 *   time-major x3_1_seq (models/match_head.py:101-111), so the aggregation kernel reads what this one wrote.
 *   workspace: seam_tower_workspace_bytes(K) bytes (about 330 KB per ROI), 1 KB aligned. */
int seam_tower_load_weights(seam_handle* h, const float* const* conv_w, const float* const* conv_b, const float* lin_w,
                            const float* lin_b, const float* bn_gamma, const float* bn_beta, const float* bn_mean,
                            const float* bn_var, float bn_eps, void* stream);
size_t seam_tower_workspace_bytes(int K);
int seam_tower_forward(seam_handle* h, const float* x, int K, float* out, const int64_t* dst_row, void* workspace,
                       size_t workspace_bytes, void* stream);

/* Host -> device upload of a slice of tracks, tracks [lo, hi) of a HOST x3_1_seq (1+Tmax, Q, 256) fp32
 * (the reference keeps every feature in host memory between the detector and the scorer,
 * evaluate_movingfashion.py:45-92, 253): one pitched asynchronous copy of the frame rows 1..Tmax into
 * the device tensor seq_dev (1+Tmax, hi-lo, 256); row 0 (the layout's dummy frame,
 * models/match_head.py:101-111) is neither read nor written.  Pinned host memory makes it asynchronous. */
int seam_upload_tracks(seam_handle* h, const float* seq_host, int Tmax, int Q, int lo, int hi, float* seq_dev,
                       void* stream);
/* seam_upload_tracks for an fp16 host x3_1_seq: the same single pitched copy with 512-byte rows into an fp16
 * device tensor (1+Tmax, hi-lo, 256) -- half the PCIe bytes; feed the result to the _f16 entry points. */
int seam_upload_tracks_f16(seam_handle* h, const void* seq_host, int Tmax, int Q, int lo, int hi, void* seq_dev,
                           void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SEAM_B200_H_ */
