/* pope_b200.h -- C ABI of libpope_b200.so: the B200-native (sm_100a) Matcher hot path of karltan0328/POPE.
 *
 * The reference is 100 % Python/PyTorch and has no FFI of its own; each entry point below replaces the
 * PyTorch op sequence of one reference function (paths relative to the reference tree) and is what a
 * ctypes binding from the reference side calls (see INTEGRATION.md):
 *
 *   pope_coarse_match   <- CoarseMatching.forward + get_coarse_match
 *                          src/matcher/utils/coarse_matching.py:87-148, :150-261 (helpers :8-25)
 *   pope_fine_gather    <- FinePreprocess.forward, unfold + gather part
 *                          src/matcher/loftr_module/fine_preprocess.py:29-47
 *   pope_fine_match     <- FineMatching.forward + get_fine_match
 *                          src/matcher/utils/fine_matching.py:15-74
 *   pope_fine_match_maps <- the two above back to back (fine_preprocess.py:40-47 + fine_matching.py:15-74), fused
 *   pope_cosine_topk    <- F.cosine_similarity + running top-3 of the crop-retrieval loop
 *                          eval_linemod_json.py:72-101 (token: segment_anything/segment_anything/dinov2_utils.py:106-111)
 *   pope_pipeline_* / pope_match_pairs_host <- the pair loop of the eval drivers, batched
 *                          eval_linemod_json.py:103-122 (Matcher.forward steps 3-5, src/matcher/matcher.py:71-79)
 *
 * Conventions
 *   - plain pointers and sizes only; every `const void*` / `void*` data pointer is a DEVICE pointer unless the
 *     function name ends in `_host`; `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *   - all buffers are caller-owned; the library keeps no global state, allocates nothing persistent and never
 *     synchronises the device (the `_host` driver synchronises its own streams before returning).
 *   - return value: 0 = ok; < 0 = argument error (pope_status_t); > 0 = a cudaError_t from a launch/copy.
 *   - dtype: element type of the feature tensors (POPE_F32 or POPE_BF16).  All softmax / expectation arithmetic
 *     is fp32 regardless; ids are int64, coordinates and confidences fp32, exactly as the reference emits them.
 *   - there is no CPU fallback: on a machine without an sm_100 device every compute entry point returns a
 *     cudaError_t.
 */
#ifndef POPE_B200_H_
#define POPE_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define POPE_B200_ABI_VERSION 1

typedef enum {
  POPE_OK = 0,
  POPE_ERR_INVALID_ARG = -1,   /* null pointer, non-positive size, thr outside (0,1], ... */
  POPE_ERR_DTYPE = -2,         /* dtype not POPE_F32 / POPE_BF16 */
  POPE_ERR_WORKSPACE = -3,     /* workspace smaller than pope_coarse_workspace_bytes() */
  POPE_ERR_SHAPE = -4,         /* shape not supported by the requested implementation */
  POPE_ERR_ALIGNMENT = -5,     /* pointer / stride not aligned as documented */
  POPE_ERR_CAPACITY = -6,      /* output capacity smaller than n_pairs * min(L, S) */
  POPE_ERR_IO = -7             /* a file could not be created / written (points_io) */
} pope_status_t;

typedef enum { POPE_F32 = 0, POPE_BF16 = 1 } pope_dtype_t;

/* which coarse kernel family runs: AUTO picks TCGEN05 for bf16 (and, given the _ex workspace, fp32) features with
 * C % 64 == 0 && C <= 256, else SIMT (fp32 FMA) */
typedef enum { POPE_COARSE_AUTO = 0, POPE_COARSE_SIMT = 1, POPE_COARSE_TCGEN05 = 2 } pope_coarse_impl_t;

/* bits of counts[n_pairs + 1] written by pope_coarse_match */
#define POPE_FLAG_NONFINITE_LSE 1u   /* a row/column log-sum-exp was inf/nan (inputs contain inf/nan) */
#define POPE_FLAG_CAND_OVERFLOW 2u   /* a row had more above-threshold cells than 1/thr allows (inputs contain nan) */
#define POPE_FLAG_ROBUST_PATH   4u   /* informational: in some pair the single-sweep tcgen05 kernel found rows (or columns) whose
                                        maxima lie more than ~186 log2 units below the strongest cell of their 32-row group
                                        (one lazily raised shift per group cannot hold both in fp32), or inf / nan; the flagged
                                        pairs were recomputed by the two-sweep online-softmax kernels; results are valid */

#define POPE_FLAG_CAPACITY      8u   /* more matches than `capacity` (possible only for L > S, when several rows tie bit for bit
                                        on one column): the lists hold the first `capacity` matches, counts[n_pairs] = capacity */

int pope_abi_version(void);
const char* pope_status_string(int status);

/* Which kernel family POPE_COARSE_AUTO resolves to for this problem: POPE_COARSE_SIMT or POPE_COARSE_TCGEN05. */
int pope_coarse_auto_impl(int dtype, int L, int S, int C);

/* Bytes of device scratch pope_coarse_match needs for this problem (row/col log-sum-exp + best-candidate keys). */
size_t pope_coarse_workspace_bytes(int n_pairs, int L, int S);
/* The same plus, for POPE_F32 features with C % 64 == 0 && C <= 256, room for the three bf16 planes of every feature
 * value that the tensor-core path for fp32 inputs works on (fp32 accuracy: a = a1 + a2 + a3, six products).  With a
 * workspace of this size POPE_COARSE_AUTO / POPE_COARSE_TCGEN05 run fp32 features on the tensor cores (thr > 0.15);
 * with the smaller one fp32 features run the fp32-FMA kernels. */
size_t pope_coarse_workspace_bytes_ex(int n_pairs, int L, int S, int C, int dtype);

/* Coarse matching for n_pairs independent image pairs.
 *   feat_c0 [n_pairs, L, C], feat_c1 [n_pairs, S, C]  contiguous, 16-byte aligned, L = h0c*w0c, S = h1c*w1c.
 *   conf(i,j) = softmax_i(S)*softmax_j(S),  S = <f0_i, f1_j> / (C * temperature); a match is a cell with
 *   conf > thr that is the maximum of its row and of its column (over the full matrix) and whose two cells are
 *   at least `border_rm` cells away from their grid borders.  The L x S matrix is never written to memory.
 *   pixel_scale = hw0_i[0] / hw0_c[0] (8 for the (8,2) backbone).
 * Outputs (capacity >= n_pairs * min(L,S) entries each), matches sorted by (pair, i):
 *   b_ids, i_ids, j_ids int64[capacity]; mconf float[capacity]; mkpts0_c, mkpts1_c float[capacity][2] (x, y);
 *   counts int32[n_pairs + 2]: matches per pair, then counts[n_pairs] = total M, counts[n_pairs+1] = POPE_FLAG_* bits.
 * Entries past M are left untouched. */
int pope_coarse_match(const void* feat_c0, const void* feat_c1, int dtype,
                      int n_pairs, int L, int S, int C,
                      int h0c, int w0c, int h1c, int w1c,
                      float pixel_scale, float temperature, float thr, int border_rm, int impl,
                      void* workspace, size_t workspace_bytes,
                      int64_t* b_ids, int64_t* i_ids, int64_t* j_ids,
                      float* mconf, float* mkpts0_c, float* mkpts1_c,
                      int32_t* counts, int64_t capacity, void* stream);

/* Gather the W x W fine-level windows of every match from both fine feature maps (no unfold is materialised).
 *   feat_f0 / feat_f1: logical [n_pairs, Cf, Hf, Wf] with arbitrary element strides (sN, sC, sH, sW); the fast
 *   path is channels-last (sC == 1), plain NCHW works through a strided path.
 *   window element ww = ky*W + kx of coarse cell (y, x) = feat[b, :, stride*y - W/2 + ky, stride*x - W/2 + kx],
 *   zero outside the map; cell ids are row-major over a grid w0c (w1c) cells wide.
 *   m_dev: optional device int32 holding the live match count (e.g. counts + n_pairs); when non-NULL, `M` is the
 *   launch capacity and rows >= *m_dev are not touched, so no host sync is needed between coarse and fine.
 * Outputs win0, win1: [M, W*W, Cf] contiguous, same dtype as the maps. */
int pope_fine_gather(const void* feat_f0, const void* feat_f1, int dtype, int n_pairs, int Cf,
                     int Hf0, int Wf0, const int64_t strides0[4],
                     int Hf1, int Wf1, const int64_t strides1[4],
                     int w0c, int w1c, int stride, int W,
                     const int64_t* b_ids, const int64_t* i_ids, const int64_t* j_ids,
                     int64_t M, const int32_t* m_dev,
                     void* win0, void* win1, void* stream);

/* Fine matching: correlate the centre row of win0 with the WW rows of win1, softmax(./sqrt(Cf)), spatial
 * expectation and std over the normalised W x W grid, then mkpts1_f = mkpts1_c + expec_xy * coord_scale with
 * coord_scale = (W/2) * hw0_i[0]/hw0_f[0].
 *   win0, win1 [M, WW, Cf] contiguous, 16-byte aligned, Cf == 128, WW == 25 (W == 5).
 * Outputs expec_f float[M][3] = (E[x], E[y], std_x + std_y), mkpts1_f float[M][2]. */
int pope_fine_match(const void* win0, const void* win1, int dtype, int64_t M, const int32_t* m_dev,
                    int WW, int Cf, const float* mkpts1_c, float coord_scale,
                    float* expec_f, float* mkpts1_f, void* stream);

/* Fused form of pope_fine_gather + pope_fine_match for pipelines that run nothing between the two (the hot-path-only
 * pipeline; inside Matcher.forward the fine transformer sits between them and the two-call form is used): the centre
 * pixel of window 0 and the W*W pixels of window 1 are read straight from the CHANNELS-LAST maps (strides[1] == 1,
 * else POPE_ERR_SHAPE), the windows are never written.  `order` (may be NULL) = processing order from
 * pope_match_order_by_ref.  Same results as the two calls up to fp32 summation order.
 * Cf == 128, W == 5. */
int pope_fine_match_maps(const void* feat_f0, const void* feat_f1, int dtype, int n_pairs, int Cf,
                         int Hf0, int Wf0, const int64_t strides0[4],
                         int Hf1, int Wf1, const int64_t strides1[4],
                         int w0c, int w1c, int stride, int W,
                         const int64_t* b_ids, const int64_t* i_ids, const int64_t* j_ids,
                         int64_t M, const int32_t* m_dev, const int32_t* order,
                         const float* mkpts1_c, float coord_scale,
                         float* expec_f, float* mkpts1_f, void* stream);

/* Optional processing order for pope_fine_match_maps: order[k] = index of the k-th match when the matches of each
 * pair are sorted by their reference cell j (counting sort, one CTA per pair).  The coarse stage emits matches sorted by
 * (pair, i), whose reference cells are scattered over image 1; processed in (pair, j) order, neighbouring warps gather
 * adjacent / overlapping windows of the fine map.  Results are written at the match's own index, so outputs do not
 * depend on the order.  counts: the int32[n_pairs+2] array written by pope_coarse_match; order: int32[capacity]. */
int pope_match_order_by_ref(const int32_t* counts, int n_pairs, int S, const int64_t* j_ids, int32_t* order,
                            void* stream);

/* Retrieval: cosine similarity (x.y / (max(|x|,eps) * max(|y|,eps))) of one query token against R reference
 * tokens, followed by the eval loop's slot-replacement top-k (slots start at 0; a score greater than any slot
 * overwrites the first arg-min slot), evaluated in reference order so slot order matches the loop.
 *   q [D], refs [R, D] contiguous, k <= 16.  Outputs scores float[R], slot_scores float[k], slot_idx int32[k] (-1 = empty). */
int pope_cosine_topk(const void* q, const void* refs, int dtype, int R, int D, int k, float eps,
                     float* scores, float* slot_scores, int32_t* slot_idx, void* stream);

/* The running top-k of the retrieval loop alone (eval_linemod_json.py:95-101) over R scores that are already on the device, in
 * crop order -- the last step of a retrieval whose crops were scored on several GPUs (each rank scores its shard with
 * pope_cosine_topk, the R scores are all-gathered in crop order, every rank runs this; the slot contents depend on the whole
 * arrival order, so they cannot be merged from per-shard top-k lists).  Outputs as pope_cosine_topk. */
int pope_running_topk(const float* scores, int R, int k, float* slot_scores, int32_t* slot_idx, void* stream);

/* Pair-batching driver with HOST buffers (the end-to-end entry point): coarse match -> window gather -> fine
 * match for n_pairs pairs, processed in chunks of `chunk_pairs` with host->device copies, kernels and
 * device->host copies overlapped on three internal streams (double-buffered device slots).
 * A pipeline is an opaque handle that owns the device slots and streams for one geometry; it is the only object
 * the library ever allocates and it is not shared between host threads.
 *   Inputs  : feat_c0 [n,L,C], feat_c1 [n,S,C]; feat_f0 [n,Hf0,Wf0,Cf], feat_f1 [n,Hf1,Wf1,Cf] (channels-last),
 *             Hf = fine_stride*h_c, Wf = fine_stride*w_c.  Host buffers should be page-locked for full PCIe speed;
 *             page-locked fine maps are not copied whole: the fine kernel reads the centre pixel of every matched cell of
 *             image 0 in place over the host link, and of image 1's map only the union of the matched cells' 5x5 windows is
 *             fetched (every needed pixel once) into the device slot (pageable maps are copied in bulk; POPE_PIPELINE_F1 =
 *             union | windows | bulk in the environment selects the form for image 1, see pope_pipeline_last_f1_mode;
 *             POPE_PIPELINE_WINDOWS_IN_PLACE=0 is the older spelling of bulk).  With a fine level attached
 *             (pope_pipeline_set_fine_level) the fine transformer needs all 25 pixels of image 0's windows, so image 0's
 *             map reaches the device in the same form as image 1's (a pageable image-0 buffer is copied whole).  With a
 *             coarse level attached (pope_pipeline_set_coarse_level) feat_c0 / feat_c1 are the backbone's fp32 maps
 *             [n,C,h0c,w0c] / [n,C,h1c,w1c] instead, whatever the pipeline's dtype.
 *   Outputs : per-pair slots of cap = min(L,S) entries: i_ids, j_ids int64[n][cap]; mconf float[n][cap];
 *             mkpts0_f, mkpts1_f float[n][cap][2]; counts int32[n]; flags (optional, may be NULL) int32[1] = OR of the
 *             POPE_FLAG_* bits of all chunks.  pope_pipeline_run returns after every copy has landed. */
typedef struct pope_pipeline pope_pipeline_t;

int pope_pipeline_create(pope_pipeline_t** out, int device, int dtype, int chunk_pairs, int C, int Cf,
                         int h0c, int w0c, int h1c, int w1c, int fine_stride, int W,
                         float pixel_scale, float fine_scale /* hw0_i[0]/hw0_f[0] */,
                         float temperature, float thr, int border_rm, int impl);
int pope_pipeline_run(pope_pipeline_t* pl, const void* feat_c0, const void* feat_c1, const void* feat_f0,
                      const void* feat_f1, int n_pairs,
                      int64_t* i_ids, int64_t* j_ids, float* mconf, float* mkpts0_f, float* mkpts1_f,
                      int32_t* counts, int32_t* flags);
int pope_pipeline_destroy(pope_pipeline_t* pl);
/* Bytes that crossed the host link towards the device during the last pope_pipeline_run: the bulk copies plus what the
 * kernels read from page-locked fine maps.  Without a fine level that is, of image 0, the centre pixel of every matched
 * cell (one Cf-vector per match: the rest of image 0's map is not needed and is not transferred), and of image 1 the union
 * of the windows (union form) or every window whole (windows form).  With a fine level image 0 is counted like image 1:
 * the pixels of its windows' union, M x 25 Cf-vectors, or the whole map. */
int64_t pope_pipeline_last_h2d_bytes(const pope_pipeline_t* pl);
/* How image 1's fine map reached the device in the last pope_pipeline_run: 0 = whole map copied (pageable buffer, or
 * POPE_PIPELINE_F1=bulk), 1 = the kernels read every match's 5x5 window in place (POPE_PIPELINE_F1=windows), 2 = the
 * union of the matched cells' windows was fetched once per pixel into the device map (POPE_PIPELINE_F1=union); -1 for a
 * null handle.  With a fine level image 0 took the same form unless its buffer is pageable.  No counterpart in the
 * reference (its loop copies whole images, eval_linemod_json.py:103-122). */
int pope_pipeline_last_f1_mode(const pope_pipeline_t* pl);
/* Attach the bf16 fine level (FinePreprocess Linears + fine transformer) to a pipeline: from now on every chunk runs
 * coarse match -> window gather -> [merge_feat/down_proj] -> n_layers encoder layers -> fine match, which is what
 * Matcher(config, fine_cuda_bf16=True) computes.  pre (may be NULL = fine_concat_coarse_feat off), layers: device
 * pointers in the packed layouts of pope_fine_merge_coarse / pope_fine_transformer below, 16-byte aligned, on the
 * pipeline's device, caller-owned and alive while the pipeline runs; layer_kinds[l] in {0 self, 1 cross}, copied.
 * Requires a POPE_BF16 pipeline with C == 256 (Cf == 128 and W == 5 are already required by pope_pipeline_create).
 * layers == NULL detaches the level again: the pipeline then runs exactly as one that never had it.
 * The first attach allocates, once per pipeline and shared by its two slots (everything that touches them runs on the one
 * compute stream), the windows win0 / win1 [chunk * min(L,S), 25, 128] bf16 and one fine scratch of
 * max(pope_fine_tf_workspace_bytes(chunk * min(L,S), 25), pope_fine_merge_workspace_bytes(chunk * min(L,S))) bytes;
 * pope_pipeline_destroy frees them.  At 16 pairs x 480x640 per chunk (76 800 windows) that is 0.98 GB of windows plus
 * 2.5 GB of scratch (computed from the sizes).
 * Returns POPE_ERR_INVALID_ARG (null handle; layers without layer_kinds or with n_layers < 1; a kind other than 0 / 1),
 * POPE_ERR_DTYPE (fp32 pipeline), POPE_ERR_SHAPE (C != 256), POPE_ERR_ALIGNMENT, or a cudaError_t from an allocation.
 * pope_pipeline_set_fine_level(...) is pope_pipeline_set_fine_level_ex(pl, POPE_BF16, ...). */
int pope_pipeline_set_fine_level(pope_pipeline_t* pl, const void* pre, const void* layers, int n_layers,
                                 const int* layer_kinds);
/* pope_pipeline_set_fine_level for either packing: dtype (POPE_BF16 or POPE_F32) names the layouts pre and layers are packed
 * in and must be the pipeline's dtype, otherwise POPE_ERR_DTYPE.  On a POPE_F32 pipeline every chunk runs the
 * fp32-accuracy level (pope_fine_merge_coarse_f32_ex / pope_fine_transformer_f32_ex, packed layouts of
 * pope_fine_merge_coarse_f32 / pope_fine_transformer_f32), which is what Matcher(config, fine_cuda_fp32=True) computes; the
 * first attach then allocates fp32 windows win0 / win1 [chunk * min(L,S), 25, 128] and one fine scratch of
 * max(pope_fine_tf_f32_workspace_bytes(chunk * min(L,S), 25), pope_fine_merge_f32_workspace_bytes(chunk * min(L,S)))
 * bytes.  At 16 pairs x 480x640 per chunk (76 800 windows) that is 1.97 GB of windows plus 9.3 GB of scratch (computed
 * from the sizes).  Every form of the fine maps (union, windows, bulk) works with either level. */
int pope_pipeline_set_fine_level_ex(pope_pipeline_t* pl, int dtype, const void* pre, const void* layers, int n_layers,
                                    const int* layer_kinds);
/* Attach the coarse level (position encoding + coarse LoFTR transformer) to a pipeline, so that it starts where the
 * backbone stops: from now on pope_pipeline_run's feat_c0 / feat_c1 are the backbone's coarse maps, host fp32
 * [n, C, h0c, w0c] / [n, C, h1c, w1c] (contiguous) whatever the pipeline's dtype, and every chunk runs
 *   copy the maps (fp32) -> pope_coarse_pos_encode_ex (to the pipeline's dtype) -> pope_coarse_transformer[_f32] -> coarse
 *   match -> ... as before
 * which is what Matcher(config, coarse_cuda_bf16=True) (POPE_BF16) or coarse_cuda_fp32=True (POPE_F32) computes after
 * its backbone; the fine level, when attached, reads the transformed features.  The maps cross the link in fp32 (the
 * encoding is added in fp32 before any rounding), 4 bytes per element in pope_pipeline_last_h2d_bytes.
 * dtype names the packing of `layers` (pope_coarse_transformer / pope_coarse_transformer_f32 layouts) and must be the
 * pipeline's dtype (POPE_ERR_DTYPE); pe: the encoding's [C, pe_h, pe_w] fp32 buffer (4-byte aligned), layers (16-byte
 * aligned): device pointers on the pipeline's device, caller-owned and alive while the pipeline runs; layer_kinds[l] in
 * {0 self, 1 cross}, copied.  Requires C == 256 and both coarse grids within pe_h x pe_w (POPE_ERR_SHAPE).
 * layers == NULL detaches the level again: the pipeline then runs exactly as one that never had it.
 * The first attach allocates, per slot, an fp32 staging buffer for one chunk's maps (chunk * (L + S) * C * 4 bytes) and,
 * shared by both slots (it is touched on the compute stream only), one transformer scratch of
 * pope_coarse_tf_workspace_bytes(chunk, L, S) (bf16) or pope_coarse_tf_f32_workspace_bytes(chunk, L, S) (fp32) bytes;
 * pope_pipeline_destroy frees them.  Returns POPE_ERR_INVALID_ARG (null handle; layers without pe or layer_kinds, n_layers
 * < 1, a non-positive pe_h / pe_w, a kind other than 0 / 1), POPE_ERR_DTYPE, POPE_ERR_SHAPE, POPE_ERR_ALIGNMENT, or a
 * cudaError_t from an allocation. */
int pope_pipeline_set_coarse_level(pope_pipeline_t* pl, int dtype, const void* pe, int pe_h, int pe_w, const void* layers,
                                   int n_layers, const int* layer_kinds);

/* One-shot convenience: create + run + destroy. */
int pope_match_pairs_host(const void* feat_c0, const void* feat_c1, const void* feat_f0, const void* feat_f1,
                          int dtype, int n_pairs, int C, int Cf,
                          int h0c, int w0c, int h1c, int w1c, int fine_stride, int W,
                          float pixel_scale, float fine_scale, float temperature, float thr, int border_rm, int impl,
                          int chunk_pairs, int device,
                          int64_t* i_ids, int64_t* j_ids, float* mconf, float* mkpts0_f, float* mkpts1_f,
                          int32_t* counts, int32_t* flags);

/* Match-list consumer of the eval loop (eval_linemod_json.py:118-119 `np.where(confidences > 0.9)` per crop and :146
 * `np.argmax(matching_score)` per query; SURVEY.md 8(f) rank 3, selection part), without copying the lists to the host:
 *   scores[p] = #{matches of pair p with mconf > thr};  best[g] = first arg-max of scores over the `group` consecutive
 *   pairs [g*group, (g+1)*group) (one query image against its retrieved crops).
 * mconf / counts: as written by pope_coarse_match (counts int32[n_pairs+2]).  scores int32[n_pairs],
 * best int32[ceil(n_pairs / group)], both on the device. */
int pope_match_scores(const float* mconf, const int32_t* counts, int n_pairs, int group, float thr, int32_t* scores,
                      int32_t* best, void* stream);

/* Packs the live matches of one batch into 32-byte records (int32[8]: global pair index = b + pair_offset, i, j, mconf,
 * x0, y0, x1, y1; floats as bit patterns): the unit of the single cross-GPU gather of match lists (SURVEY.md 8(e)).
 * m_dev: device pointer to the live match count (counts + n_pairs of pope_coarse_match); records: int32[capacity * 8].
 * base_dev (may be NULL): device int64 holding the number of records already in `records`; the batch is appended behind
 * them (the caller advances the counter), so a job's records stay contiguous without a compaction pass. */
int pope_pack_records(const int64_t* b_ids, const int64_t* i_ids, const int64_t* j_ids, const float* mconf,
                      const float* mkpts0_f, const float* mkpts1_f, const int32_t* m_dev, int64_t capacity,
                      int pair_offset, int32_t* records, const int64_t* base_dev, void* stream);

/* The compact form of the same record, 20 bytes (int32[5]: global pair index, i | j << 16, mconf, x1, y1): the keypoint of
 * image 0 is implied by i (mkpts0_f = mkpts0_c = (i % w0c, i / w0c) * pixel_scale, fine_matching.py:66).  Needs
 * L, S <= 65536.  records: int32[capacity * 5]; the other arguments as pope_pack_records. */
int pope_pack_records_compact(const int64_t* b_ids, const int64_t* i_ids, const int64_t* j_ids, const float* mconf,
                              const float* mkpts1_f, const int32_t* m_dev, int64_t capacity, int pair_offset,
                              int32_t* records, const int64_t* base_dev, void* stream);

/* ---- batched relative pose from the match lists (SURVEY.md 8(f) rank 3) --------------------------------------------------
 * Replaces the per-pair `estimate_pose(kpts0, kpts1, K0, K1, thresh, conf)` of the reference (src/utils/metrics.py:69-94:
 * cv2.findEssentialMat(..., threshold, prob=conf, method=cv2.RANSAC) followed by cv2.recoverPose) for a whole batch of match
 * lists that are still on the device.  mkpts0 / mkpts1: float32 [capacity, 2] pixel coordinates, the matches of pair p at
 * rows [sum(counts[:p]), sum(counts[:p+1])) (the layout pope_fine_match_maps leaves; lists are clipped at `capacity`);
 * counts: int32 [n_pairs] (device);
 * K0 / K1: float64 [n_pairs, 9] intrinsics (device).  thresh is in pixels, conf the RANSAC confidence, max_iters
 * (<= POPE_POSE_MAX_ITERS; OpenCV's default is 1000) the iteration bound; seed selects the minimal samples (counter-based
 * hash, see csrc/pose_math.cuh).  Outputs (device): R float64 [n_pairs, 9], t float64 [n_pairs, 3] (unit norm), E float64
 * [n_pairs, 9], inliers uint8 [capacity] (the mask recoverPose returns: RANSAC inliers that pass the cheirality test),
 * n_inliers / status / iters int32 [n_pairs]; status 0 is the reference's `return None` (fewer than 5 matches, no model, or
 * no point in front of both cameras), iters the number of minimal samples the equivalent sequential loop consumed.
 * Results equal a sequential RANSAC over the same samples with OpenCV's adaptive iteration bound; they are deterministic in
 * (inputs, seed).  All arithmetic is float64.  Workspace: about 0.37 MB per pair plus 33 bytes per row of capacity.
 * n_pairs <= 65535 per call.  The call is stream-ordered without host synchronisation (CUDA-graph capturable). */
#define POPE_POSE_MAX_ITERS 1024
size_t pope_pose_workspace_bytes(int n_pairs, int64_t capacity);
int pope_estimate_pose_batch(const float* mkpts0, const float* mkpts1, const int32_t* counts, int n_pairs, int64_t capacity,
                             const double* K0, const double* K1, double thresh, double conf, int max_iters, uint64_t seed,
                             double* R, double* t, double* E, uint8_t* inliers, int32_t* n_inliers, int32_t* status,
                             int32_t* iters, void* workspace, size_t workspace_bytes, void* stream);

/* ---- on-disk match format (host code; SURVEY.md 8(f) rank 4) ------------------------------------------------------------
 * numpy.savetxt(path, a) as the reference uses it (linemod.py:168-171: '%.18e', one space between columns, '\n' after
 * every row; a 1-D array = one value per line = cols 1): byte-identical output, read back by pose/dataset.py with
 * numpy.loadtxt.  data: host memory, row-major [rows, cols]. */
int pope_savetxt_f32(const char* path, const float* data, int64_t rows, int cols);
int pope_savetxt_f64(const char* path, const double* data, int64_t rows, int cols);
/* All pairs of a batch at once, from the host pipeline's per-pair slots (pope_pipeline_run / pope_match_pairs_host:
 * mkpts0_f, mkpts1_f float32[n_pairs, capacity, 2], counts int32[n_pairs]): for every pair with at least min_matches
 * matches (the reference skips pairs with fewer than 5, linemod.py:143-146) writes <dir>/mkpts0/<names[p]>.txt and
 * <dir>/mkpts1/<names[p]>.txt on n_threads host threads (<= 0: all cores).  *written = number of pairs written. */
int pope_write_match_files(const char* dir, const char* const* names, int n_pairs, const float* mkpts0,
                           const float* mkpts1, const int32_t* counts, int64_t capacity, int min_matches, int n_threads,
                           int32_t* written);

/* numpy.loadtxt(path, delimiter=' ') as pose/dataset.py:75-101 reads those files back: values separated by blanks, one row
 * per line, '#' comments and empty lines skipped; values written with '%.18e' come back bit for bit.  out: host memory for
 * `capacity` values; *rows, *cols receive the shape (0, 0 for an empty file).  POPE_ERR_CAPACITY if the file holds more
 * values, POPE_ERR_SHAPE for ragged rows or a token that is not a number, POPE_ERR_IO if the file cannot be read. */
int pope_loadtxt_f64(const char* path, double* out, int64_t capacity, int64_t* rows, int* cols);
/* The inverse of pope_write_match_files: fills the per-pair slots mkpts0 / mkpts1 float32[n_pairs, capacity, 2] and counts
 * int32[n_pairs] from <dir>/mkpts0/<names[p]>.txt and <dir>/mkpts1/<names[p]>.txt on n_threads host threads; counts[p] = -1
 * where the pair has no files (pairs below min_matches were never written), lists longer than capacity are truncated. */
int pope_read_match_files(const char* dir, const char* const* names, int n_pairs, float* mkpts0, float* mkpts1,
                          int32_t* counts, int64_t capacity, int n_threads);

/* The two crops the reference stores beside the match files (linemod.py:172-173: cv2.imwrite(<dir>/img0/<pair>.png, crop)),
 * read back with cv2.imread (pose/dataset.py:102-103).  img: host memory, 8 bits per channel in OpenCV's order ([height,
 * width, channels] with channels = 1 grey, 3 BGR, 4 BGRA), `pitch` bytes between rows; level = zlib level 0..9 (OpenCV's
 * default is 1).  The file decodes to exactly the input pixels; its bytes are not libpng's (other filter choice). */
int pope_write_png(const char* path, const unsigned char* img, int height, int width, int channels, int64_t pitch, int level);
/* n densely packed images of possibly different sizes on n_threads host threads (<= 0: all cores). */
int pope_write_png_batch(const char* const* paths, const unsigned char* const* imgs, const int32_t* heights,
                         const int32_t* widths, int channels, int n, int level, int n_threads);

/* ---- fine-level transformer and FinePreprocess Linears (bf16; SURVEY.md 8(f) rank 1) ---------------------------------
 * Replace src/matcher/loftr_module/transformer.py:34-58,95-104 + linear_attention.py:21-47 (LocalFeatureTransformer with
 * d_model 128, 8 heads, 'linear' attention) and fine_preprocess.py:50-57 (down_proj / merge_feat) of the reference.
 *
 * Packed weights of ONE LoFTREncoderLayer, POPE_FINE_TF_LAYER_BYTES bytes, matrices bf16 row-major [out, in] exactly like
 * nn.Linear.weight, LayerNorm parameters fp32:
 *   +0       q_proj.weight | k_proj.weight | v_proj.weight   [384, 128]
 *   +98304   merge.weight                                    [128, 128]
 *   +131072  mlp.0.weight                                    [256, 256]
 *   +262144  mlp.2.weight                                    [128, 256]
 *   +327680  norm1.weight, norm1.bias, norm2.weight, norm2.bias   4 x [128] fp32
 * Packed FinePreprocess weights, POPE_FINE_PRE_BYTES bytes:
 *   +0       down_proj.weight [128, 256] bf16     +65536  merge_feat.weight [128, 256] bf16
 *   +131072  down_proj.bias [128] fp32            +131584 merge_feat.bias [128] fp32                                   */
#define POPE_FINE_TF_LAYER_BYTES 329728
#define POPE_FINE_PRE_BYTES 132096

/* Bytes of device scratch for m_windows windows of window_tokens tokens (5 activation planes of [m*tokens, 128] bf16). */
size_t pope_fine_tf_workspace_bytes(int64_t m_windows, int window_tokens);

/* feat0, feat1: [m_windows, window_tokens, 128] bf16, updated IN PLACE by n_layers encoder layers;
 * layer_kinds[l] = 0 ('self': each side attends to itself) or 1 ('cross': feat0 attends to feat1, then feat1 to the new
 * feat0), weights = n_layers consecutive packed layers.  Never synchronises; m_windows == 0 is a no-op. */
int pope_fine_transformer(void* feat0, void* feat1, int64_t m_windows, int window_tokens, const void* weights,
                          int n_layers, const int* layer_kinds, void* workspace, size_t workspace_bytes, void* stream);

/* pope_fine_transformer bounded by a live count kept on the device, so that it can follow pope_coarse_match /
 * pope_fine_gather without a host sync (and be captured in a CUDA graph).  m_windows is the launch capacity: tensor maps,
 * grids and the workspace are sized by it.  m_dev (may be NULL = all m_windows windows): device int32 live window count,
 * e.g. counts + n_pairs of pope_coarse_match; windows at or past min(*m_dev, m_windows) are never written and their
 * contents never reach a live window.  A live count of 0 is a no-op.  Same results as pope_fine_transformer on the live
 * windows, bit for bit.  pope_fine_transformer(...) is pope_fine_transformer_ex(..., m_dev = NULL, ...). */
int pope_fine_transformer_ex(void* feat0, void* feat1, int64_t m_windows, const int32_t* m_dev, int window_tokens,
                             const void* weights, int n_layers, const int* layer_kinds,
                             void* workspace, size_t workspace_bytes, void* stream);

/* Bytes of device scratch pope_fine_merge_coarse needs (gathered + projected coarse rows, per-window vectors). */
size_t pope_fine_merge_workspace_bytes(int64_t m_windows);

/* FinePreprocess' coarse-context mixing, IN PLACE on the gathered windows win0/win1 [m, window_tokens, 128] bf16:
 *   c = down_proj(cat(feat_c0[b_ids, i_ids], feat_c1[b_ids, j_ids]));  win = merge_feat(cat(win, repeat(c)))
 * feat_c0 [N, L, 256], feat_c1 [N, S, 256] bf16; ids are device int64 arrays of length m_windows. */
int pope_fine_merge_coarse(void* win0, void* win1, int64_t m_windows, int window_tokens, const void* feat_c0,
                           const void* feat_c1, int L, int S, int C, const int64_t* b_ids, const int64_t* i_ids,
                           const int64_t* j_ids, const void* weights, void* workspace, size_t workspace_bytes,
                           void* stream);

/* pope_fine_merge_coarse bounded by a live count kept on the device (the convention of pope_fine_transformer_ex):
 * m_windows is the capacity (length of the id arrays and of the windows, workspace sized by it), m_dev (may be NULL)
 * the device int32 live count; ids, windows and scratch rows at or past min(*m_dev, m_windows) are never read or written
 * (scratch: rows of either side).  Same results as pope_fine_merge_coarse on the live windows, bit for bit. */
int pope_fine_merge_coarse_ex(void* win0, void* win1, int64_t m_windows, const int32_t* m_dev, int window_tokens,
                              const void* feat_c0, const void* feat_c1, int L, int S, int C,
                              const int64_t* b_ids, const int64_t* i_ids, const int64_t* j_ids, const void* weights,
                              void* workspace, size_t workspace_bytes, void* stream);

/* ---- fine-level transformer and FinePreprocess Linears at fp32 accuracy -------------------------------------------------
 * The same layers on fp32 windows, computed on the bf16 tensor cores with every GEMM operand split into three bf16 terms
 * w = w1 + w2 + w3 (24 mantissa bits) and the six significant products accumulated in fp32; activations, the attention,
 * the LayerNorms, biases and residuals are fp32.  Results agree with the fp32 modules up to rounding.
 *
 * Packed weights: the bf16 layouts above with every matrix as three consecutive bf16 planes [plane][out][in] (w1 = bf16(w),
 * w2 = bf16(w - w1), w3 = bf16(w - w1 - w2), each residual exact in fp32) at 3x its bf16 offset, the fp32 tail unchanged.
 * ONE LoFTREncoderLayer, POPE_FINE_TF_F32_LAYER_BYTES bytes:
 *   +0       q_proj | k_proj | v_proj   3 planes of [384, 128]  (planes 98304 bytes apart)
 *   +294912  merge.weight               3 planes of [128, 128]  (32768 bytes apart)
 *   +393216  mlp.0.weight               3 planes of [256, 256]  (131072 bytes apart)
 *   +786432  mlp.2.weight               3 planes of [128, 256]  (65536 bytes apart)
 *   +983040  norm1.weight, norm1.bias, norm2.weight, norm2.bias   4 x [128] fp32
 * FinePreprocess, POPE_FINE_PRE_F32_BYTES bytes:
 *   +0       down_proj.weight  3 planes of [128, 256] (65536 bytes apart)
 *   +196608  merge_feat.weight 3 planes of [128, 256] (65536 bytes apart)
 *   +393216  down_proj.bias [128] fp32            +393728 merge_feat.bias [128] fp32                                   */
#define POPE_FINE_TF_F32_LAYER_BYTES 985088
#define POPE_FINE_PRE_F32_BYTES 394240

/* Bytes of device scratch of pope_fine_transformer_f32: 5 fp32 activation planes and 9 bf16 split planes of
 * [m_windows * window_tokens, 128], 4 864 bytes per token (19.8 GB at 162 812 windows of 25 tokens). */
size_t pope_fine_tf_f32_workspace_bytes(int64_t m_windows, int window_tokens);

/* pope_fine_transformer on fp32 windows [m_windows, window_tokens, 128] (contiguous, updated IN PLACE) with layers packed
 * as above.  Same arguments and error codes; pointers 16-byte aligned (POPE_ERR_ALIGNMENT), m_windows * window_tokens
 * below 2^31 - 128 (POPE_ERR_SHAPE).  Never synchronises; m_windows == 0 is a no-op; each window's output depends on that
 * window's inputs only, bit for bit. */
int pope_fine_transformer_f32(void* feat0, void* feat1, int64_t m_windows, int window_tokens, const void* weights,
                              int n_layers, const int* layer_kinds, void* workspace, size_t workspace_bytes, void* stream);

/* pope_fine_transformer_f32 bounded by a live count kept on the device (the convention of pope_fine_transformer_ex), so
 * that the fp32-accuracy level can follow pope_coarse_match / pope_fine_gather without a host sync (and be captured in a
 * CUDA graph).  m_windows is the launch capacity: tensor maps, grids and the workspace are sized by it.  m_dev (may be
 * NULL = all m_windows windows): device int32 live window count; windows, ids and scratch rows at or past
 * min(*m_dev, m_windows) are never read or written, and their contents never reach a live window.  A live count of 0
 * is a no-op.  Same results as pope_fine_transformer_f32 on the live windows, bit for bit, and the same error codes.
 * pope_fine_transformer_f32(...) is pope_fine_transformer_f32_ex(..., m_dev = NULL, ...). */
int pope_fine_transformer_f32_ex(void* feat0, void* feat1, int64_t m_windows, const int32_t* m_dev, int window_tokens,
                                 const void* weights, int n_layers, const int* layer_kinds,
                                 void* workspace, size_t workspace_bytes, void* stream);

/* Bytes of device scratch of pope_fine_merge_coarse_f32 (gathered and projected coarse rows with their split planes,
 * per-window vectors; 8 704 bytes per window, for any window size). */
size_t pope_fine_merge_f32_workspace_bytes(int64_t m_windows);

/* pope_fine_merge_coarse on fp32 windows win0/win1 [m, window_tokens, 128] and fp32 feat_c0 [N, L, 256] / feat_c1
 * [N, S, 256] with weights packed as above.  Same arguments and error codes; windows, coarse features, weights and
 * workspace 16-byte aligned (POPE_ERR_ALIGNMENT), m * window_tokens below 2^31 - 128 (POPE_ERR_SHAPE). */
int pope_fine_merge_coarse_f32(void* win0, void* win1, int64_t m_windows, int window_tokens, const void* feat_c0,
                               const void* feat_c1, int L, int S, int C, const int64_t* b_ids, const int64_t* i_ids,
                               const int64_t* j_ids, const void* weights, void* workspace, size_t workspace_bytes,
                               void* stream);

/* pope_fine_merge_coarse_f32 bounded by a live count kept on the device (the convention of pope_fine_transformer_ex):
 * m_windows is the capacity (length of the id arrays and of the windows, workspace sized by it), m_dev (may be NULL)
 * the device int32 live count; ids, windows and scratch rows at or past min(*m_dev, m_windows) are never read or written
 * (scratch: rows of either side).  Same results as pope_fine_merge_coarse_f32 on the live windows, bit for bit, and the
 * same error codes.  pope_fine_merge_coarse_f32(...) is pope_fine_merge_coarse_f32_ex(..., m_dev = NULL, ...). */
int pope_fine_merge_coarse_f32_ex(void* win0, void* win1, int64_t m_windows, const int32_t* m_dev, int window_tokens,
                                  const void* feat_c0, const void* feat_c1, int L, int S, int C,
                                  const int64_t* b_ids, const int64_t* i_ids, const int64_t* j_ids, const void* weights,
                                  void* workspace, size_t workspace_bytes, void* stream);

/* ---- coarse-level transformer (bf16) ----------------------------------------------------------------------------------
 * Replace src/matcher/matcher.py:57-58 (pos_encoding + rearrange to token-major) and transformer.py:34-58,95-104 +
 * linear_attention.py:21-47 for LocalFeatureTransformer(config['coarse']): d_model 256, 8 heads, 'linear' attention,
 * no masks.  The attention is global over each pair's source tokens.
 *
 * Packed weights of ONE d_model-256 LoFTREncoderLayer, POPE_COARSE_TF_LAYER_BYTES bytes, matrices bf16 row-major
 * [out, in] exactly like nn.Linear.weight, LayerNorm parameters fp32:
 *   +0        q_proj.weight | k_proj.weight | v_proj.weight   [768, 256]
 *   +393216   merge.weight                                    [256, 256]
 *   +524288   mlp.0.weight                                    [512, 512]
 *   +1048576  mlp.2.weight                                    [256, 512]
 *   +1310720  norm1.weight, norm1.bias, norm2.weight, norm2.bias   4 x [256] fp32                                       */
#define POPE_COARSE_TF_LAYER_BYTES 1314816

/* Bytes of device scratch for n_pairs pairs of L and S tokens (5 activation planes of [n_pairs * max(L, S), 256] bf16,
 * the attention's per-chunk partial sums and its reduced KV); 0 for a non-positive or too large shape. */
size_t pope_coarse_tf_workspace_bytes(int64_t n_pairs, int L, int S);

/* feat0: [n_pairs, L, 256], feat1: [n_pairs, S, 256] bf16, contiguous, updated IN PLACE by n_layers encoder layers;
 * layer_kinds[l] = 0 ('self') or 1 ('cross': feat0 attends to feat1, then feat1 to the new feat0), weights = n_layers
 * consecutive packed layers.  Pointers 16-byte aligned (POPE_ERR_ALIGNMENT).  n_pairs * max(L, S) must stay below 2^31
 * - 256 and n_pairs <= 65535 (POPE_ERR_SHAPE).  Argument errors return before any CUDA call; never synchronises,
 * allocates nothing; n_pairs == 0 is a no-op.  Each pair's output depends on that pair's inputs only, bit for bit. */
int pope_coarse_transformer(void* feat0, void* feat1, int64_t n_pairs, int L, int S, const void* weights, int n_layers,
                            const int* layer_kinds, void* workspace, size_t workspace_bytes, void* stream);

/* ---- coarse-level transformer at fp32 accuracy ------------------------------------------------------------------------
 * The same layers on fp32 features, computed on the bf16 tensor cores with every GEMM operand split into three bf16 terms
 * w = w1 + w2 + w3 (24 mantissa bits) and the six significant products accumulated in fp32; activations, the attention,
 * the LayerNorms and the residuals are fp32.  Results agree with the fp32 modules up to rounding.
 *
 * Packed weights of ONE layer, POPE_COARSE_TF_F32_LAYER_BYTES bytes: every matrix as three consecutive bf16 planes
 * [plane][out][in] (w1 = bf16(w), w2 = bf16(w - w1), w3 = bf16(w - w1 - w2), each residual exact in fp32), LayerNorm
 * parameters fp32:
 *   +0        q_proj | k_proj | v_proj   3 planes of [768, 256]  (planes 393216 bytes apart)
 *   +1179648  merge.weight               3 planes of [256, 256]  (131072 bytes apart)
 *   +1572864  mlp.0.weight               3 planes of [512, 512]  (524288 bytes apart)
 *   +3145728  mlp.2.weight               3 planes of [256, 512]  (262144 bytes apart)
 *   +3932160  norm1.weight, norm1.bias, norm2.weight, norm2.bias   4 x [256] fp32                                       */
#define POPE_COARSE_TF_F32_LAYER_BYTES 3936256

/* Bytes of device scratch of pope_coarse_transformer_f32 (5 fp32 activation planes and 9 bf16 split planes of
 * [n_pairs * max(L, S), 256], the attention's partial sums and reduced KV); 0 for a non-positive or too large shape. */
size_t pope_coarse_tf_f32_workspace_bytes(int64_t n_pairs, int L, int S);

/* pope_coarse_transformer on fp32 features [n_pairs, L, 256] / [n_pairs, S, 256] (contiguous, updated IN PLACE) with
 * weights packed as above.  Same argument checks, limits and guarantees as pope_coarse_transformer. */
int pope_coarse_transformer_f32(void* feat0, void* feat1, int64_t n_pairs, int L, int S, const void* weights, int n_layers,
                                const int* layer_kinds, void* workspace, size_t workspace_bytes, void* stream);

/* PositionEncodingSine + flatten(2).transpose(1, 2) + .to(bfloat16):
 *   out[b, y * W + x, c] = bf16(feat[b, c, y, x] + pe[c, y, x])      (fp32 sum, one round to nearest even)
 * feat: [n, C, H, W] fp32 contiguous (4-byte aligned), pe: the encoding's [C, pe_h, pe_w] fp32 buffer, out: [n, H * W, C]
 * bf16 (16-byte aligned).  C must be 256 and H <= pe_h, W <= pe_w (POPE_ERR_SHAPE); n == 0 is a no-op. */
int pope_coarse_pos_encode(const void* feat, const void* pe, int64_t n, int C, int H, int W, int pe_h, int pe_w, void* out,
                           void* stream);

/* pope_coarse_pos_encode with the output's element type: out_dtype = POPE_BF16 is pope_coarse_pos_encode itself;
 * out_dtype = POPE_F32 writes out [n, H * W, C] fp32 (16-byte aligned),
 *   out[b, y * W + x, c] = feat[b, c, y, x] + pe[c, y, x]      (one fp32 add, nothing rounded after it)
 * which is bit for bit `(feat + pe[..., :H, :W]).flatten(2).transpose(1, 2)` in torch: the token-major input of
 * pope_coarse_transformer_f32.  Any other out_dtype returns POPE_ERR_DTYPE; the other checks are those of
 * pope_coarse_pos_encode.  pope_coarse_pos_encode(...) is pope_coarse_pos_encode_ex(..., POPE_BF16, stream). */
int pope_coarse_pos_encode_ex(const void* feat, const void* pe, int64_t n, int C, int H, int W, int pe_h, int pe_w,
                              void* out, int out_dtype, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* POPE_B200_H_ */
