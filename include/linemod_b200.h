/* linemod_b200.h -- C-ABI of the B200-native LINEMOD match + ICP pose-refinement path.
 *
 * This is the drop-in boundary: the entry points below are what a binding of the reference's
 * `linemodLevelup_pybind` module (reference: linemodLevelup/pybind11.cpp:7-35) binds instead of the
 * C++ classes `linemodLevelup::Detector` (linemodLevelup/linemodLevelup.h:264-375) and `poseRefine`
 * (linemodLevelup.h:8-19).  Plain pointers and sizes only; no torch / OpenCV types.  All calls are
 * blocking; one in-flight call per handle.  Every function returns 0 on success or a negative
 * LM_E_* code, with a human-readable message available from lm_last_error() (thread-local).
 * There is NO CPU fallback: without a CUDA device lm_create() fails.
 *
 * Citations "LL.cpp:n" = linemodLevelup/linemodLevelup.cpp of meiqua/6DPose @ 619be57.
 */
#ifndef LINEMOD_B200_H
#define LINEMOD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LM_OK 0
#define LM_E_INVALID (-1) /* bad argument / a CV_Assert of the reference would fire */
#define LM_E_CUDA (-2)    /* CUDA runtime error */
#define LM_E_STATE (-3)   /* call order (no bank / no frame uploaded) */
#define LM_E_CAPACITY (-4)

#define LM_MAX_LEVELS 4
#define LM_MAX_MODALITIES 2

typedef struct lm_detector lm_detector; /* replaces linemodLevelup::Detector, LL.h:264 */

/* One detection.  Replaces linemodLevelup::Match (LL.h:225-258); class_index indexes the class list
 * given to lm_load_bank (the host shim maps it back to the class_id string). */
typedef struct lm_match {
  int32_t x, y;
  float similarity;
  int32_t class_index;
  int32_t template_id;
} lm_match;

/* Pre-finish record of a candidate that survived refinement (LL.cpp:1855-1938), produced by the GPU
 * stages.  `work` indexes the matched-template sequence of this call (global across shards); `seq` is
 * the candidate's index in its shard's pre-sort order (template order, then ascending coarse cell;
 * LL.cpp:1797-1939).  Records are appended unordered; sorting by (work, seq) restores the reference's
 * pre-sort order.  16 bytes: the all-gather payload. */
typedef struct lm_record {
  int16_t x, y;
  float similarity;
  int32_t work;
  int32_t seq;
} lm_record;

/* A result block in device memory = this header followed by `capacity` lm_record slots. */
typedef struct lm_result_header {
  int32_t count;             /* records kept (may exceed capacity: only `capacity` were stored) */
  int32_t coarse_candidates; /* candidates that passed the coarse threshold (LL.cpp:1836-1852) */
  int32_t capacity;
  int32_t shard;
} lm_result_header;

const char* lm_last_error(void);

/* Detector(num_features, T) / Detector(T) / Detector(): LL.cpp:1663-1692.  `T` has n_levels entries
 * (sampling step per pyramid level).  `device` is the CUDA ordinal; -1 creates a host-only handle that
 * can hold a bank, compute selections / shard ranges and run lm_finish (the merge step of a multi-GPU
 * match) but refuses every GPU stage with LM_E_STATE. */
int lm_create(int device, int n_levels, const int* T, lm_detector** out);
void lm_destroy(lm_detector* d);

/* Replace the template bank (class_templates, LL.h:361-362).  Flattened:
 *   class_begin[n_classes+1]  global template ranges per class, in the caller's class order
 *   tmeta[G][n_slots][4]      {width, height, feat_begin, feat_count}; n_slots = n_levels*2, slot =
 *                             level*2 + modality (LL.cpp:1964)
 *   feats[n_feats][3]         {x, y, label} (struct Feature, LL.h:23-34)
 * Fails with LM_E_INVALID on label outside [0,8), negative coordinates, or > 8191 features in a
 * template (CV_Assert LL.cpp:1291). */
int lm_load_bank(lm_detector* d, int n_classes, const int32_t* class_begin, int n_slots, const int32_t* tmeta,
                 const int32_t* feats, int64_t n_feats);

/* Select which templates a call matches, in order: the concatenation of the given classes' template
 * ranges (Detector::match's class_ids loop, LL.cpp:1753-1769), then the slice [shard_index/shard_count)
 * of that sequence (contiguous, balanced by features x positions) -- the multi-GPU template shard.
 * n_classes_sel < 0 selects all classes in bank order. */
int lm_select(lm_detector* d, const int32_t* class_sel, int n_classes_sel, int shard_index, int shard_count);
/* Same with the shard layout chosen: LM_SHARD_CONTIGUOUS (lm_select's: one block of the sequence per shard) or
 * LM_SHARD_INTERLEAVED (shard r takes elements r, r + N, r + 2N, ...: neighbouring templates -- views and in-plane
 * variants that pass or fail together -- are dealt round the ranks, which evens out the candidate load).  Records
 * carry the global index in the selected sequence either way, so lm_finish is unchanged. */
#define LM_SHARD_CONTIGUOUS 0
#define LM_SHARD_INTERLEAVED 1
int lm_select_layout(lm_detector* d, const int32_t* class_sel, int n_classes_sel, int shard_index, int shard_count, int layout);
/* Index of this shard's first element inside the selected sequence and the shard's length (contiguous layout: the
 * shard is [begin, begin + count); interleaved: begin + k * shard_count, k < count). */
int lm_shard_range(lm_detector* d, int64_t* begin, int64_t* count);

/* Frame upload: quantized one-hot label images (output of QuantizedPyramid::quantize, LL.cpp:583-587,
 * 882-886) for every (level, modality), host pointers, index level*2+modality; rows/cols per level.
 * Fails where the reference asserts: rows%T, cols%T (LL.cpp:1217-1218), rows*cols%16 (LL.cpp:1136). */
int lm_upload_quantized(lm_detector* d, const uint8_t* const* quantized, const int* rows, const int* cols);

/* Same, but the label images already live in device memory (borrowed: they must stay valid and
 * unchanged until the stages enqueued on them have completed).  No copy is made. */
int lm_bind_quantized_device(lm_detector* d, const uint8_t* const* d_quantized, const int* rows, const int* cols);

/* Frame upload from the RAW images, quantization front-end on the GPU: rgb u8 rows x cols x 3, depth u16
 * rows x cols (mm), optional masks u8 rows x cols (255 = valid, NULL = none) -- the arguments of
 * Detector::match (LL.cpp:1702-1719).  Produces the same label images as the reference's
 * ColorGradientPyramid / DepthNormalPyramid (LL.cpp:350-505, 557-587, 729-886; parameters of
 * Detector(num_features, T): weak threshold 10, distance 2000 mm, difference 50 mm). */
int lm_upload_images(lm_detector* d, const uint8_t* rgb, const uint16_t* depth, int rows, int cols,
                     const uint8_t* mask_color, const uint8_t* mask_depth);

/* GPU stages on the uploaded frame: spread/response/linearize (LL.cpp:1094-1243), coarse similarity
 * scan + threshold (LL.cpp:1284-1354, 1836-1852), local 16x16 refinement up the pyramid
 * (LL.cpp:1366-1428, 1855-1938).  Leaves the ordered candidate records in device memory. */
int lm_run(lm_detector* d, float threshold);
/* lm_run split in two for pipelining: lm_enqueue issues every stage on the detector's stream and
 * returns without synchronising; lm_complete waits, and re-runs the refinement stage if the record
 * buffer was too small for the number of coarse candidates. */
int lm_enqueue(lm_detector* d, float threshold);
int lm_complete(lm_detector* d);
/* Everything lm_enqueue does lazily on a new bank / selection / frame size (feature addresses for the frame size,
 * shard work lists, run buffers), done now: the first lm_enqueue afterwards only launches.  Needs a frame uploaded or
 * bound (for its size).  SPMD callers use it so that no rank's first frame lags the others'. */
int lm_prepare(lm_detector* d);

/* Result block of the stages: by default an internal device buffer that grows on demand.  A caller
 * that wants the block in its own device memory (e.g. the send buffer of an NCCL all-gather) sets it
 * here; capacity is in records, the block is sizeof(lm_result_header) + capacity*sizeof(lm_record)
 * bytes.  d_block = NULL returns to the internal buffer. */
int lm_set_result_buffer(lm_detector* d, void* d_block, int64_t capacity_records);
int lm_device_result(lm_detector* d, void** d_block, int64_t* capacity_records);

/* Multi-GPU exchange fused into the refinement kernels (one process per GPU, template shards from
 * lm_select; the reference has no counterpart: its template loop is serial, LL.cpp:1797).  Every rank
 * owns an exchange buffer of 2 frame slots x `world` result blocks; once connected, the exact refinement
 * kernel (k_refine_bits / k_refine) stores every kept record into the block [slot][rank] of EVERY rank's buffer with peer stores over NVLink (local
 * stores for itself), its last CTA publishes the block header and a frame sequence flag, and a collector
 * kernel on the same stream waits for all `world` flags and packs the blocks into this handle's result
 * block.  lm_complete / lm_fetch_records / lm_device_result then see the kept records of ALL shards: no
 * separate collective, no host round trip between refinement and exchange.  All ranks must enqueue the
 * same frames in the same order (SPMD); capacity_records is per rank and per frame.  A collector that waits
 * longer than LINEMOD_B200_PEER_TIMEOUT_MS (default 1000) for a peer fails the frame (LM_E_STATE from
 * lm_complete) and raises a per-device abort flag every later collector honours at once; lm_peer_export
 * clears it.
 *   lm_peer_export        allocate the buffer, return its CUDA IPC handle (LM_PEER_HANDLE_BYTES bytes)
 *   lm_peer_connect       handles[world][LM_PEER_HANDLE_BYTES] of all ranks (own entry ignored)
 *   lm_peer_connect_local same, for handles living in ONE process: bases[world] from lm_peer_base
 *   lm_peer_disconnect    back to the single-GPU result block (callers barrier first) */
#define LM_PEER_HANDLE_BYTES 64
#define LM_MAX_PEERS 16
int lm_peer_export(lm_detector* d, int world, int64_t capacity_records, uint8_t* handle_out);
int lm_peer_base(lm_detector* d, void** base);
int lm_peer_connect(lm_detector* d, int rank, int world, const uint8_t* handles);
int lm_peer_connect_local(lm_detector* d, int rank, int world, void* const* bases);
int lm_peer_disconnect(lm_detector* d);

/* Copy the kept records of the last completed run to the host, sorted by (work, seq). */
int lm_fetch_records(lm_detector* d, lm_record* out, int64_t cap, int64_t* n_out);

/* Host finisher: order records by (work, seq), map work -> (class_index, template_id) for the current
 * selection (work indices are global in the selected sequence), then the reference's
 * std::sort + std::unique (LL.cpp:1772-1774).  `records` may be the concatenation of all shards'
 * records in any order. */
int lm_finish(lm_detector* d, const lm_record* records, int64_t n, lm_match* out, int64_t cap, int64_t* n_out);

/* Post-match stage on the device (SURVEY.md 8f-3).  The reference's callers turn the match list into boxes
 * (x, y, x+width, y+height, similarity), run a greedy NMS at IoU 0.5 and refine the first three survivors
 * with poseRefine (linemod_and_levelup_test.py:34-61, 325-367; linemod_ros/detect.py:41-81, 94-134).  Here
 * the NMS runs on the device behind the refinement kernel, on the kept records where they lie (all shards'
 * records with a connected peer exchange), and only the top_k survivors are copied to the host.
 *   lm_set_boxes      wh[n_templates][2]: box size per template in bank order (the drivers take it from their
 *                     template-info files); NULL / never called = Template::width/height of level 0 (LL.h:36-45)
 *   lm_enqueue_post   after lm_enqueue, same stream; top_k <= 0 = every survivor (at most 1024)
 *   lm_complete_post  waits; out[n_out] in pick order (best first); n_records = kept records the NMS saw
 *   lm_match_top      lm_upload_quantized + lm_enqueue + lm_enqueue_post + lm_complete_post
 * IoU as in the reference's nms(): float64, "+1" pixel convention, suppressed when ovr > threshold.  Equal
 * similarities (whose order the reference leaves to an unstable sort) are taken in template_id, class, y, x
 * order. */
int lm_set_boxes(lm_detector* d, const int32_t* wh, int64_t n_templates);
int lm_enqueue_post(lm_detector* d, double iou_threshold, int top_k);
int lm_complete_post(lm_detector* d, lm_match* out, int64_t cap, int64_t* n_out, int64_t* n_records);
int lm_match_top(lm_detector* d, const uint8_t* const* quantized, const int* rows, const int* cols, float threshold,
                 double iou_threshold, int top_k, lm_match* out, int64_t cap, int64_t* n_out, int64_t* n_records);

/* Convenience = lm_upload_quantized + lm_run + lm_fetch_records + lm_finish (single GPU):
 * Detector::match after quantization. */
int lm_match_quantized(lm_detector* d, const uint8_t* const* quantized, const int* rows, const int* cols,
                       float threshold, lm_match* out, int64_t cap, int64_t* n_out);

/* Detector::match proper (LL.cpp:1702-1777): raw images in, matches out. */
int lm_match_images(lm_detector* d, const uint8_t* rgb, const uint16_t* depth, int rows, int cols, const uint8_t* mask_color,
                    const uint8_t* mask_depth, float threshold, lm_match* out, int64_t cap, int64_t* n_out);

/* Template extraction of Detector::addTemplate (LL.cpp:1943-1975) for n_views views at once, on this handle's
 * device and stream with its pyramid levels L; the loaded bank and the uploaded frame are not touched.  View v is
 * rgb[v] (u8 rows x cols x 3), depth[v] (u16 rows x cols, mm) and masks[v] (u8 rows x cols, nonzero = object; masks
 * NULL or masks[v] NULL = no mask).  Per view and pyramid level it runs the GPU front-end of lm_upload_images
 * (labels without the mask), then ColorGradientPyramid::extractTemplate (LL.cpp:589-643: mask border, squared
 * magnitude > 55^2) and DepthNormalPyramid::extractTemplate (LL.cpp:888-966: mask eroded twice, per-label
 * chessboard distance transform, score = distance / candidates of the label), the stable sort by score and
 * selectScatteredFeatures (LL.cpp:279-318) with the reference's float32 arithmetic, and cropTemplates
 * (LL.cpp:234-277) on the host.  Outputs, feature for feature what the reference produces:
 *   ok[n_views]                  1 = extracted, 0 = too few candidates for some level / modality (addTemplate -1)
 *   tmeta[n_views][2L][4]        {width, height, first, count} per slot level*2 + modality, cropped; count =
 *                                num_features >> level, first = offset of the slot inside the view's features
 *   feats[n_views][F][3]         {x, y, label} in selection order, F = sum over levels of 2 * (num_features >> level)
 * Entries of views with ok = 0 are zero.  Views go through in chunks sized by free device memory.  LM_E_INVALID: a
 * null pointer, num_features >> (L - 1) < 1, rows or cols not a multiple of 2^(L-1) (the GPU pyrDown and
 * decimation serve even sizes; the host addTemplate serves the others) or above 16384.  A host-only handle
 * (device -1) gets LM_E_STATE.  Blocking. */
int lm_extract_templates(lm_detector* d, int num_features, int n_views, const uint8_t* const* rgb, const uint16_t* const* depth,
                         const uint8_t* const* masks, int rows, int cols, int32_t* ok, int32_t* tmeta, int32_t* feats);

/* ---- introspection used by the parity tests and the benchmark ---- */
/* Quantized label image of (level, modality) of the uploaded frame: rows*cols bytes. */
int lm_debug_quantized(lm_detector* d, int level, int modality, uint8_t* out, int64_t cap);
/* Linear memories of (level, modality) of the last lm_run: [8][T*T][(cols/T)*(rows/T)] bytes. */
int lm_debug_linear_memories(lm_detector* d, int level, int modality, uint8_t* out, int64_t cap);
/* Counters of the last lm_run: [0] templates scanned, [1] coarse candidates, [2] algorithmic bytes of
 * the coarse scan (sum over templates, modalities of features x positions; SURVEY 8d),
 * [3] algorithmic bytes of the refinement (features x 256 per refined candidate and level: the reference's work,
 * whichever kernel disposed of the candidate), [4] records kept after refinement, [5] bytes of the byte linear
 * memories the exact refinement kernel read (it stops early, exactly, on candidates that can no longer reach the
 * threshold), [6] the part of [3] that belongs to candidates the bit-sliced upper-bound filter dropped,
 * [7] bytes of H-planes that filter read.  [0],[2] describe this handle's shard.  `out8` has 8 entries. */
int lm_counters(lm_detector* d, int64_t* out8);
/* Per-stage device time in microseconds, from CUDA events recorded on the detector's stream around
 * each stage: [0] linear memories, [1] coarse scan, [2] candidate offsets, [3] refinement (= [5] + [6] + [7]),
 * [4] total, [5] candidate list + filter planes, [6] upper-bound filter, [7] exact refinement of the survivors (+ the
 * collector of the multi-GPU exchange).
 * lm_set_timing(d, slots) with slots > 0 enables it and keeps the last `slots` runs (0 disables);
 * lm_stage_times synchronises and returns the mean over the recorded runs.  `out8` has 8 entries. */
int lm_set_timing(lm_detector* d, int slots);
int lm_stage_times(lm_detector* d, float* out8);
/* The CUDA stream all work of this handle is issued on (cudaStream_t as void*). */
void* lm_stream(lm_detector* d);
/* Number of kernel launches issued by this handle since creation. */
int64_t lm_launch_count(lm_detector* d);

/* ---- poseRefine (reference: linemodLevelup/linemodLevelup.h:8-19, linemodLevelup.cpp:27-155) ---- */
typedef struct lm_icp lm_icp; /* replaces class poseRefine's compute; the R/t/residual state lives in the caller */

int lm_icp_create(int device, lm_icp** out);
void lm_icp_destroy(lm_icp* h);

/* poseRefine::process.  sceneDepth / modelDepth: u16 millimetres, row-major; sceneK / modelK / R: 9 floats
 * row-major; t: 3 floats (mm); detectX/Y: the match position.  max_iterations: Open3D's
 * ICPConvergenceCriteria::max_iteration_ (the reference uses the default, 30).  Outputs: R_out 9
 * doubles row-major (getR), t_out 3 doubles in mm (getT), residual = ICP fitness (getResidual), or -1
 * with R_out/t_out untouched when the model box does not fit the scene at the match position
 * (early return, LL.cpp:52-55). */
int lm_icp_process(lm_icp* h, const uint16_t* scene_depth, int srows, int scols, const uint16_t* model_depth, int mrows,
                   int mcols, const float* sceneK, const float* modelK, const float* R, const float* t, int detectX,
                   int detectY, int max_iterations, double* R_out, double* t_out, float* residual);

/* The same for n hypotheses against one scene image in one launch (what the callers do for the top
 * matches after NMS, linemod_and_levelup_test.py:351-367): model_depths[i], modelK + 9i, R + 9i,
 * t + 3i, detect_xy[2i..2i+1]; outputs R_out + 9i, t_out + 3i, residual[i]. */
int lm_icp_process_batch(lm_icp* h, int n_hyp, const uint16_t* scene_depth, int srows, int scols,
                         const uint16_t* const* model_depths, int mrows, int mcols, const float* sceneK, const float* modelK,
                         const float* R, const float* t, const int32_t* detect_xy, int max_iterations, double* R_out,
                         double* t_out, float* residual);

/* Of the last hypothesis processed: [0] points in the down-sampled cloud, [1] ICP iterations run,
 * [2] inlier rmse (m), [3] device time of the normals + ICP kernels of the last call (us). */
int lm_icp_last_stats(lm_icp* h, double* out4);
/* NOT the reference's behaviour (default off): register the model cloud against the down-sampled SCENE
 * cloud, which is what LL.cpp:109 evidently meant to do (it down-samples the model cloud twice). */
int lm_icp_set_use_scene_cloud(lm_icp* h, int on);
int64_t lm_icp_launch_count(lm_icp* h);

#ifdef __cplusplus
}
#endif
#endif
