// linemod_b200.cu -- hand-written sm_100a kernels + C-ABI for the LINEMOD match hot path.
//
// Reference being replaced: linemodLevelup::Detector::match and everything below it
// (linemodLevelup/linemodLevelup.cpp of meiqua/6DPose @ 619be57, "LL.cpp"):
//   kernels (lm_kernels.cuh): k_linear_memories_band, k_coarse_packed / k_coarse_bytes, k_scan_counts, k_refine_prep,
//                             k_refine_filter_w, k_refine_bits / k_refine, k_peer_collect
//   lm_finish (host)   <- std::sort + std::unique                       LL.cpp:1772-1774
//   lm_extract_templates <- Detector::addTemplate's extraction, batched over views (lm_train.cuh; cropTemplates on
//                           the host)                                   LL.cpp:234-318, 589-643, 888-966, 1943-1975
// Integer results (raw scores, x, y, template ids) are bit-exact; the float similarity is produced by
// the same two IEEE operations as the reference ((raw * 100.f) / (4 * n)).
//
// No tensor cores: bit-plane lookups / carry-save counters / small reductions.  No CPU fallback.

#include "linemod_b200.h"

#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

// --------------------------------------------------------------------------------------------
// error plumbing
// --------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#define CU(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(LM_E_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
  } while (0)

extern "C" const char* lm_last_error(void) { return g_err; }

// shared with lm_icp.cu
int lm_fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

#include "lm_kernels.cuh"
#include "lm_frontend.cuh"
#include "lm_post.cuh"
#include "lm_train.cuh"

#include <cub/device/device_segmented_sort.cuh>

// Launch with programmatic stream serialization (see lm_pdl_wait in lm_kernels.cuh).
template <typename... KArgs, typename... Args>
static cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}


// --------------------------------------------------------------------------------------------
// host side
// --------------------------------------------------------------------------------------------
#define LM_MAX_ROUNDS 5
#define LM_BITS_SMEM_LIMIT (200 * 1024)
#define LM_BAND_SMEM_LIMIT (160 * 1024)
#define LM_K2_SMEM_MAX (222 * 1024)  // dynamic shared memory of k_coarse_packed: bit-planes + the teams' partial counters
#define LM_CAND_DEFAULT (4ll << 20)  // candidate-list entries allocated up front (x 12 bytes)
#define LM_TEV 7  // timing events per frame: start, K1, K2, scan, prep, filter, end

struct LevelHost {
  int T = 0, rows = 0, cols = 0, Wd = 0, Hd = 0, plane = 0;
  uint8_t* d_q[LM_MAX_MODALITIES] = {nullptr, nullptr};           // owned upload buffers
  const uint8_t* q_src[LM_MAX_MODALITIES] = {nullptr, nullptr};  // what K1 reads (owned or caller's device memory)
  uint8_t* d_lm = nullptr;
  size_t lm_bytes = 0;
  uint32_t mod_stride = 0;
  uint32_t* d_bp = nullptr;  // lowest level only: spread bit-planes [M][8][lbw]
  int lbw = 0, nwords = 0, rounds = 0;
  int bp_zero = 0;   // words of zeros behind the bit-planes (where skipped / padding descriptors point)
};

struct lm_detector {
  int device = 0;
  cudaStream_t stream = nullptr;
  // host uploads: the upper-level label images travel on a second stream while the lowest level's linear
  // memories and the coarse scan already run (they only need the lowest level)
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_upper = nullptr;
  bool upper_pending = false;
  int L = 0, M = LM_MAX_MODALITIES;
  int T[LM_MAX_LEVELS] = {0};
  LevelHost lv[LM_MAX_LEVELS];
  bool have_frame = false, have_run = false;

  // bank (host)
  int n_classes = 0, S = 0, G = 0;
  std::vector<int32_t> class_begin, tmeta, feats;
  std::vector<uint8_t> feat_slot;  // slot (level*M+modality) of every feature
  // bank (device), prepared for the current frame size
  TSlot* d_tslot = nullptr;
  uint32_t* d_fbase = nullptr;
  uint32_t* d_fxy = nullptr;
  uint4* d_fdesc4 = nullptr;         // lowest-level features for k_coarse_packed: byte offsets of the label's plane window and of
                                     // its two neighbour labels' (x, y, z) + bit shift (w); per (template, modality) padded to
                                     // a multiple of 8 with entries that point at the all-zero words behind the planes
  int2* d_k2info = nullptr;          // [G][M]: first descriptor, padded count
  std::vector<uint8_t> bits_ok;      // per template: the bit-sliced coarse kernel may take it
  std::vector<uint8_t> safe;         // per template: refinement never skips a feature (LL.cpp:1394)
  uint8_t* d_safe = nullptr;
  uint16_t* d_galign = nullptr;      // [G][S][16] feature counts per (address & 15) group
  // refinement filter (k_refine_filter_w) on the first refined level lr = L - 2: column-major H-planes + descriptors
  bool filter_ok = false;            // the current frame size / bank allow it
  int last_planes_level = -1;        // level the last K1 built in planes mode (its byte linear memories are stale)
  uint32_t* d_rp = nullptr; size_t rp_words = 0; int rp_nyb = 0;
  uint32_t* d_rdesc = nullptr;       // per feature of level lr, grouped per template, padded to multiples of 32
  uint8_t* d_rlab = nullptr;         // label per descriptor (8 = padding): k_refine_bits derives the neighbour planes
  bool shard_all_eligible = false;   // every template of the shard is taken by the filter (no byte-wise refinement)
  uint32_t* d_surv2 = nullptr;       // candidates of the templates the filter does not take
  std::vector<int2> h_rfeat;         // per template: first descriptor, count (feeds h_finfo)
  int4* d_finfo = nullptr;           // per work item of the shard: first descriptor, count, width | height << 16,
                                     // flags | need << 8 (need: for the threshold of the call, see filter_thresholds)
  std::vector<int4> h_finfo;         // .w = flags only
  std::vector<int4> h_finfo_up;      // upload staging
  bool finfo_valid = false; float finfo_threshold = 0.f;
  uint2* d_cand = nullptr; int64_t cand_cap = 0;   // ordered candidate list (k_refine_prep)
  int64_t cand_need = 0;             // candidates of a frame that overflowed the list
  uint32_t* d_surv = nullptr;        // survivors of the filter [cand_cap]
  int* d_queue = nullptr;            // [0] next candidate, [1] survivors
  int prep_rows[LM_MAX_LEVELS] = {0}, prep_cols[LM_MAX_LEVELS] = {0};
  bool prepared = false;
  std::vector<TSlot> h_tslot;
  std::vector<uint8_t> feat_skip_low;

  // selection / shard
  std::vector<int32_t> sel;  // global template ids of the whole selected sequence
  int64_t shard_begin = 0, shard_count = 0;  // contiguous layout: [begin, begin + count) of sel
  int shard_index = 0, shard_n = 1;
  int shard_layout = LM_SHARD_CONTIGUOUS;
  int64_t work_base = 0, work_stride = 1;    // entry w of the shard is sel[work_base + w * work_stride]
  std::vector<int32_t> shard_sel;            // global template ids of this shard, in order
  int32_t* d_work = nullptr;
  int32_t* d_items_bits = nullptr; int n_items_bits = 0;    // work items per coarse kernel
  int32_t* d_items_bytes = nullptr; int n_items_bytes = 0;
  bool work_dirty = true;

  // per-run buffers
  uint32_t* d_mask = nullptr; size_t mask_elems = 0;  // [n_work][nwords] coarse pass bits
  uint16_t* d_raw = nullptr; size_t raw_elems = 0;    // [n_work][plane] coarse raw scores (passing cells)
  int32_t* d_cnt = nullptr; int32_t* d_off = nullptr; size_t cnt_elems = 0;
  // result block (device): lm_result_header + capacity records; internal unless the caller set one
  lm_result_header* d_res = nullptr; int64_t res_cap = 0; bool res_external = false;
  lm_result_header* d_res_own = nullptr; int64_t res_cap_own = 0;
  unsigned long long* d_counters = nullptr;
  unsigned long long* h_counters = nullptr;  // pinned
  lm_result_header* h_res = nullptr; int64_t h_res_cap = 0;  // pinned staging: header + records
  int64_t h_valid = 0;                                       // records already copied to h_res
  float last_threshold = 0.f;

  std::vector<int> class_of;            // template -> class (lm_finish), rebuilt when the bank changes
  std::vector<int32_t> order_cnt;       // order_records scratch
  std::vector<lm_record> order_tmp, finish_rec;
  std::vector<uint8_t> finish_keys;

  // post-match stage (lm_post.cuh): greedy NMS on the device, top-k survivors to the host
  std::vector<int32_t> boxes;           // [G][2] caller's box sizes (empty: L0 template width/height)
  PostInfo* d_post_info = nullptr; int64_t post_info_n = 0; bool post_dirty = true;
  lm_match* d_post_out = nullptr; lm_match* h_post_out = nullptr;  // LM_POST_MAX survivors
  int32_t* d_post_counts = nullptr; int32_t* h_post_counts = nullptr;
  uint8_t* d_post_live = nullptr; int64_t post_live_cap = 0;
  bool post_pending = false, post_retry = false;
  double post_iou = 0.5; int post_top_k = 0;

  // multi-GPU exchange fused into k_refine (lm_peer_*)
  uint8_t* px_buf = nullptr;            // this rank's exchange buffer (IPC-exportable cudaMalloc)
  int64_t px_cap = 0;                   // records per block
  int px_world = 0, px_rank = -1;       // px_rank >= 0: connected
  bool px_ipc = false;                  // peer bases opened with cudaIpcOpenMemHandle
  uint8_t* px_base[LM_MAX_PEERS] = {nullptr};
  int32_t px_seq = 0;
  unsigned long long px_timeout_ns = 1000000000ull;  // collector gives up on a peer after 1 s (LINEMOD_B200_PEER_TIMEOUT_MS)
  PeerExchange* d_px = nullptr;         // device copy of the descriptor (static after connect)
  PeerExchange h_px;

  // GPU quantization front-end (lm_upload_images): per level colour image, unfiltered bins, gate, normals, masks
  struct FeLevel {
    int rows = 0, cols = 0;
    uint8_t* src = nullptr; uint8_t* qun = nullptr; uint8_t* strong = nullptr; uint8_t* normal = nullptr;
    uint8_t* mask[LM_MAX_MODALITIES] = {nullptr, nullptr};
  } fe[LM_MAX_LEVELS];
  uint16_t* fe_depth = nullptr; uint8_t* fe_nraw = nullptr;
  bool fe_lut = false;

  bool timing = false;
  std::vector<cudaEvent_t> tev;  // timing slots x LM_TEV events (ring)
  int64_t timing_runs = 0;
  cudaEvent_t* ev = nullptr;     // the slot used by the run being enqueued
  int64_t launches = 0;
  int64_t alg_scan_bytes = 0;
  int sm_count = 148;
};

static void free_level(LevelHost& l) {
  for (int m = 0; m < LM_MAX_MODALITIES; ++m) {
    if (l.d_q[m]) cudaFree(l.d_q[m]);
    l.d_q[m] = nullptr;
    l.q_src[m] = nullptr;
  }
  if (l.d_lm) cudaFree(l.d_lm);
  l.d_lm = nullptr;
  if (l.d_bp) cudaFree(l.d_bp);
  l.d_bp = nullptr;
}

extern "C" int lm_create(int device, int n_levels, const int* T, lm_detector** out) {
  if (!out) return fail(LM_E_INVALID, "out is null");
  if (n_levels < 1 || n_levels > LM_MAX_LEVELS) return fail(LM_E_INVALID, "pyramid levels must be 1..%d", LM_MAX_LEVELS);
  for (int l = 0; l < n_levels; ++l)
    if (T[l] < 1 || T[l] > 16) return fail(LM_E_INVALID, "T[%d]=%d outside 1..16", l, T[l]);
  if (device == -1) {
    // host-only handle: bank / selection / shard ranges / lm_finish work, every GPU stage refuses to run
    lm_detector* d = new lm_detector();
    d->device = -1;
    d->L = n_levels;
    for (int l = 0; l < n_levels; ++l) d->T[l] = T[l];
    *out = d;
    return LM_OK;
  }
  int ndev = 0;
  cudaError_t e = cudaGetDeviceCount(&ndev);
  if (e != cudaSuccess || ndev == 0)
    return fail(LM_E_CUDA, "no CUDA device available (%s); this library has no CPU fallback", cudaGetErrorString(e));
  if (device < 0 || device >= ndev) return fail(LM_E_INVALID, "device %d out of range (have %d)", device, ndev);
  CU(cudaSetDevice(device));
  lm_detector* d = new lm_detector();
  d->device = device;
  d->L = n_levels;
  for (int l = 0; l < n_levels; ++l) d->T[l] = T[l];
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  d->sm_count = prop.multiProcessorCount;
  // function attributes are per DEVICE: every handle raises the dynamic shared-memory limits on its own device
  // (a process may hold handles on several GPUs, e.g. lm_peer_connect_local across devices)
  CU(cudaFuncSetAttribute(k_linear_memories_band, cudaFuncAttributeMaxDynamicSharedMemorySize, LM_BAND_SMEM_LIMIT));
  CU(cudaFuncSetAttribute(k_coarse_packed<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LM_K2_SMEM_MAX));
  CU(cudaFuncSetAttribute(k_coarse_packed<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
  CU(cudaStreamCreateWithFlags(&d->stream, cudaStreamNonBlocking));
  CU(cudaStreamCreateWithFlags(&d->copy_stream, cudaStreamNonBlocking));
  CU(cudaEventCreateWithFlags(&d->ev_fork, cudaEventDisableTiming));
  CU(cudaEventCreateWithFlags(&d->ev_upper, cudaEventDisableTiming));
  CU(cudaMalloc(&d->d_counters, 8 * sizeof(unsigned long long)));
  CU(cudaMemset(d->d_counters, 0, 8 * sizeof(unsigned long long)));
  CU(cudaMallocHost(&d->h_counters, 8 * sizeof(unsigned long long)));
  memset(d->h_counters, 0, 8 * sizeof(unsigned long long));
  CU(cudaMalloc(&d->d_queue, 4 * sizeof(int)));
  CU(cudaMemset(d->d_queue, 0, 4 * sizeof(int)));
  *out = d;
  return LM_OK;
}

static void peer_release(lm_detector* d) {
  if (d->px_ipc)
    for (int r = 0; r < d->px_world; ++r)
      if (r != d->px_rank && d->px_base[r]) cudaIpcCloseMemHandle(d->px_base[r]);
  for (int r = 0; r < LM_MAX_PEERS; ++r) d->px_base[r] = nullptr;
  d->px_rank = -1;
  d->px_ipc = false;
  if (d->px_buf) cudaFree(d->px_buf);
  d->px_buf = nullptr;
  if (d->d_px) cudaFree(d->d_px);
  d->d_px = nullptr;
  d->px_world = 0;
  d->px_cap = 0;
}

extern "C" void lm_destroy(lm_detector* d) {
  if (!d) return;
  if (d->device < 0) { delete d; return; }
  cudaSetDevice(d->device);
  if (d->stream) cudaStreamSynchronize(d->stream);
  peer_release(d);
  for (int l = 0; l < LM_MAX_LEVELS; ++l) free_level(d->lv[l]);
  cudaFree(d->d_tslot); cudaFree(d->d_fbase); cudaFree(d->d_fxy); cudaFree(d->d_fdesc4); cudaFree(d->d_k2info); cudaFree(d->d_work);
  cudaFree(d->d_items_bits); cudaFree(d->d_items_bytes); cudaFree(d->d_safe); cudaFree(d->d_galign);
  cudaFree(d->d_mask); cudaFree(d->d_raw); cudaFree(d->d_cnt); cudaFree(d->d_off);
  cudaFree(d->d_res_own); cudaFree(d->d_counters);
  cudaFree(d->d_finfo); cudaFree(d->d_rlab); cudaFree(d->d_surv2);
  cudaFree(d->d_rp); cudaFree(d->d_rdesc); cudaFree(d->d_cand); cudaFree(d->d_surv); cudaFree(d->d_queue);
  cudaFreeHost(d->h_counters); cudaFreeHost(d->h_res);
  cudaFree(d->d_post_info); cudaFree(d->d_post_out); cudaFree(d->d_post_counts); cudaFree(d->d_post_live);
  cudaFreeHost(d->h_post_out); cudaFreeHost(d->h_post_counts);
  for (int l = 0; l < LM_MAX_LEVELS; ++l) {
    cudaFree(d->fe[l].src); cudaFree(d->fe[l].qun); cudaFree(d->fe[l].strong); cudaFree(d->fe[l].normal);
    cudaFree(d->fe[l].mask[0]); cudaFree(d->fe[l].mask[1]);
  }
  cudaFree(d->fe_depth); cudaFree(d->fe_nraw);
  for (cudaEvent_t e : d->tev) cudaEventDestroy(e);
  if (d->copy_stream) { cudaStreamSynchronize(d->copy_stream); cudaStreamDestroy(d->copy_stream); }
  if (d->ev_fork) cudaEventDestroy(d->ev_fork);
  if (d->ev_upper) cudaEventDestroy(d->ev_upper);
  if (d->stream) cudaStreamDestroy(d->stream);
  delete d;
}

extern "C" void* lm_stream(lm_detector* d) { return d ? (void*)d->stream : nullptr; }
extern "C" int64_t lm_launch_count(lm_detector* d) { return d ? d->launches : 0; }

extern "C" int lm_load_bank(lm_detector* d, int n_classes, const int32_t* class_begin, int n_slots, const int32_t* tmeta,
                            const int32_t* feats, int64_t n_feats) {
  if (!d) return fail(LM_E_INVALID, "null detector");
  if (n_classes < 0 || !class_begin) return fail(LM_E_INVALID, "bad class table");
  if (n_slots != d->L * d->M)
    return fail(LM_E_INVALID, "template pyramids have %d templates, detector expects %d (levels x modalities)", n_slots,
                d->L * d->M);
  const int G = class_begin[n_classes];
  if (class_begin[0] != 0) return fail(LM_E_INVALID, "class_begin[0] must be 0");
  for (int c = 0; c < n_classes; ++c)
    if (class_begin[c + 1] < class_begin[c]) return fail(LM_E_INVALID, "class_begin not monotone");
  std::vector<uint8_t> slot_of((size_t)n_feats, 255);
  for (int g = 0; g < G; ++g)
    for (int s = 0; s < n_slots; ++s) {
      const int32_t* m4 = tmeta + ((size_t)g * n_slots + s) * 4;
      if (m4[2] < 0 || m4[3] < 0 || (int64_t)m4[2] + m4[3] > n_feats)
        return fail(LM_E_INVALID, "template %d slot %d: feature range out of bounds", g, s);
      if (m4[3] > 8191)  // CV_Assert(templ.features.size() <= 8191), LL.cpp:1291
        return fail(LM_E_INVALID, "template %d slot %d has %d features (> 8191)", g, s, m4[3]);
      if (m4[0] < 0 || m4[1] < 0 || m4[0] > 32767 || m4[1] > 32767)
        return fail(LM_E_INVALID, "template %d slot %d: width/height outside 0..32767", g, s);
      for (int i = 0; i < m4[3]; ++i) {
        const int32_t* f = feats + ((size_t)m4[2] + i) * 3;
        if (f[2] < 0 || f[2] > 7) return fail(LM_E_INVALID, "feature label %d outside [0,8)", f[2]);
        if (f[0] < 0 || f[1] < 0 || f[0] > 32767 || f[1] > 32767)
          return fail(LM_E_INVALID, "feature coordinate (%d,%d) outside 0..32767", f[0], f[1]);
        slot_of[(size_t)m4[2] + i] = (uint8_t)s;
      }
    }
  if (d->device >= 0) CU(cudaSetDevice(d->device));
  d->n_classes = n_classes;
  d->S = n_slots;
  d->G = G;
  d->class_begin.assign(class_begin, class_begin + n_classes + 1);
  d->tmeta.assign(tmeta, tmeta + (size_t)G * n_slots * 4);
  d->class_of.clear();
  d->boxes.clear();  // box sizes belong to the bank they were set for
  d->post_dirty = true;
  d->feats.assign(feats, feats + (size_t)n_feats * 3);
  d->feat_slot.swap(slot_of);
  cudaFree(d->d_tslot); cudaFree(d->d_fbase); cudaFree(d->d_fxy); cudaFree(d->d_fdesc4); cudaFree(d->d_k2info);
  d->d_tslot = nullptr; d->d_fbase = nullptr; d->d_fxy = nullptr; d->d_fdesc4 = nullptr; d->d_k2info = nullptr;
  if (d->device >= 0 && G > 0) CU(cudaMalloc(&d->d_tslot, sizeof(TSlot) * (size_t)G * n_slots));
  if (d->device >= 0 && n_feats > 0) {
    CU(cudaMalloc(&d->d_fbase, sizeof(uint32_t) * (size_t)n_feats));
    CU(cudaMalloc(&d->d_fxy, sizeof(uint32_t) * (size_t)n_feats));
  }
  d->prepared = false;
  d->have_run = false;
  // default selection: everything, one shard
  return lm_select(d, nullptr, -1, 0, 1);
}

// Which accumulator width the reference would use and whether it would assert (LL.cpp:1813-1824).
static int check_paths(const lm_detector* d, int g) {
  for (int l = 0; l < d->L; ++l) {
    int width = -1;
    for (int m = 0; m < d->M; ++m) {
      const int nf = d->tmeta[((size_t)g * d->S + l * d->M + m) * 4 + 3];
      if (width <= 0) width = nf < 64 ? 1 : (nf < 8192 ? 2 : width);
      if (width == 1 && nf > 63) return -1;  // CV_Assert(features.size() <= 63), LL.cpp:1457/1551
    }
  }
  return 0;
}

extern "C" int lm_select(lm_detector* d, const int32_t* class_sel, int n_classes_sel, int shard_index, int shard_count) {
  return lm_select_layout(d, class_sel, n_classes_sel, shard_index, shard_count, LM_SHARD_CONTIGUOUS);
}

extern "C" int lm_select_layout(lm_detector* d, const int32_t* class_sel, int n_classes_sel, int shard_index, int shard_count,
                                int layout) {
  if (!d) return fail(LM_E_INVALID, "null detector");
  if (layout != LM_SHARD_CONTIGUOUS && layout != LM_SHARD_INTERLEAVED) return fail(LM_E_INVALID, "unknown shard layout %d", layout);
  if (shard_count < 1 || shard_index < 0 || shard_index >= shard_count) return fail(LM_E_INVALID, "bad shard %d/%d", shard_index, shard_count);
  std::vector<int32_t> sel;
  if (n_classes_sel < 0) {
    sel.resize(d->G);
    for (int g = 0; g < d->G; ++g) sel[g] = g;
  } else {
    for (int i = 0; i < n_classes_sel; ++i) {
      const int c = class_sel[i];
      if (c < 0 || c >= d->n_classes) return fail(LM_E_INVALID, "class index %d out of range", c);
      for (int g = d->class_begin[c]; g < d->class_begin[c + 1]; ++g) sel.push_back(g);
    }
  }
  for (int32_t g : sel)
    if (check_paths(d, g) != 0)
      return fail(LM_E_INVALID, "template %d: first modality has < 64 features but another has > 63 "
                                "(the reference asserts in similarity_64)", g);
  // contiguous shard, balanced by lowest-level feature count (the coarse scan's work per template)
  const int low = (d->L - 1) * d->M;
  std::vector<int64_t> cum(sel.size() + 1, 0);
  for (size_t i = 0; i < sel.size(); ++i) {
    int64_t c = 1;
    for (int m = 0; m < d->M; ++m) c += d->tmeta[((size_t)sel[i] * d->S + low + m) * 4 + 3];
    cum[i + 1] = cum[i] + c;
  }
  auto cut = [&](int k) -> int64_t {
    if (k <= 0) return 0;
    if (k >= shard_count) return (int64_t)sel.size();
    const int64_t target = cum.back() * k / shard_count;
    return (int64_t)(std::lower_bound(cum.begin(), cum.end(), target) - cum.begin());
  };
  d->shard_index = shard_index;
  d->shard_n = shard_count;
  d->shard_layout = layout;
  if (layout == LM_SHARD_INTERLEAVED) {
    // entry w of shard r is element r + w * N of the selected sequence: neighbouring templates (views / in-plane
    // variants of one another, which pass or fail together) are dealt round the ranks, so the candidate load per
    // rank evens out where contiguous blocks do not
    d->work_base = shard_index;
    d->work_stride = shard_count;
    d->shard_begin = shard_index;
    d->shard_count = ((int64_t)sel.size() - shard_index + shard_count - 1) / shard_count;
    if (d->shard_count < 0) d->shard_count = 0;
  } else {
    d->shard_begin = cut(shard_index);
    d->shard_count = cut(shard_index + 1) - d->shard_begin;
    d->work_base = d->shard_begin;
    d->work_stride = 1;
  }
  d->shard_sel.resize((size_t)d->shard_count);
  for (int64_t w = 0; w < d->shard_count; ++w) d->shard_sel[(size_t)w] = sel[(size_t)(d->work_base + w * d->work_stride)];
  d->sel.swap(sel);  // after the cuts: the lambda reads `sel`
  d->work_dirty = true;
  d->post_dirty = true;
  d->have_run = false;
  return LM_OK;
}

extern "C" int lm_shard_range(lm_detector* d, int64_t* begin, int64_t* count) {
  if (!d) return fail(LM_E_INVALID, "null detector");
  if (begin) *begin = d->shard_begin;
  if (count) *count = d->shard_count;
  return LM_OK;
}

// Feature addresses depend on the frame size (Wd, Hd); recomputed when it changes.
static int prepare_bank(lm_detector* d) {
  bool same = d->prepared;
  for (int l = 0; l < d->L && same; ++l) same = d->prep_rows[l] == d->lv[l].rows && d->prep_cols[l] == d->lv[l].cols;
  if (same) return LM_OK;
  const size_t nf = d->feat_slot.size();
  std::vector<uint32_t> fbase(nf, 0), fxy(nf, 0);
  const int low_level = d->L - 1;
  for (size_t i = 0; i < nf; ++i) {
    const int s = d->feat_slot[i];
    if (s == 255) continue;  // feature not referenced by any template
    const int l = s / d->M, m = s % d->M;
    const LevelHost& lv = d->lv[l];
    const int x = d->feats[3 * i], y = d->feats[3 * i + 1], lab = d->feats[3 * i + 2];
    const int T = lv.T;
    const uint64_t a = (uint64_t)m * lv.mod_stride + (uint64_t)lab * T * T * lv.plane +
                       (uint64_t)((y % T) * T + (x % T)) * lv.plane + (uint64_t)(y / T) * lv.Wd + (x / T);
    fbase[i] = (uint32_t)a;
    uint32_t v = (uint32_t)x | ((uint32_t)y << 16);
    if (x >= lv.cols || y >= lv.rows) v |= LM_SKIP_BIT;  // LL.cpp:1330
    fxy[i] = v;
  }
  d->h_tslot.resize((size_t)d->G * d->S);
  for (int g = 0; g < d->G; ++g)
    for (int s = 0; s < d->S; ++s) {
      const int32_t* m4 = &d->tmeta[((size_t)g * d->S + s) * 4];
      const LevelHost& lv = d->lv[s / d->M];
      const int wf = (m4[0] - 1) / lv.T + 1, hf = (m4[1] - 1) / lv.T + 1;  // LL.cpp:1299-1300
      TSlot t;
      t.x = m4[2];
      t.y = m4[3];
      t.z = (lv.Hd - hf) * lv.Wd + (lv.Wd - wf) + 1;  // LL.cpp:1309
      t.w = (int)((uint32_t)m4[0] | ((uint32_t)m4[1] << 16));
      d->h_tslot[(size_t)g * d->S + s] = t;
    }
  // the bit-sliced coarse kernel counts in 8 bits and masks once: it takes templates with at most 255
  // lowest-level features in total and the same template_positions in every modality
  d->bits_ok.assign((size_t)d->G, 0);
  {
    const LevelHost& lv = d->lv[low_level];
    for (int g = 0; g < d->G && lv.d_bp; ++g) {
      int total = 0;
      bool same = true;
      const TSlot& t0 = d->h_tslot[(size_t)g * d->S + low_level * d->M];
      for (int m = 0; m < d->M; ++m) {
        const TSlot& t = d->h_tslot[(size_t)g * d->S + low_level * d->M + m];
        total += t.y;
        same = same && t.z == t0.z;
      }
      d->bits_ok[g] = (total <= 255 && same) ? 1 : 0;
    }
  }
  // k_coarse_packed descriptors: per lowest-level feature the byte offsets (inside the bit-plane buffer) of the window
  // start of its label's plane and of the two neighbouring labels' planes, and the bit shift.  Features outside the
  // image (LL.cpp:1330) and the padding to a multiple of 8 per (template, modality) point at the zero words behind the
  // planes, so the kernel's loop has neither a skip branch nor a bounds check.
  cudaFree(d->d_fdesc4); d->d_fdesc4 = nullptr;
  cudaFree(d->d_k2info); d->d_k2info = nullptr;
  {
    const LevelHost& lv = d->lv[low_level];
    if (lv.d_bp && d->G > 0) {
      std::vector<uint4> f4;
      std::vector<int2> k2((size_t)d->G * d->M);
      const uint32_t zoff = (uint32_t)((size_t)d->M * 8 * lv.lbw) * 4u;  // byte offset of the zero words
      const int T = lv.T;
      for (int g = 0; g < d->G; ++g)
        for (int m = 0; m < d->M; ++m) {
          const int32_t* tm = &d->tmeta[((size_t)g * d->S + low_level * d->M + m) * 4];
          k2[(size_t)g * d->M + m].x = (int)f4.size();
          for (int k = 0; k < tm[3]; ++k) {
            const size_t i = (size_t)tm[2] + k;
            const int x = d->feats[3 * i], y = d->feats[3 * i + 1], lab = d->feats[3 * i + 2];
            if (x >= lv.cols || y >= lv.rows) {
              f4.push_back(make_uint4(zoff, zoff, zoff, 0u));
              continue;
            }
            const uint64_t inner = (uint64_t)((y % T) * T + (x % T)) * lv.plane + (uint64_t)(y / T) * lv.Wd + (x / T);
            const uint64_t wh = (uint64_t)(m * 8 + lab) * lv.lbw + (inner >> 5);
            const uint64_t wm = (uint64_t)(m * 8 + ((lab + 7) & 7)) * lv.lbw + (inner >> 5);
            const uint64_t wp = (uint64_t)(m * 8 + ((lab + 1) & 7)) * lv.lbw + (inner >> 5);
            f4.push_back(make_uint4((uint32_t)(wh * 4), (uint32_t)(wm * 4), (uint32_t)(wp * 4), (uint32_t)(inner & 31)));
          }
          while ((f4.size() - (size_t)k2[(size_t)g * d->M + m].x) % 8) f4.push_back(make_uint4(zoff, zoff, zoff, 0u));
          k2[(size_t)g * d->M + m].y = (int)(f4.size() - (size_t)k2[(size_t)g * d->M + m].x);
        }
      CU(cudaMalloc(&d->d_fdesc4, std::max<size_t>(f4.size(), 1) * sizeof(uint4)));
      CU(cudaMalloc(&d->d_k2info, k2.size() * sizeof(int2)));
      if (!f4.empty()) CU(cudaMemcpyAsync(d->d_fdesc4, f4.data(), f4.size() * sizeof(uint4), cudaMemcpyHostToDevice, d->stream));
      CU(cudaMemcpyAsync(d->d_k2info, k2.data(), k2.size() * sizeof(int2), cudaMemcpyHostToDevice, d->stream));
      CU(cudaStreamSynchronize(d->stream));
    }
  }
  // "safe" templates: at every refined level the clamp range is regular (max >= border) and every
  // feature lies inside the template box, so no feature can leave the image once a clamped patch
  // offset is applied (LL.cpp:1394 never skips) -- the refinement kernel then drops the per-feature test
  d->safe.assign((size_t)d->G, 0);
  for (int g = 0; g < d->G; ++g) {
    bool ok = true;
    for (int l = 0; l + 1 < d->L && ok; ++l) {
      const LevelHost& lv = d->lv[l];
      const int32_t* t0 = &d->tmeta[((size_t)g * d->S + l * d->M) * 4];
      const int border = 8 * lv.T;
      ok = lv.cols - t0[0] - border >= border && lv.rows - t0[1] - border >= border;
      for (int m = 0; m < d->M && ok; ++m) {
        const int32_t* tm = &d->tmeta[((size_t)g * d->S + l * d->M + m) * 4];
        for (int k = 0; k < tm[3] && ok; ++k) {
          const int32_t* f = &d->feats[3 * ((size_t)tm[2] + k)];
          ok = f[0] <= t0[0] && f[1] <= t0[1];
        }
      }
    }
    d->safe[g] = ok ? 1 : 0;
  }
  // refined levels: store each template's features grouped by (address & 15) -- sums do not depend
  // on the order, and the refinement kernel then knows the row alignment of a whole group at once
  std::vector<uint16_t> galign((size_t)d->G * d->S * 16, 0);
  for (int g = 0; g < d->G; ++g)
    for (int s = 0; s < d->S - d->M; ++s) {  // every slot above the lowest level
      const int32_t* tm = &d->tmeta[((size_t)g * d->S + s) * 4];
      const size_t b0 = (size_t)tm[2];
      const int n = tm[3];
      std::vector<int> order(n);
      for (int k = 0; k < n; ++k) order[k] = k;
      std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return (fbase[b0 + a] & 15u) < (fbase[b0 + b] & 15u); });
      std::vector<uint32_t> tb(n), tx(n);
      for (int k = 0; k < n; ++k) {
        tb[k] = fbase[b0 + order[k]];
        tx[k] = fxy[b0 + order[k]];
        ++galign[((size_t)g * d->S + s) * 16 + (tb[k] & 15u)];
      }
      for (int k = 0; k < n; ++k) { fbase[b0 + k] = tb[k]; fxy[b0 + k] = tx[k]; }
    }
  cudaFree(d->d_galign);
  d->d_galign = nullptr;
  if (!galign.empty()) {
    CU(cudaMalloc(&d->d_galign, galign.size() * sizeof(uint16_t)));
    CU(cudaMemcpyAsync(d->d_galign, galign.data(), galign.size() * sizeof(uint16_t), cudaMemcpyHostToDevice, d->stream));
  }
  // refinement filter (k_refine_filter_w) on the first refined level: column-major H-planes [M*8*T*T][nyb][Wd] and one
  // descriptor per feature = plane word offset (incl. x / T) : 23 | y / T : 9.  Eligible templates ("safe", so that
  // the 16x16 patch of every feature is a true 2-D window of the level, and at most 511 features at that level) get
  // bit 1 of their flag byte; the others go to k_refine unfiltered.
  d->filter_ok = false;
  std::vector<uint32_t> rdesc;
  std::vector<uint8_t> rlab;
  std::vector<int2> rfeat((size_t)d->G, make_int2(0, 0));
  if (d->L >= 2) {
    const int lr = d->L - 2;
    const LevelHost& lv = d->lv[lr];
    const int T = lv.T, T2 = T * T;
    const int nyb = lv.Hd >= 16 ? ((lv.Hd - 16) >> 4) + 1 : 0;
    const size_t words = (size_t)d->M * 8 * T2 * nyb * lv.Wd;
    // all-zero tail behind the planes: where the padding descriptors (and nothing else) point
    const size_t tail = (size_t)(nyb + 1) * lv.Wd + 64;
    if (lv.Wd % 4 == 0 && lv.Wd >= 16 && lv.Hd >= 16 && lv.Hd <= 512 && words > 0 && words + tail <= (1u << 23)) {
      d->filter_ok = true;
      d->rp_nyb = nyb;
      if (words != d->rp_words) {
        cudaFree(d->d_rp);
        d->d_rp = nullptr;
        d->rp_words = words;
        CU(cudaMalloc(&d->d_rp, (words + tail) * 4));
        CU(cudaMemsetAsync(d->d_rp, 0, (words + tail) * 4, d->stream));  // halves no row block covers stay zero
      }
      for (int g = 0; g < d->G; ++g) {
        int nfl = 0;
        for (int m = 0; m < d->M; ++m) nfl += d->tmeta[((size_t)g * d->S + lr * d->M + m) * 4 + 3];
        if (!d->safe[g] || nfl < 1 || nfl > 511) continue;
        d->safe[g] |= 2;
        rfeat[(size_t)g] = make_int2((int)rdesc.size(), nfl);
        for (int m = 0; m < d->M; ++m) {
          const int32_t* tm = &d->tmeta[((size_t)g * d->S + lr * d->M + m) * 4];
          for (int k = 0; k < tm[3]; ++k) {
            const int32_t* f = &d->feats[3 * ((size_t)tm[2] + k)];
            const uint32_t pb = (uint32_t)((m * 8 + f[2]) * T2 + (f[1] % T) * T + (f[0] % T));
            rdesc.push_back((pb * (uint32_t)nyb * (uint32_t)lv.Wd + (uint32_t)(f[0] / T)) | ((uint32_t)(f[1] / T) << 23));
            rlab.push_back((uint8_t)f[2]);
          }
        }
        while (rdesc.size() % 32) {  // padding: the zero tail, row 0
          rdesc.push_back((uint32_t)words);
          rlab.push_back(8);
        }
      }
    }
  }
  d->h_rfeat = rfeat;
  cudaFree(d->d_rdesc); d->d_rdesc = nullptr;
  cudaFree(d->d_rlab); d->d_rlab = nullptr;
  if (d->filter_ok) {
    CU(cudaMalloc(&d->d_rlab, std::max<size_t>(rlab.size(), 1)));
    if (!rlab.empty()) CU(cudaMemcpyAsync(d->d_rlab, rlab.data(), rlab.size(), cudaMemcpyHostToDevice, d->stream));
    CU(cudaMalloc(&d->d_rdesc, std::max<size_t>(rdesc.size(), 1) * 4));
    if (!rdesc.empty()) CU(cudaMemcpyAsync(d->d_rdesc, rdesc.data(), rdesc.size() * 4, cudaMemcpyHostToDevice, d->stream));
  }
  cudaFree(d->d_safe);
  d->d_safe = nullptr;
  if (d->G) {
    CU(cudaMalloc(&d->d_safe, (size_t)d->G));
    CU(cudaMemcpyAsync(d->d_safe, d->safe.data(), (size_t)d->G, cudaMemcpyHostToDevice, d->stream));
  }
  if (nf) {
    CU(cudaMemcpyAsync(d->d_fbase, fbase.data(), nf * 4, cudaMemcpyHostToDevice, d->stream));
    CU(cudaMemcpyAsync(d->d_fxy, fxy.data(), nf * 4, cudaMemcpyHostToDevice, d->stream));
  }
  if (d->G) CU(cudaMemcpyAsync(d->d_tslot, d->h_tslot.data(), sizeof(TSlot) * d->h_tslot.size(), cudaMemcpyHostToDevice, d->stream));
  CU(cudaStreamSynchronize(d->stream));  // host vectors go out of scope
  d->feat_skip_low.assign(nf, 0);
  for (size_t i = 0; i < nf; ++i) d->feat_skip_low[i] = (fxy[i] & LM_SKIP_BIT) ? 1 : 0;
  for (int l = 0; l < d->L; ++l) { d->prep_rows[l] = d->lv[l].rows; d->prep_cols[l] = d->lv[l].cols; }
  d->prepared = true;
  d->work_dirty = true;
  d->post_dirty = true;
  return LM_OK;
}

static int prepare_work(lm_detector* d) {
  if (!d->work_dirty) return LM_OK;
  const int64_t n = d->shard_count;
  cudaFree(d->d_work); d->d_work = nullptr;
  if (n > 0) {
    CU(cudaMalloc(&d->d_work, sizeof(int32_t) * (size_t)n));
    CU(cudaMemcpyAsync(d->d_work, d->shard_sel.data(), sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, d->stream));
    CU(cudaStreamSynchronize(d->stream));
  }
  {
    std::vector<int32_t> ib, iy;
    for (int64_t i = 0; i < n; ++i) (d->bits_ok[d->shard_sel[(size_t)i]] ? ib : iy).push_back((int32_t)i);
    cudaFree(d->d_items_bits); d->d_items_bits = nullptr;
    cudaFree(d->d_items_bytes); d->d_items_bytes = nullptr;
    d->n_items_bits = (int)ib.size();
    d->n_items_bytes = (int)iy.size();
    if (!ib.empty()) {
      CU(cudaMalloc(&d->d_items_bits, sizeof(int32_t) * ib.size()));
      CU(cudaMemcpyAsync(d->d_items_bits, ib.data(), sizeof(int32_t) * ib.size(), cudaMemcpyHostToDevice, d->stream));
    }
    if (!iy.empty()) {
      CU(cudaMalloc(&d->d_items_bytes, sizeof(int32_t) * iy.size()));
      CU(cudaMemcpyAsync(d->d_items_bytes, iy.data(), sizeof(int32_t) * iy.size(), cudaMemcpyHostToDevice, d->stream));
    }
    CU(cudaStreamSynchronize(d->stream));
  }
  if ((size_t)n + 1 > d->cnt_elems) {
    cudaFree(d->d_cnt); cudaFree(d->d_off);
    d->cnt_elems = (size_t)n + 1;
    CU(cudaMalloc(&d->d_cnt, sizeof(int32_t) * d->cnt_elems));
    CU(cudaMalloc(&d->d_off, sizeof(int32_t) * d->cnt_elems));
  }
  cudaFree(d->d_finfo);
  d->d_finfo = nullptr;
  d->h_finfo.clear();
  if (d->filter_ok && n > 0) {
    const int lr = d->L - 2;
    d->h_finfo.resize((size_t)n);
    for (int64_t i = 0; i < n; ++i) {
      const int g = d->shard_sel[(size_t)i];
      const int32_t* t0 = &d->tmeta[((size_t)g * d->S + lr * d->M) * 4];
      d->h_finfo[(size_t)i] = make_int4(d->h_rfeat[(size_t)g].x, d->h_rfeat[(size_t)g].y,
                                        (int)((uint32_t)t0[0] | ((uint32_t)t0[1] << 16)), (int)d->safe[(size_t)g]);
    }
    CU(cudaMalloc(&d->d_finfo, sizeof(int4) * (size_t)n));
    d->finfo_valid = false;  // the threshold-dependent part is filled in by lm_enqueue
    d->shard_all_eligible = true;
    for (const int4& f : d->h_finfo) d->shard_all_eligible = d->shard_all_eligible && (f.w & 2);
  }
  // per-template candidate counts are accumulated with atomics and re-zeroed by k_scan_counts
  CU(cudaMemsetAsync(d->d_cnt, 0, sizeof(int32_t) * d->cnt_elems, d->stream));
  CU(cudaStreamSynchronize(d->stream));
  // algorithmic bytes of the coarse scan for this shard (SURVEY 8d): sum features x positions
  const int low = (d->L - 1) * d->M;
  int64_t bytes = 0;
  for (int64_t i = 0; i < n; ++i) {
    const int g = d->shard_sel[(size_t)i];
    for (int m = 0; m < d->M; ++m) {
      const TSlot& t = d->h_tslot[(size_t)g * d->S + low + m];
      if (t.z <= 0) continue;
      int live = 0;
      for (int k = 0; k < t.y; ++k) live += d->feat_skip_low[(size_t)t.x + k] ? 0 : 1;
      bytes += (int64_t)live * t.z;
    }
  }
  d->alg_scan_bytes = bytes;
  d->work_dirty = false;
  return LM_OK;
}

// Smallest raw score that survives remove_if(similarity < threshold) (LL.cpp:1935-1937), host twin of lm_min_kept_raw:
// the same two IEEE single-precision operations ((raw * 100.f) / (4 * n)).
static int host_min_kept_raw(float threshold, int nfeat) {
  int lo = 0, hi = 4 * nfeat + 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    volatile float prod = (float)mid * 100.f;
    volatile float score = prod / (float)(4 * nfeat);
    if (!(score < threshold)) hi = mid; else lo = mid + 1;
  }
  return lo;
}

// finfo[w].w = flags | need << 8 for this threshold: need = number of features whose label bit must be set at some cell
// of the patch for the candidate to be able to reach raw_keep (see k_refine_filter_w).
static int filter_thresholds(lm_detector* d, float threshold) {
  if (!d->filter_ok || !d->d_finfo || d->h_finfo.empty()) return LM_OK;
  if (d->finfo_valid && memcmp(&threshold, &d->finfo_threshold, sizeof(float)) == 0) return LM_OK;
  d->h_finfo_up = d->h_finfo;
  int last_nf = -1, last_need = 0;
  for (int4& f : d->h_finfo_up) {
    if (!(f.w & 2)) continue;
    if (f.y != last_nf) {
      last_nf = f.y;
      const int over = host_min_kept_raw(threshold, f.y) - f.y;
      last_need = over > 0 ? (over + 2) / 3 : 0;
    }
    f.w |= last_need << 8;
  }
  CU(cudaMemcpyAsync(d->d_finfo, d->h_finfo_up.data(), sizeof(int4) * d->h_finfo_up.size(), cudaMemcpyHostToDevice, d->stream));
  d->finfo_valid = true;
  d->finfo_threshold = threshold;
  return LM_OK;
}

static int check_frame_dims(lm_detector* d, const int* rows, const int* cols) {
  for (int l = 0; l < d->L; ++l) {
    const int T = d->T[l];
    if (rows[l] <= 0 || cols[l] <= 0) return fail(LM_E_INVALID, "level %d: empty image", l);
    if (rows[l] % T || cols[l] % T)  // CV_Assert LL.cpp:1217-1218
      return fail(LM_E_INVALID, "level %d: %dx%d not a multiple of T=%d", l, cols[l], rows[l], T);
    if (((int64_t)rows[l] * cols[l]) % 16)  // CV_Assert LL.cpp:1136
      return fail(LM_E_INVALID, "level %d: rows*cols not a multiple of 16", l);
    if (rows[l] > 32767 || cols[l] > 32767) return fail(LM_E_INVALID, "level %d: image side > 32767", l);
  }
  const int l = d->L - 1;
  if ((int64_t)(rows[l] / d->T[l]) * (cols[l] / d->T[l]) > 65536)
    return fail(LM_E_INVALID, "lowest level has more than 65536 sampled positions");
  return LM_OK;
}

// (Re)allocate the per-level device buffers for a frame size.
static int size_levels(lm_detector* d, const int* rows, const int* cols, bool need_upload_buffers) {
  for (int l = 0; l < d->L; ++l) {
    LevelHost& lv = d->lv[l];
    if (lv.rows != rows[l] || lv.cols != cols[l] || lv.T != d->T[l]) {
      free_level(lv);
      lv.T = d->T[l]; lv.rows = rows[l]; lv.cols = cols[l];
      lv.Wd = cols[l] / lv.T; lv.Hd = rows[l] / lv.T; lv.plane = lv.Wd * lv.Hd;
      const size_t per_mod = (size_t)8 * lv.T * lv.T * lv.plane;
      // slack: the coarse scan reads up to one plane past a feature's base, the 16x16 patch up to 16 rows
      const size_t slack = (size_t)lv.plane + 16 * (size_t)lv.Wd + 256;
      if (per_mod * d->M + slack > 0xFFFFFFFFull) return fail(LM_E_INVALID, "level %d: linear memories exceed 4 GiB", l);
      lv.mod_stride = (uint32_t)per_mod;
      lv.lm_bytes = per_mod * d->M + slack;
      CU(cudaMalloc(&lv.d_lm, lv.lm_bytes));
      CU(cudaMemsetAsync(lv.d_lm, 0, lv.lm_bytes, d->stream));
      lv.nwords = (lv.plane + 31) / 32;
      lv.rounds = (lv.nwords + 31) / 32;
      if (l == d->L - 1 && lv.rounds <= LM_MAX_ROUNDS) {
        // label block: T*T*plane bits, then slack for the reads of lanes beyond the last word
        const size_t bits = (size_t)lv.T * lv.T * lv.plane;
        lv.lbw = (int)(((bits + 31) / 32 + 32 * (size_t)lv.rounds + 4 + 3) & ~(size_t)3);
        lv.bp_zero = (lv.nwords + 32 * lv.rounds + 8 + 3) & ~3;  // a lane reads words idx and idx + 1 of a window
        const size_t words = (size_t)d->M * 8 * lv.lbw + lv.bp_zero;
        CU(cudaMalloc(&lv.d_bp, words * 4));
        CU(cudaMemsetAsync(lv.d_bp, 0, words * 4, d->stream));
      }
      d->prepared = false;  // feature addresses depend on the frame size
    }
    if (need_upload_buffers)
      for (int m = 0; m < d->M; ++m)
        if (!lv.d_q[m]) CU(cudaMalloc(&lv.d_q[m], (size_t)rows[l] * cols[l]));
  }
  return LM_OK;
}

static int upload_quantized(lm_detector* d, const uint8_t* const* quantized, const int* rows, const int* cols, bool sync);

extern "C" int lm_upload_quantized(lm_detector* d, const uint8_t* const* quantized, const int* rows, const int* cols) {
  return upload_quantized(d, quantized, rows, cols, true);
}

static int upload_quantized(lm_detector* d, const uint8_t* const* quantized, const int* rows, const int* cols, bool sync) {
  if (d && d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  if (!d || !quantized || !rows || !cols) return fail(LM_E_INVALID, "null argument");
  CU(cudaSetDevice(d->device));
  int rc = check_frame_dims(d, rows, cols);
  if (rc) return rc;
  rc = size_levels(d, rows, cols, true);
  if (rc) return rc;
  for (int i = 0; i < d->L * d->M; ++i)
    if (!quantized[i]) return fail(LM_E_INVALID, "quantized[%d] is null", i);
  // lowest level first, on the main stream: its linear memories and the coarse scan need nothing else.  The
  // larger upper levels follow on the copy stream (ordered behind everything already enqueued) and are joined
  // in front of the upper levels' linear memories (enqueue_stages).
  const bool fork = d->L > 1;
  if (fork) {
    CU(cudaEventRecord(d->ev_fork, d->stream));
    CU(cudaStreamWaitEvent(d->copy_stream, d->ev_fork, 0));
  }
  for (int l = d->L - 1; l >= 0; --l) {
    LevelHost& lv = d->lv[l];
    cudaStream_t st = (fork && l < d->L - 1) ? d->copy_stream : d->stream;
    for (int m = 0; m < d->M; ++m) {
      CU(cudaMemcpyAsync(lv.d_q[m], quantized[l * d->M + m], (size_t)rows[l] * cols[l], cudaMemcpyHostToDevice, st));
      lv.q_src[m] = lv.d_q[m];
    }
  }
  if (fork) {
    CU(cudaEventRecord(d->ev_upper, d->copy_stream));
    d->upper_pending = true;
  }
  if (sync) {  // caller's buffers are only borrowed for the call
    CU(cudaStreamSynchronize(d->stream));
    if (fork) CU(cudaStreamSynchronize(d->copy_stream));
  }
  d->have_frame = true;
  d->have_run = false;
  return LM_OK;
}

extern "C" int lm_bind_quantized_device(lm_detector* d, const uint8_t* const* d_quantized, const int* rows, const int* cols) {
  if (d && d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  if (!d || !d_quantized || !rows || !cols) return fail(LM_E_INVALID, "null argument");
  CU(cudaSetDevice(d->device));
  int rc = check_frame_dims(d, rows, cols);
  if (rc) return rc;
  rc = size_levels(d, rows, cols, false);
  if (rc) return rc;
  for (int l = 0; l < d->L; ++l)
    for (int m = 0; m < d->M; ++m) {
      if (!d_quantized[l * d->M + m]) return fail(LM_E_INVALID, "d_quantized[%d] is null", l * d->M + m);
      d->lv[l].q_src[m] = d_quantized[l * d->M + m];
    }
  if (d->upper_pending) CU(cudaStreamWaitEvent(d->stream, d->ev_upper, 0));  // an earlier upload nobody consumed
  d->upper_pending = false;
  d->have_frame = true;
  d->have_run = false;
  return LM_OK;
}

// ---- GPU quantization front-end: Detector::match's modality processing (LL.cpp:1709-1741) -------------
extern "C" int lm_upload_images(lm_detector* d, const uint8_t* rgb, const uint16_t* depth, int rows, int cols,
                                const uint8_t* mask_color, const uint8_t* mask_depth) {
  if (!d || !rgb || !depth) return fail(LM_E_INVALID, "null argument");
  if (d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  CU(cudaSetDevice(d->device));
  int lrows[LM_MAX_LEVELS], lcols[LM_MAX_LEVELS];
  for (int l = 0; l < d->L; ++l) {
    lrows[l] = l ? lrows[l - 1] / 2 : rows;  // Size(src.cols / 2, src.rows / 2), LL.cpp:564, 866
    lcols[l] = l ? lcols[l - 1] / 2 : cols;
  }
  int rc = check_frame_dims(d, lrows, lcols);
  if (rc) return rc;
  rc = size_levels(d, lrows, lcols, true);
  if (rc) return rc;
  cudaStream_t st = d->stream;
  if (d->upper_pending) CU(cudaStreamWaitEvent(st, d->ev_upper, 0));  // an earlier upload nobody consumed
  if (!d->fe_lut) {
    // NORMAL_LUT[.][vy][vx] of normal_lut.i: 45-degree sector (offset by half a sector) of atan2(vy-10, vx-10);
    // the rule reproduces all 8000 entries of the reference table (tests/test_frontend.py)
    uint8_t lut[400];
    for (int vy = 0; vy < 20; ++vy)
      for (int vx = 0; vx < 20; ++vx) {
        double a = atan2((double)(vy - 10), (double)(vx - 10)) * 180.0 / 3.14159265358979323846;
        a = fmod(a + 360.0, 360.0);
        lut[vy * 20 + vx] = (uint8_t)(1u << (((int)(fmod(a + 22.5, 360.0) / 45.0)) % 8));
      }
    CU(cudaMemcpyToSymbolAsync(c_normal_lut, lut, sizeof(lut), 0, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    d->fe_lut = true;
  }
  for (int l = 0; l < d->L; ++l) {
    lm_detector::FeLevel& f = d->fe[l];
    if (f.rows != lrows[l] || f.cols != lcols[l]) {
      cudaFree(f.src); cudaFree(f.qun); cudaFree(f.strong); cudaFree(f.normal); cudaFree(f.mask[0]); cudaFree(f.mask[1]);
      f = lm_detector::FeLevel();
      f.rows = lrows[l]; f.cols = lcols[l];
      const size_t n = (size_t)f.rows * f.cols;
      CU(cudaMalloc(&f.src, n * 3)); CU(cudaMalloc(&f.qun, n)); CU(cudaMalloc(&f.strong, n)); CU(cudaMalloc(&f.normal, n));
      CU(cudaMalloc(&f.mask[0], n)); CU(cudaMalloc(&f.mask[1], n));
      if (l == 0) {
        cudaFree(d->fe_depth); cudaFree(d->fe_nraw);
        CU(cudaMalloc(&d->fe_depth, n * 2)); CU(cudaMalloc(&d->fe_nraw, n));
      }
    }
  }
  const size_t n0 = (size_t)rows * cols;
  CU(cudaMemcpyAsync(d->fe[0].src, rgb, n0 * 3, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(d->fe_depth, depth, n0 * 2, cudaMemcpyHostToDevice, st));
  const uint8_t* masks[2] = {mask_color, mask_depth};
  for (int m = 0; m < 2; ++m)
    if (masks[m]) CU(cudaMemcpyAsync(d->fe[0].mask[m], masks[m], n0, cudaMemcpyHostToDevice, st));
  auto grid2 = [](int w, int h) { return dim3((unsigned)((w + 31) / 32), (unsigned)((h + 7) / 8)); };
  for (int l = 0; l < d->L; ++l) {
    lm_detector::FeLevel& f = d->fe[l];
    LevelHost& lv = d->lv[l];
    if (l > 0) {
      lm_detector::FeLevel& up = d->fe[l - 1];
      CU(launch_pdl(k_fe_pyrdown, grid2(f.cols, f.rows), dim3(256), 0, st, (const uint8_t*)up.src, up.rows, up.cols, f.src, f.rows, f.cols));
      for (int m = 0; m < 2; ++m)
        if (masks[m])
          CU(launch_pdl(k_fe_decimate, grid2(f.cols, f.rows), dim3(256), 0, st, (const uint8_t*)up.mask[m], up.cols, f.mask[m], f.rows,
                        f.cols, (const uint8_t*)nullptr, (uint8_t*)nullptr));
      d->launches += 1 + (masks[0] ? 1 : 0) + (masks[1] ? 1 : 0);
    }
    // colour: weak threshold 10 -> gate on squared magnitude > 100 (ColorGradient(10, nf, 55), LL.cpp:1687)
    CU(launch_pdl(k_fe_gradient, grid2(f.cols, f.rows), dim3(FE_TW, FE_TH), 0, st, (const uint8_t*)f.src, f.rows, f.cols, 100, f.qun, f.strong,
                  (int32_t*)nullptr));
    CU(launch_pdl(k_fe_hysteresis, grid2(f.cols, f.rows), dim3(256), 0, st, (const uint8_t*)f.qun, (const uint8_t*)f.strong,
                  (const uint8_t*)(masks[0] ? f.mask[0] : nullptr), f.rows, f.cols, lv.d_q[0]));
    d->launches += 2;
    // depth: DepthNormal(2000, 50, nf, 2), LL.cpp:1688; upper levels decimate the LABELS (LL.cpp:865-868)
    if (l == 0) {
      CU(launch_pdl(k_fe_normals, grid2(f.cols, f.rows), dim3(256), 0, st, (const uint16_t*)d->fe_depth, f.rows, f.cols, 2000, 50, d->fe_nraw));
      CU(launch_pdl(k_fe_median, grid2(f.cols, f.rows), dim3(256), 0, st, (const uint8_t*)d->fe_nraw,
                    (const uint8_t*)(masks[1] ? f.mask[1] : nullptr), f.rows, f.cols, f.normal, lv.d_q[1]));
      d->launches += 2;
    } else {
      lm_detector::FeLevel& up = d->fe[l - 1];
      CU(launch_pdl(k_fe_decimate, grid2(f.cols, f.rows), dim3(256), 0, st, (const uint8_t*)up.normal, up.cols, f.normal, f.rows, f.cols,
                    (const uint8_t*)(masks[1] ? f.mask[1] : nullptr), lv.d_q[1]));
      d->launches += 1;
    }
    lv.q_src[0] = lv.d_q[0];
    lv.q_src[1] = lv.d_q[1];
  }
  CU(cudaStreamSynchronize(st));  // the caller's images are only borrowed for the call
  CU(cudaGetLastError());
  d->upper_pending = false;
  d->have_frame = true;
  d->have_run = false;
  return LM_OK;
}

static LevelDev level_dev(const LevelHost& h) {
  LevelDev v;
  v.lm = h.d_lm; v.T = h.T; v.rows = h.rows; v.cols = h.cols; v.Wd = h.Wd; v.Hd = h.Hd; v.plane = h.plane;
  v.off = h.T / 2 + (h.T % 2 - 1);
  v.mod_stride = h.mod_stride;
  return v;
}


// K1 launch plan: block ranges per level (lowest level first), kernel variant and shared memory.  planes_level >= 0: that
// level is built in planes mode (column-major H-planes only, no byte linear memories; see spread_planes_block).
struct K1Plan {
  LinMemParams p;
  bool band = false;
  size_t smem = 0;
  int blocks = 0;
};

static void plan_k1(lm_detector* d, int planes_level, bool with_bit_planes, K1Plan& k) {
  LinMemParams& p = k.p;
  memset(&p, 0, sizeof(p));
  p.L = d->L; p.M = d->M; p.block_offset = 0;
  bool band = true;
  size_t smem = 0;
  for (int l = 0; l < d->L; ++l) {
    const LevelHost& lv = d->lv[l];
    band = band && (lv.cols % 4 == 0) && (lv.Wd % 4 == 0) && (lv.plane % 4 == 0);
    // the most segments (a divisor of Wd / 4, so that a segment keeps a multiple of 4 positions) that still
    // leave every thread of the CTA one 4-position group of one grid: equal, light CTAs on every level
    int nseg = 1;
    if (lv.Wd % 4 == 0)
      for (int j = 1; j <= 16 && j <= lv.Wd / 4; ++j)
        if ((lv.Wd / 4) % j == 0 && (lv.T * lv.T * (lv.Wd / 4)) / j >= 128) nseg = j;
    p.lv[l].nseg = nseg;
    const size_t wp = (size_t)((lv.Wd / nseg * lv.T + lv.T + 3 + 4) & ~3);
    size_t need = wp * (size_t)(2 * (2 * lv.T - 1) + lv.T);
    if (l == planes_level) {
      // positions per segment: T*T * pseg = one (grid, column) item per thread of the 128-thread CTA where possible
      int pseg = 4;
      for (int c : {32, 16, 8})
        if (lv.Wd % c == 0 && lv.T * lv.T * c <= 128) { pseg = c; break; }
      p.lv[l].pseg = pseg;
      const size_t wpp = (size_t)((pseg * lv.T + lv.T + 3 + 4) & ~3);
      need = wpp * (size_t)(2 * (16 * lv.T + lv.T - 1) + 16 * lv.T);
    }
    smem = std::max(smem, need);
  }
  band = band && smem <= LM_BAND_SMEM_LIMIT;
  int blocks = 0;
  // block index order = lowest level first: its CTAs are the heavy ones (T*T = 64 grids per position row plus
  // the bit-plane atomics), started last they would be the tail of the launch
  for (int l = d->L - 1; l >= 0; --l) {
    const LevelHost& lv = d->lv[l];
    LinMemLevel& q = p.lv[l];
    for (int m = 0; m < d->M; ++m) q.q[m] = lv.q_src[m];
    q.lm = lv.d_lm; q.bp = with_bit_planes ? lv.d_bp : nullptr; q.lbw = lv.lbw;
    q.T = lv.T; q.rows = lv.rows; q.cols = lv.cols; q.Wd = lv.Wd; q.Hd = lv.Hd; q.plane = lv.plane;
    q.mod_stride = lv.mod_stride;
    q.rp = nullptr; q.nyb = 0;
    if (band && l == planes_level) {
      q.rp = d->d_rp; q.nyb = d->rp_nyb;
      blocks += ((lv.Hd + 15) / 16) * (lv.Wd / q.pseg);
    } else {
      blocks += band ? lv.Hd * q.nseg : (lv.T * lv.T * lv.plane + 255) / 256;
    }
    q.block_end = blocks;
  }
  k.band = band;
  k.smem = smem;
  k.blocks = blocks;
}

static int launch_k1(lm_detector* d, const K1Plan& k, int first_block, int n_blocks) {
  if (n_blocks <= 0) return LM_OK;
  LinMemParams p = k.p;
  p.block_offset = first_block;
  if (k.band) CU(launch_pdl(k_linear_memories_band, dim3((unsigned)n_blocks, (unsigned)d->M), dim3(128), k.smem, d->stream, p));
  else CU(launch_pdl(k_linear_memories, dim3((unsigned)n_blocks, (unsigned)d->M), dim3(256), 0, d->stream, p));
  ++d->launches;
  return LM_OK;
}

// Which refinement path the current bank / shard / frame size take (see enqueue_stages).
static bool use_filter(const lm_detector* d) { return d->filter_ok && d->d_rp != nullptr && d->d_finfo != nullptr; }
static bool use_bits(const lm_detector* d) { return use_filter(d) && d->L == 2; }
// level built in planes mode by K1, or -1: only when nothing reads that level's byte linear memories
static int planes_level(const lm_detector* d) { return use_bits(d) && d->shard_all_eligible ? d->L - 2 : -1; }

// Enqueue every GPU stage of one frame on the detector's stream; no host synchronisation.
static int enqueue_stages(lm_detector* d, float threshold, bool refine_only) {
  const int n_work = (int)d->shard_count;
  const LevelHost& low = d->lv[d->L - 1];
  cudaStream_t st = d->stream;
  // fused multi-GPU exchange: k_refine appends into block [frame slot][rank] of every rank's buffer
  PeerExchange px;
  memset(&px, 0, sizeof(px));
  lm_result_header* px_block = nullptr;
  if (d->px_rank >= 0) {
    if (refine_only) return fail(LM_E_STATE, "refinement re-run is not available with a connected peer exchange");
    ++d->px_seq;
    px = d->h_px;
    px_block = reinterpret_cast<lm_result_header*>(d->px_buf + (size_t)(d->px_seq & 1) * px.slot_bytes +
                                                   (size_t)px.rank * px.block_bytes);
  }
  if (d->timing && !refine_only) {
    d->ev = d->tev.data() + LM_TEV * (size_t)(d->timing_runs % (int64_t)(d->tev.size() / LM_TEV));
    ++d->timing_runs;
  }
  K1Plan k1;
  int k1_done = 0;
  if (!refine_only) {
    if (d->timing) CU(cudaEventRecord(d->ev[0], st));
    // K1: one launch for every level and modality.  Bit-planes are OR-ed in: zero at allocation, re-zeroed by the
    // refinement kernel after every frame.  With a host upload in flight (upper levels still on the copy stream) the
    // launch is split: the lowest level now, the levels above it behind the coarse scan, once their images have landed.
    plan_k1(d, planes_level(d), true, k1);
    d->last_planes_level = k1.band ? planes_level(d) : -1;
    k1_done = d->upper_pending ? k1.p.lv[d->L - 1].block_end : k1.blocks;
    int rc1 = launch_k1(d, k1, 0, k1_done);
    if (rc1) return rc1;
    if (d->timing) CU(cudaEventRecord(d->ev[1], st));
    // K2
    bool scan_fused = false;
    if (d->n_items_bits > 0) {
      BitScanParams bp;
      bp.bp = low.d_bp; bp.bp_words = (uint32_t)((size_t)d->M * 8 * low.lbw + low.bp_zero);  // planes + the zero words
      bp.lbw = low.lbw; bp.plane = low.plane; bp.nwords = low.nwords;
      bp.tslot = d->d_tslot; bp.fdesc4 = d->d_fdesc4; bp.k2info = d->d_k2info; bp.work = d->d_work;
      bp.zero_off = (uint32_t)((size_t)d->M * 8 * low.lbw) * 4u;
      bp.items = d->d_items_bits; bp.n_items = d->n_items_bits;
      bp.S = d->S; bp.M = d->M; bp.slot_low = (d->L - 1) * d->M;
      bp.threshold = threshold;
      bp.mask = d->d_mask; bp.raw = d->d_raw; bp.cnt = d->d_cnt;
      const bool fuse_scan = d->n_items_bytes == 0;
      scan_fused = fuse_scan;
      bp.off = fuse_scan ? d->d_off : nullptr;
      bp.n_work = n_work;
      bp.hdr = px.world > 0 ? px_block : d->d_res;
      bp.capacity = (int)(px.world > 0 ? d->px_cap : d->res_cap);
      bp.shard = d->shard_index;
      bp.counters = d->d_counters;
      bp.queue = d->d_queue;
      bp.ticket = reinterpret_cast<int*>(d->d_counters + 3);
      const size_t plane_bytes = ((size_t)bp.bp_words * 4 + 15) & ~(size_t)15;
      const bool smem = plane_bytes <= LM_BITS_SMEM_LIMIT;
      // tasks of 32 words (full rounds + packed remainders).  One task per warp (or per TEAM of S warps when the shard has
      // fewer tasks than the GPU has warp slots: the team deals the task's features, so the kernel's latency follows the
      // shard) and one round per CTA: the CTA size follows the shard, so a small shard spreads over all SMs.
      // (upper estimate: every template counted with all nwords words; the kernel tabulates the exact tasks.  The sizes
      // below are the ones the round's records were measured with: N=1 24 warps x 148 CTAs, one round; N=8 S=4, 16 x 116)
      const long long tasks = (long long)d->n_items_bits * (low.nwords / 32) +
                              ((long long)d->n_items_bits * (low.nwords % 32) + 31) / 32;
      const long long slots = (long long)d->sm_count * (LM_PACK_THREADS / 32);
      const size_t part_room = LM_K2_SMEM_MAX - (smem ? plane_bytes : (size_t)LM_K2_SMEM_MAX - 64 * 1024);
      int S = 1;
      while (S < 8 && tasks * (S * 2) <= slots) {
        const int S2 = S * 2;
        long long w2 = (tasks * S2 + d->sm_count - 1) / d->sm_count;
        w2 = std::min<long long>(LM_PACK_THREADS / 32, std::max<long long>(std::max(4, S2), (w2 + S2 - 1) / S2 * S2));
        if ((size_t)(w2 / S2) * (S2 - 1) * 16 * 32 * 4 > part_room) break;
        S = S2;
      }
      bp.split = S;
      const int unit = std::max(4, S);
      int wpc = (int)((tasks * S + d->sm_count - 1) / d->sm_count);
      wpc = std::min(LM_PACK_THREADS / 32, std::max(unit, (wpc + unit - 1) / unit * unit));
      const int grid = (int)std::max<long long>(1, std::min<long long>(d->sm_count, (tasks * S + wpc - 1) / wpc));
      const size_t smem_bytes = (smem ? plane_bytes : 0) + (size_t)(wpc / S) * (S - 1) * 16 * 32 * 4;
      cudaError_t e = cudaSuccess;
      if (smem) {
        e = launch_pdl(k_coarse_packed<true>, dim3(grid), dim3(wpc * 32), smem_bytes, st, bp);
      } else {
        e = launch_pdl(k_coarse_packed<false>, dim3(grid), dim3(wpc * 32), smem_bytes, st, bp);
      }
      if (e != cudaSuccess) return fail(LM_E_CUDA, "k_coarse_packed launch failed: %s", cudaGetErrorString(e));
      ++d->launches;
    }
    if (d->n_items_bytes > 0) {
      ByteScanParams sp;
      sp.lv = level_dev(low);
      sp.tslot = d->d_tslot; sp.fbase = d->d_fbase; sp.fxy = d->d_fxy; sp.work = d->d_work;
      sp.items = d->d_items_bytes;
      sp.S = d->S; sp.M = d->M; sp.slot_low = (d->L - 1) * d->M; sp.nwords = low.nwords;
      sp.threshold = threshold;
      sp.mask = d->d_mask; sp.raw = d->d_raw; sp.cnt = d->d_cnt;
      int bs = ((low.plane + 3) / 4 + 31) / 32 * 32;
      bs = std::max(32, std::min(bs, 1024));
      CU(launch_pdl(k_coarse_bytes, dim3(d->n_items_bytes), dim3(bs), 0, st, sp));
      ++d->launches;
    }
    if (d->timing) CU(cudaEventRecord(d->ev[2], st));
    if (!scan_fused) {
      CU(launch_pdl(k_scan_counts, dim3(1), dim3(1024), 0, st, d->d_cnt, d->d_off, n_work,
                    px.world > 0 ? px_block : d->d_res, (int)(px.world > 0 ? d->px_cap : d->res_cap), d->shard_index,
                    d->d_counters, d->d_queue));
      ++d->launches;
    }
    if (d->timing) CU(cudaEventRecord(d->ev[3], st));
    if (k1_done < k1.blocks) {  // the upper levels' linear memories, behind their images
      CU(cudaStreamWaitEvent(st, d->ev_upper, 0));
      int rc2 = launch_k1(d, k1, k1_done, k1.blocks - k1_done);
      if (rc2) return rc2;
    }
    d->upper_pending = false;
  }
  if (refine_only) {
    CU(cudaMemsetAsync(d->d_counters, 0, 8 * sizeof(unsigned long long), st));  // [3] (the coarse scan's ticket) is 0 between launches
    CU(cudaMemsetAsync(d->d_queue, 0, 4 * sizeof(int), st));
    CU(cudaMemsetAsync(&d->d_res->count, 0, sizeof(int32_t), st));
  }
  const bool filter = use_filter(d);
  // two pyramid levels: the filtered level is the last one, its survivors are finished bit-sliced (k_refine_bits)
  const bool bits_mode = use_bits(d);
  const LevelHost& lref = d->lv[d->L >= 2 ? d->L - 2 : 0];
  {
    // ordered candidate list (+ the filter's H-planes of the first refined level)
    PrepParams pp;
    pp.off = d->d_off; pp.mask = d->d_mask;
    pp.n_work = n_work; pp.nwords = low.nwords;
    pp.cand = d->d_cand; pp.cand_cap = (int)d->cand_cap;
    pp.expand_blocks = std::max(1, std::min((n_work + 7) / 8, d->sm_count * 8));
    pp.lm = lref.d_lm; pp.rp = (filter && d->last_planes_level < 0) ? d->d_rp : nullptr;  // else: K1 wrote the planes
    pp.Wd = lref.Wd; pp.Hd = lref.Hd; pp.plane = lref.plane; pp.nyb = d->rp_nyb;
    pp.n_pb = d->M * 8 * lref.T * lref.T;
    const int plane_blocks = pp.rp ? (int)(((size_t)pp.n_pb * pp.nyb * (pp.Wd / 4) + 255) / 256) : 0;
    CU(launch_pdl(k_refine_prep, dim3((unsigned)(pp.expand_blocks + plane_blocks)), dim3(256), 0, st, pp));
    ++d->launches;
  }
  if (d->timing && !refine_only) CU(cudaEventRecord(d->ev[4], st));
  if (filter) {
    FilterParams fp;
    fp.rp = d->d_rp; fp.Wd = lref.Wd;
    fp.rdesc = d->d_rdesc; fp.finfo = d->d_finfo;
    fp.low = level_dev(low); fp.ref = level_dev(lref);
    fp.cand = d->d_cand; fp.off = d->d_off; fp.n_work = n_work; fp.cand_cap = (int)d->cand_cap;
    fp.surv = d->d_surv; fp.surv2 = bits_mode ? d->d_surv2 : nullptr; fp.queue = d->d_queue; fp.counters = d->d_counters;
    CU(launch_pdl(k_refine_filter_w, dim3((unsigned)(d->sm_count * LM_FILTER_MIN_CTAS)), dim3(256), 0, st, fp));
    ++d->launches;
  }
  if (d->timing && !refine_only) CU(cudaEventRecord(d->ev[5], st));
  const bool bytes_pass = !bits_mode || !d->shard_all_eligible;  // byte-wise exact refinement needed for this shard
  if (bits_mode) {
    // exact refinement of the survivors, bit-sliced, from the same H-planes
    RefineBitsParams bq;
    bq.rp = d->d_rp; bq.Wd = lref.Wd; bq.label_stride = lref.T * lref.T * d->rp_nyb * lref.Wd;
    bq.rdesc = d->d_rdesc; bq.rlab = d->d_rlab; bq.finfo = d->d_finfo;
    bq.low = level_dev(low); bq.ref = level_dev(lref);
    bq.cand = d->d_cand; bq.off = d->d_off; bq.n_work = n_work; bq.cand_cap = (int)d->cand_cap;
    bq.surv = d->d_surv; bq.queue = d->d_queue;
    bq.threshold = threshold;
    bq.work_begin = (int)d->work_base; bq.work_stride = (int)d->work_stride;
    bq.hdr = px.world > 0 ? px_block : d->d_res;
    bq.capacity = (int32_t)(px.world > 0 ? d->px_cap : d->res_cap);
    bq.px = px.world > 0 ? d->d_px : nullptr; bq.px_seq = d->px_seq;
    bq.publish = bytes_pass ? 0 : 1;
    bq.counters = d->d_counters;
    bq.bp_clear = low.d_bp; bq.bp_words = low.d_bp ? (uint32_t)((size_t)d->M * 8 * low.lbw) : 0u;
    CU(launch_pdl(k_refine_bits, dim3((unsigned)(d->sm_count * 6)), dim3(256), 0, st, bq));
    ++d->launches;
  }
  if (bytes_pass) {
    // persistent grid: the candidate total is read on the device (no host round trip)
    RefineParams rp;
    for (int l = 0; l < d->L; ++l) rp.lv[l] = level_dev(d->lv[l]);
    rp.tslot = d->d_tslot; rp.fbase = d->d_fbase; rp.fxy = d->d_fxy; rp.work = d->d_work;
    rp.off = d->d_off; rp.cand = d->d_cand; rp.cand_cap = (int)d->cand_cap; rp.raw = d->d_raw;
    rp.surv = filter ? (bits_mode ? d->d_surv2 : d->d_surv) : nullptr; rp.queue = d->d_queue;
    rp.surv_slot = bits_mode ? 2 : 1;
    rp.publish = 1;
    rp.n_work = n_work; rp.L = d->L; rp.S = d->S; rp.M = d->M;
    rp.work_begin = (int)d->work_base;
    rp.work_stride = (int)d->work_stride;
    rp.threshold = threshold;
    rp.hdr = d->d_res; rp.capacity = (int32_t)d->res_cap;
    rp.px = px.world > 0 ? d->d_px : nullptr;
    rp.px_seq = d->px_seq;
    if (px.world > 0) {
      rp.hdr = px_block;
      rp.capacity = (int32_t)d->px_cap;
    }
    rp.counters = d->d_counters;
    rp.safe = d->d_safe; rp.galign = d->d_galign;
    rp.bp_clear = bits_mode ? nullptr : low.d_bp;
    rp.bp_words = (!bits_mode && low.d_bp) ? (uint32_t)((size_t)d->M * 8 * low.lbw) : 0u;
    // 4 CTAs are resident per SM (64 registers x 256 threads); 16 per SM = four waves of equal shares, which
    // balances the very uneven per-candidate cost (row-wise early exit) better than one persistent wave
    // (measured: 4 -> 251 us, 8 -> 241, 12..32 -> 229)
    // behind the filter the work items are its few survivors: four warps share one (k_refine<true>)
    if (filter) CU(launch_pdl(k_refine<true>, dim3(d->sm_count * 16), dim3(256), 0, st, rp));
    else CU(launch_pdl(k_refine<false>, dim3(d->sm_count * 16), dim3(256), 0, st, rp));
    ++d->launches;
  }
  if (px.world > 0) {
    // collector: waits for all ranks' frame flags, packs the blocks into the ordinary result block
    CU(launch_pdl(k_peer_collect, dim3(1), dim3(1024), 0, st, px, d->px_seq, (int32_t)d->px_cap, d->d_res, (int32_t)d->res_cap,
                  d->d_counters + 2, d->px_timeout_ns));
    ++d->launches;
  }
  if (d->timing && !refine_only) CU(cudaEventRecord(d->ev[6], st));
  return LM_OK;
}

// header + the first records in one copy; the common case needs no second round trip
#define LM_FIRST_FETCH 4096

static int enqueue_readback(lm_detector* d) {
  cudaStream_t st = d->stream;
  const int64_t first = std::min<int64_t>(d->res_cap, LM_FIRST_FETCH);
  CU(cudaMemcpyAsync(d->h_res, d->d_res, sizeof(lm_result_header) + sizeof(lm_record) * (size_t)first,
                     cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(d->h_counters, d->d_counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  d->h_valid = first;
  return LM_OK;
}

static int ensure_run_buffers(lm_detector* d) {
  const int64_t n_work = d->shard_count;
  const LevelHost& low = d->lv[d->L - 1];
  const size_t need_m = (size_t)std::max<int64_t>(n_work, 1) * low.nwords;
  if (need_m > d->mask_elems) {
    cudaFree(d->d_mask);
    d->d_mask = nullptr;
    d->mask_elems = need_m;
    CU(cudaMalloc(&d->d_mask, sizeof(uint32_t) * need_m));
  }
  const size_t need_r = (size_t)std::max<int64_t>(n_work, 1) * low.plane;
  if (need_r > d->raw_elems) {
    cudaFree(d->d_raw);
    d->d_raw = nullptr;
    d->raw_elems = need_r;
    CU(cudaMalloc(&d->d_raw, sizeof(uint16_t) * need_r));
  }
  // ordered candidate list + survivor list: worst case one entry per (template, cell); capped (a frame that overflows
  // the cap is redone from k_refine_prep with a larger list, like the result block)
  {
    const int64_t worst = std::max<int64_t>(n_work, 1) * low.plane;
    const int64_t want = std::min<int64_t>(worst, std::max<int64_t>(LM_CAND_DEFAULT, d->cand_need));
    if (want > d->cand_cap) {
      cudaFree(d->d_cand); cudaFree(d->d_surv); cudaFree(d->d_surv2);
      d->d_cand = nullptr; d->d_surv = nullptr; d->d_surv2 = nullptr;
      d->cand_cap = want;
      CU(cudaMalloc(&d->d_cand, sizeof(uint2) * (size_t)want));
      CU(cudaMalloc(&d->d_surv, sizeof(uint32_t) * (size_t)want));
      CU(cudaMalloc(&d->d_surv2, sizeof(uint32_t) * (size_t)want));
    }
  }
  if (d->px_rank >= 0 && d->res_external) return fail(LM_E_STATE, "lm_set_result_buffer and a connected peer exchange exclude each other");
  if (d->px_rank >= 0 && d->res_cap_own < d->px_cap * d->px_world) {
    cudaFree(d->d_res_own);
    d->d_res_own = nullptr;
    d->res_cap_own = d->px_cap * d->px_world;
    CU(cudaMalloc(&d->d_res_own, sizeof(lm_result_header) + sizeof(lm_record) * (size_t)d->res_cap_own));
  }
  if (!d->res_external) {
    if (d->res_cap_own == 0) {
      d->res_cap_own = 1 << 16;
      CU(cudaMalloc(&d->d_res_own, sizeof(lm_result_header) + sizeof(lm_record) * (size_t)d->res_cap_own));
    }
    d->d_res = d->d_res_own;
    d->res_cap = d->res_cap_own;
  }
  if (d->h_res_cap < d->res_cap) {
    cudaFreeHost(d->h_res);
    d->h_res = nullptr;
    d->h_res_cap = d->res_cap;
    CU(cudaMallocHost(&d->h_res, sizeof(lm_result_header) + sizeof(lm_record) * (size_t)d->h_res_cap));
  }
  return LM_OK;
}

// More kept records than slots in the internal result block: grow it and redo the refinement stage only (the coarse
// outputs of the frame are still in place).  The header travels through a stack copy (the pinned staging block is
// reallocated by ensure_run_buffers) with the new capacity patched in.
static int grow_and_rerun(lm_detector* d) {
  lm_result_header hdr = *d->h_res;
  const bool more_records = (int64_t)hdr.count > d->res_cap;
  const bool more_cands = (int64_t)hdr.coarse_candidates > d->cand_cap;
  if (more_records && d->res_external)
    return fail(LM_E_CAPACITY, "%d records kept, caller's result buffer holds %lld", hdr.count, (long long)d->res_cap);
  if (d->px_rank >= 0)
    return fail(LM_E_CAPACITY, "%d records kept of %d candidates: beyond the result block (%lld) or the candidate list (%lld) of a "
                "connected peer exchange", hdr.count, hdr.coarse_candidates, (long long)d->res_cap, (long long)d->cand_cap);
  CU(cudaStreamSynchronize(d->stream));
  if (more_cands) d->cand_need = (int64_t)hdr.coarse_candidates;  // ensure_run_buffers reallocates the lists
  if (more_records || (more_cands && !d->res_external)) {
    // with a truncated candidate list the kept count is a lower bound: leave room, a second pass grows again if needed
    const int64_t want = std::max<int64_t>((int64_t)hdr.count * 2, d->res_cap_own);
    if (want > d->res_cap_own) {
      cudaFree(d->d_res_own);
      d->d_res_own = nullptr;
      d->res_cap_own = want;
      CU(cudaMalloc(&d->d_res_own, sizeof(lm_result_header) + sizeof(lm_record) * (size_t)d->res_cap_own));
    }
  }
  int rc = ensure_run_buffers(d);
  if (rc) return rc;
  hdr.capacity = (int32_t)d->res_cap;
  hdr.count = 0;
  CU(cudaMemcpy(d->d_res, &hdr, sizeof(hdr), cudaMemcpyHostToDevice));
  rc = enqueue_stages(d, d->last_threshold, true);
  if (rc) return rc;
  rc = enqueue_readback(d);
  if (rc) return rc;
  CU(cudaStreamSynchronize(d->stream));
  CU(cudaGetLastError());
  return LM_OK;
}

extern "C" int lm_enqueue(lm_detector* d, float threshold) {
  if (d && d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  if (!d) return fail(LM_E_INVALID, "null detector");
  if (!d->have_frame) return fail(LM_E_STATE, "no frame uploaded");
  if (d->S == 0) return fail(LM_E_STATE, "no template bank loaded");
  CU(cudaSetDevice(d->device));
  int rc = prepare_bank(d);
  if (rc) return rc;
  rc = prepare_work(d);
  if (rc) return rc;
  rc = ensure_run_buffers(d);
  if (rc) return rc;
  d->last_threshold = threshold;
  rc = filter_thresholds(d, threshold);
  if (rc) return rc;
  return enqueue_stages(d, threshold, false);
}

extern "C" int lm_prepare(lm_detector* d) {
  if (d && d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  if (!d) return fail(LM_E_INVALID, "null detector");
  if (!d->have_frame) return fail(LM_E_STATE, "no frame uploaded (the frame size decides the feature addresses)");
  if (d->S == 0) return fail(LM_E_STATE, "no template bank loaded");
  CU(cudaSetDevice(d->device));
  int rc = prepare_bank(d);
  if (rc) return rc;
  rc = prepare_work(d);
  if (rc) return rc;
  return ensure_run_buffers(d);
}

extern "C" int lm_complete(lm_detector* d) {
  if (d && d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  if (!d) return fail(LM_E_INVALID, "null detector");
  CU(cudaSetDevice(d->device));
  int rc = enqueue_readback(d);
  if (rc) return rc;
  CU(cudaStreamSynchronize(d->stream));
  CU(cudaGetLastError());
  if (d->px_rank >= 0) {
    if (d->h_counters[2] == 1)
      return fail(LM_E_STATE, "peer exchange: a rank did not publish frame %d within %llu ms (or an earlier frame already timed out "
                  "on this device); disconnect and reconnect the exchange", d->px_seq, d->px_timeout_ns / 1000000ull);
    if (d->h_counters[2] == 2)
      return fail(LM_E_CAPACITY, "peer exchange: a shard kept more than %lld records (capacity given to lm_peer_export)",
                  (long long)d->px_cap);
  }
  for (int pass = 0; pass < 3 && ((int64_t)d->h_res->count > d->res_cap || (int64_t)d->h_res->coarse_candidates > d->cand_cap); ++pass) {
    rc = grow_and_rerun(d);
    if (rc) return rc;
  }
  d->have_run = true;
  return LM_OK;
}

extern "C" int lm_run(lm_detector* d, float threshold) {
  int rc = lm_enqueue(d, threshold);
  if (rc) return rc;
  return lm_complete(d);
}

extern "C" int lm_set_result_buffer(lm_detector* d, void* d_block, int64_t capacity_records) {
  if (d && d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  if (!d) return fail(LM_E_INVALID, "null detector");
  if (d_block && capacity_records < 1) return fail(LM_E_INVALID, "capacity must be >= 1");
  if (capacity_records > 0x7FFFFFFF) return fail(LM_E_INVALID, "capacity too large");
  if (d_block && d->px_rank >= 0) return fail(LM_E_STATE, "lm_set_result_buffer and a connected peer exchange exclude each other");
  CU(cudaSetDevice(d->device));
  CU(cudaStreamSynchronize(d->stream));
  d->res_external = d_block != nullptr;
  if (d->res_external) {
    d->d_res = (lm_result_header*)d_block;
    d->res_cap = capacity_records;
  }
  d->have_run = false;
  return LM_OK;
}

static size_t peer_buffer_bytes(int world, int64_t cap) {
  return 2 * (size_t)world * (sizeof(lm_result_header) + sizeof(lm_record) * (size_t)cap) +
         sizeof(int32_t) * (2 * LM_MAX_PEERS + 4);
}

extern "C" int lm_peer_export(lm_detector* d, int world, int64_t capacity_records, uint8_t* handle_out) {
  if (d && d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  if (!d) return fail(LM_E_INVALID, "null detector");
  if (world < 1 || world > LM_MAX_PEERS) return fail(LM_E_INVALID, "world %d outside 1..%d", world, LM_MAX_PEERS);
  if (capacity_records < 1 || capacity_records > (1 << 24)) return fail(LM_E_INVALID, "capacity outside 1..2^24");
  if (peer_buffer_bytes(world, capacity_records) > 0xF0000000ull) return fail(LM_E_INVALID, "exchange buffer too large");
  CU(cudaSetDevice(d->device));
  CU(cudaStreamSynchronize(d->stream));
  peer_release(d);
  const size_t bytes = peer_buffer_bytes(world, capacity_records);
  CU(cudaMalloc(&d->px_buf, bytes));
  CU(cudaMemset(d->px_buf, 0, bytes));
  CU(cudaDeviceSynchronize());
  d->px_world = world;
  d->px_cap = capacity_records;
  d->px_seq = 0;
  {
    const int zero = 0;  // a fresh exchange starts with the device's abort flag down
    CU(cudaMemcpyToSymbol(g_px_abort, &zero, sizeof(int)));
    const char* ms = getenv("LINEMOD_B200_PEER_TIMEOUT_MS");
    const long long v = ms ? atoll(ms) : 1000;
    d->px_timeout_ns = (unsigned long long)(v < 1 ? 1 : (v > 600000 ? 600000 : v)) * 1000000ull;
  }
  if (handle_out) {
    static_assert(sizeof(cudaIpcMemHandle_t) <= LM_PEER_HANDLE_BYTES, "IPC handle size");
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, d->px_buf));
    memset(handle_out, 0, LM_PEER_HANDLE_BYTES);
    memcpy(handle_out, &h, sizeof(h));
  }
  return LM_OK;
}

extern "C" int lm_peer_base(lm_detector* d, void** base) {
  if (!d || !base) return fail(LM_E_INVALID, "null argument");
  if (!d->px_buf) return fail(LM_E_STATE, "lm_peer_export has not been called");
  *base = d->px_buf;
  return LM_OK;
}

static int peer_connect_common(lm_detector* d, int rank, int world) {
  if (d && d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  if (!d) return fail(LM_E_INVALID, "null detector");
  if (!d->px_buf) return fail(LM_E_STATE, "lm_peer_export has not been called");
  if (world != d->px_world) return fail(LM_E_INVALID, "world %d differs from the exported one (%d)", world, d->px_world);
  if (rank < 0 || rank >= world) return fail(LM_E_INVALID, "rank %d outside 0..%d", rank, world - 1);
  if (d->px_rank >= 0) return fail(LM_E_STATE, "already connected");
  if (d->res_external) return fail(LM_E_STATE, "lm_set_result_buffer and the peer exchange exclude each other");
  return LM_OK;
}

static int peer_upload_descriptor(lm_detector* d) {
  PeerExchange px;
  memset(&px, 0, sizeof(px));
  for (int r = 0; r < d->px_world; ++r) px.base[r] = d->px_base[r];
  px.world = d->px_world; px.rank = d->px_rank;
  px.block_bytes = (uint32_t)(sizeof(lm_result_header) + sizeof(lm_record) * (size_t)d->px_cap);
  px.slot_bytes = px.block_bytes * (uint32_t)d->px_world;
  px.flags_offset = 2u * px.slot_bytes;
  d->h_px = px;
  if (!d->d_px) CU(cudaMalloc(&d->d_px, sizeof(PeerExchange)));
  CU(cudaMemcpy(d->d_px, &px, sizeof(px), cudaMemcpyHostToDevice));
  return LM_OK;
}

extern "C" int lm_peer_connect(lm_detector* d, int rank, int world, const uint8_t* handles) {
  int rc = peer_connect_common(d, rank, world);
  if (rc) return rc;
  if (!handles) return fail(LM_E_INVALID, "null handles");
  CU(cudaSetDevice(d->device));
  for (int r = 0; r < world; ++r) {
    if (r == rank) { d->px_base[r] = d->px_buf; continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + (size_t)r * LM_PEER_HANDLE_BYTES, sizeof(h));
    void* ptr = nullptr;
    cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
      for (int q = 0; q < r; ++q)
        if (q != rank && d->px_base[q]) cudaIpcCloseMemHandle(d->px_base[q]);
      for (int q = 0; q < LM_MAX_PEERS; ++q) d->px_base[q] = nullptr;
      return fail(LM_E_CUDA, "cudaIpcOpenMemHandle(rank %d): %s", r, cudaGetErrorString(e));
    }
    d->px_base[r] = (uint8_t*)ptr;
  }
  d->px_ipc = true;
  d->px_rank = rank;
  d->have_run = false;
  return peer_upload_descriptor(d);
}

extern "C" int lm_peer_connect_local(lm_detector* d, int rank, int world, void* const* bases) {
  int rc = peer_connect_common(d, rank, world);
  if (rc) return rc;
  if (!bases) return fail(LM_E_INVALID, "null bases");
  CU(cudaSetDevice(d->device));
  for (int r = 0; r < world; ++r) {
    if (!bases[r]) return fail(LM_E_INVALID, "bases[%d] is null", r);
    cudaPointerAttributes at;
    CU(cudaPointerGetAttributes(&at, bases[r]));
    if (at.type != cudaMemoryTypeDevice) return fail(LM_E_INVALID, "bases[%d] is not device memory", r);
    if (at.device != d->device) {
      int can = 0;
      CU(cudaDeviceCanAccessPeer(&can, d->device, at.device));
      if (!can) return fail(LM_E_STATE, "device %d cannot access device %d", d->device, at.device);
      cudaError_t e = cudaDeviceEnablePeerAccess(at.device, 0);
      if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(LM_E_CUDA, "cudaDeviceEnablePeerAccess: %s", cudaGetErrorString(e));
      (void)cudaGetLastError();
    }
    d->px_base[r] = (uint8_t*)bases[r];
  }
  d->px_base[rank] = d->px_buf;
  d->px_ipc = false;
  d->px_rank = rank;
  d->have_run = false;
  return peer_upload_descriptor(d);
}

extern "C" int lm_peer_disconnect(lm_detector* d) {
  if (!d) return fail(LM_E_INVALID, "null detector");
  if (d->device < 0) return LM_OK;
  CU(cudaSetDevice(d->device));
  CU(cudaStreamSynchronize(d->stream));
  peer_release(d);
  d->have_run = false;
  return LM_OK;
}

extern "C" int lm_device_result(lm_detector* d, void** d_block, int64_t* capacity_records) {
  if (!d) return fail(LM_E_INVALID, "null detector");
  if (!d->d_res) return fail(LM_E_STATE, "no result block yet (call lm_enqueue / lm_run first)");
  if (d_block) *d_block = d->d_res;
  if (capacity_records) *capacity_records = d->res_cap;
  return LM_OK;
}

static bool record_order(const lm_record& a, const lm_record& b) {
  if (a.work != b.work) return a.work < b.work;
  return a.seq < b.seq;
}

// (work, seq) order = the order in which the reference's loops produce the matches (LL.cpp:1797-1939).  The
// records arrive grouped by nothing (atomic append) but with few per template: one counting pass over `work`
// and an insertion sort by `seq` inside each template's run -- O(n + templates) instead of n log n compares.
static void order_records(lm_detector* d, lm_record* r, int64_t n) {
  if (n < 2 || std::is_sorted(r, r + n, record_order)) return;
  const int64_t n_sel = (int64_t)d->sel.size();
  bool in_range = n_sel > 0 && n_sel <= (1 << 22);
  for (int64_t i = 0; in_range && i < n; ++i) in_range = r[i].work >= 0 && r[i].work < n_sel;
  if (!in_range) {
    std::sort(r, r + n, record_order);
    return;
  }
  std::vector<int32_t>& cnt = d->order_cnt;
  cnt.assign((size_t)n_sel + 1, 0);
  for (int64_t i = 0; i < n; ++i) ++cnt[(size_t)r[i].work + 1];
  for (int64_t w = 0; w < n_sel; ++w) cnt[(size_t)w + 1] += cnt[(size_t)w];
  std::vector<lm_record>& tmp = d->order_tmp;
  tmp.resize((size_t)n);
  for (int64_t i = 0; i < n; ++i) {  // place, keeping each run sorted by seq
    const int32_t w = r[i].work;
    int32_t at = cnt[(size_t)w]++;
    tmp[(size_t)at] = r[i];
  }
  // cnt[w] is now the END of run w; runs are short: insertion sort by seq
  int32_t b = 0;
  for (int64_t w = 0; w < n_sel; ++w) {
    const int32_t e = cnt[(size_t)w];
    for (int32_t i = b + 1; i < e; ++i) {
      const lm_record x = tmp[(size_t)i];
      int32_t j = i - 1;
      while (j >= b && tmp[(size_t)j].seq > x.seq) { tmp[(size_t)j + 1] = tmp[(size_t)j]; --j; }
      tmp[(size_t)j + 1] = x;
    }
    b = e;
  }
  memcpy(r, tmp.data(), sizeof(lm_record) * (size_t)n);
}

extern "C" int lm_fetch_records(lm_detector* d, lm_record* out, int64_t cap, int64_t* n_out) {
  if (!d || !n_out) return fail(LM_E_INVALID, "null argument");
  if (!d->have_run) return fail(LM_E_STATE, "lm_run has not been called");
  CU(cudaSetDevice(d->device));
  const int64_t n = d->h_res->count;
  *n_out = n;
  if (n > cap) return fail(LM_E_CAPACITY, "%lld records, capacity %lld", (long long)n, (long long)cap);
  lm_record* h = reinterpret_cast<lm_record*>(d->h_res + 1);
  if (n > d->h_valid) {  // the rest, beyond the first-fetch window
    CU(cudaMemcpyAsync(h + d->h_valid, reinterpret_cast<lm_record*>(d->d_res + 1) + d->h_valid,
                       sizeof(lm_record) * (size_t)(n - d->h_valid), cudaMemcpyDeviceToHost, d->stream));
    CU(cudaStreamSynchronize(d->stream));
    d->h_valid = n;
  }
  if (n > 0) {
    memcpy(out, h, sizeof(lm_record) * (size_t)n);
    order_records(d, out, n);  // the reference's pre-sort order
  }
  return LM_OK;
}

namespace {
struct HostMatch {  // LL.h:225-258 with class_index standing in for the class_id string
  int x, y;
  float similarity;
  int class_index, template_id;
  // operator< (similarity descending, then template_id ascending) lives in lm_finish's 64-bit sort keys
  bool operator==(const HostMatch& o) const {
    return x == o.x && y == o.y && similarity == o.similarity && class_index == o.class_index;
  }
};
}  // namespace

extern "C" int lm_finish(lm_detector* d, const lm_record* records, int64_t n, lm_match* out, int64_t cap, int64_t* n_out) {
  if (!d || !n_out || (n > 0 && !records)) return fail(LM_E_INVALID, "null argument");
  if ((int)d->class_of.size() != d->G) {
    d->class_of.resize((size_t)d->G);
    for (int c = 0; c < d->n_classes; ++c)
      for (int g = d->class_begin[c]; g < d->class_begin[c + 1]; ++g) d->class_of[(size_t)g] = c;
  }
  const std::vector<int>& class_of = d->class_of;
  // (work, seq) order = class order -> template_id -> coarse cell, the order in which the reference's loops insert
  // the matches (LL.cpp:1797-1939); callers that fetched the records through lm_fetch_records pass them sorted
  const lm_record* rec = records;
  if (!std::is_sorted(records, records + n, record_order)) {
    d->finish_rec.assign(records, records + n);
    order_records(d, d->finish_rec.data(), n);
    rec = d->finish_rec.data();
  }
  // std::sort(matches) with Match::operator< (similarity descending, then template_id ascending; LL.h:233-240,
  // LL.cpp:1772) on 16-byte keys: the comparator induces the same strict weak order on the same input sequence, so
  // libstdc++'s introsort takes the same decisions and leaves the same permutation (ties included) as it would on
  // the Match structs -- with one integer compare per step instead of a float and an int compare.
  struct SortKey {
    uint64_t key;  // ~order(similarity) : 32 | template_id : 32
    uint32_t idx;
    uint32_t pad;
    bool operator<(const SortKey& o) const { return key < o.key; }
  };
  static thread_local std::vector<HostMatch> v;  // scratch, reused between calls
  v.resize((size_t)n);
  std::vector<uint8_t>& keybuf = d->finish_keys;
  keybuf.resize(sizeof(SortKey) * (size_t)std::max<int64_t>(n, 1));
  SortKey* keys = reinterpret_cast<SortKey*>(keybuf.data());
  for (int64_t i = 0; i < n; ++i) {
    const lm_record& r = rec[i];
    if (r.work < 0 || (size_t)r.work >= d->sel.size())
      return fail(LM_E_INVALID, "record %lld: work index %d out of range", (long long)i, r.work);
    const int g = d->sel[r.work];
    const int c = class_of[g];
    const int tid = g - d->class_begin[c];
    v[(size_t)i] = HostMatch{r.x, r.y, r.similarity, c, tid};
    uint32_t b;
    memcpy(&b, &r.similarity, 4);
    if ((b << 1) == 0u) b = 0u;                                       // -0.0f == 0.0f for operator<
    const uint32_t ord = (b & 0x80000000u) ? ~b : (b | 0x80000000u);  // monotone in the float value
    keys[i].key = ((uint64_t)(~ord) << 32) | (uint32_t)tid;           // descending similarity, ascending template_id
    keys[i].idx = (uint32_t)i;
    keys[i].pad = 0;
  }
  std::sort(keys, keys + n);  // LL.cpp:1772
  // std::unique (LL.cpp:1773-1774): drop an element equal (x, y, similarity, class) to the last one KEPT
  int64_t m = 0;
  int64_t last = -1;
  for (int64_t i = 0; i < n; ++i) {
    const HostMatch& h = v[keys[i].idx];
    if (last >= 0 && v[(size_t)last] == h) continue;
    last = keys[i].idx;
    if (m < cap) {
      out[m].x = h.x; out[m].y = h.y; out[m].similarity = h.similarity;
      out[m].class_index = h.class_index; out[m].template_id = h.template_id;
    }
    ++m;
  }
  *n_out = m;
  if (m > cap) return fail(LM_E_CAPACITY, "%lld matches, capacity %lld", (long long)m, (long long)cap);
  return LM_OK;
}

// ---- post-match stage (SURVEY 8f-3) -------------------------------------------------------------
#define LM_POST_MAX 1024

extern "C" int lm_set_boxes(lm_detector* d, const int32_t* wh, int64_t n_templates) {
  if (!d) return fail(LM_E_INVALID, "null detector");
  if (!wh) {
    d->boxes.clear();
  } else {
    if (n_templates != d->G) return fail(LM_E_INVALID, "%lld box sizes for a bank of %d templates", (long long)n_templates, d->G);
    for (int64_t i = 0; i < 2 * n_templates; ++i)
      if (wh[i] < 0 || wh[i] > 32767) return fail(LM_E_INVALID, "box size outside 0..32767");
    d->boxes.assign(wh, wh + 2 * n_templates);
  }
  d->post_dirty = true;
  return LM_OK;
}

static int prepare_post(lm_detector* d) {
  if (!d->d_post_out) {
    CU(cudaMalloc(&d->d_post_out, sizeof(lm_match) * LM_POST_MAX));
    CU(cudaMallocHost(&d->h_post_out, sizeof(lm_match) * LM_POST_MAX));
    CU(cudaMalloc(&d->d_post_counts, sizeof(int32_t) * 4));
    CU(cudaMallocHost(&d->h_post_counts, sizeof(int32_t) * 4));
  }
  if (d->post_live_cap < d->res_cap) {
    cudaFree(d->d_post_live);
    d->d_post_live = nullptr;
    d->post_live_cap = d->res_cap;
    CU(cudaMalloc(&d->d_post_live, (size_t)d->post_live_cap));
  }
  if (!d->post_dirty) return LM_OK;
  if (!d->boxes.empty() && (int64_t)d->boxes.size() != 2 * (int64_t)d->G) {
    d->boxes.clear();  // the bank changed under the caller's boxes
    return fail(LM_E_STATE, "box sizes were set for another bank: call lm_set_boxes again");
  }
  const int64_t n = (int64_t)d->sel.size();
  std::vector<int> class_of(d->G);
  for (int c = 0; c < d->n_classes; ++c)
    for (int g = d->class_begin[c]; g < d->class_begin[c + 1]; ++g) class_of[g] = c;
  std::vector<PostInfo> info((size_t)std::max<int64_t>(n, 1));
  for (int64_t i = 0; i < n; ++i) {
    const int g = d->sel[i];
    PostInfo& q = info[i];
    q.class_index = class_of[g];
    q.template_id = g - d->class_begin[class_of[g]];
    if (d->boxes.empty()) {  // Template::width / height of the first modality at level 0 (LL.h:36-45)
      q.width = d->tmeta[((size_t)g * d->S) * 4 + 0];
      q.height = d->tmeta[((size_t)g * d->S) * 4 + 1];
    } else {
      q.width = d->boxes[2 * (size_t)g];
      q.height = d->boxes[2 * (size_t)g + 1];
    }
  }
  if (d->post_info_n < (int64_t)info.size()) {
    cudaFree(d->d_post_info);
    d->d_post_info = nullptr;
    d->post_info_n = (int64_t)info.size();
    CU(cudaMalloc(&d->d_post_info, sizeof(PostInfo) * info.size()));
  }
  CU(cudaMemcpyAsync(d->d_post_info, info.data(), sizeof(PostInfo) * info.size(), cudaMemcpyHostToDevice, d->stream));
  CU(cudaStreamSynchronize(d->stream));
  d->post_dirty = false;
  return LM_OK;
}

extern "C" int lm_enqueue_post(lm_detector* d, double iou_threshold, int top_k) {
  if (d && d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  if (!d) return fail(LM_E_INVALID, "null detector");
  if (!d->d_res) return fail(LM_E_STATE, "no stages enqueued (call lm_enqueue first)");
  if (top_k > LM_POST_MAX) return fail(LM_E_INVALID, "top_k %d > %d", top_k, LM_POST_MAX);
  if (!(iou_threshold >= 0.0)) return fail(LM_E_INVALID, "IoU threshold must be >= 0");
  CU(cudaSetDevice(d->device));
  int rc = prepare_post(d);
  if (rc) return rc;
  PostParams p;
  p.hdr = d->d_res; p.capacity = (int32_t)d->res_cap;
  p.info = d->d_post_info; p.n_sel = (int32_t)d->sel.size();
  p.iou_threshold = iou_threshold; p.top_k = top_k;
  p.out = d->d_post_out; p.out_capacity = LM_POST_MAX;
  p.out_counts = d->d_post_counts; p.live = d->d_post_live;
  CU(launch_pdl(k_post_nms, dim3(1), dim3(1024), 0, d->stream, p));
  ++d->launches;
  d->post_iou = iou_threshold;
  d->post_top_k = top_k;
  d->post_pending = true;
  return LM_OK;
}

extern "C" int lm_complete_post(lm_detector* d, lm_match* out, int64_t cap, int64_t* n_out, int64_t* n_records) {
  if (d && d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  if (!d || !n_out) return fail(LM_E_INVALID, "null argument");
  if (!d->post_pending) return fail(LM_E_STATE, "lm_enqueue_post has not been called");
  CU(cudaSetDevice(d->device));
  cudaStream_t st = d->stream;
  CU(cudaMemcpyAsync(d->h_post_counts, d->d_post_counts, sizeof(int32_t) * 4, cudaMemcpyDeviceToHost, st));
  // the common top-k is small: fetch a first window with the counts, the rest only if there is more
  const int first = 16;
  CU(cudaMemcpyAsync(d->h_post_out, d->d_post_out, sizeof(lm_match) * first, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(d->h_counters, d->d_counters, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  CU(cudaGetLastError());
  d->post_pending = false;
  if (d->px_rank >= 0 && d->h_counters[2] == 1)
    return fail(LM_E_STATE, "peer exchange: a rank did not publish frame %d within %llu ms", d->px_seq, d->px_timeout_ns / 1000000ull);
  if (d->px_rank >= 0 && d->h_counters[2] == 2) return fail(LM_E_CAPACITY, "peer exchange: a shard kept more than %lld records", (long long)d->px_cap);
  const int64_t n = d->h_post_counts[0];
  if (n_records) *n_records = d->h_post_counts[1];
  if ((int64_t)d->h_post_counts[1] > d->res_cap || (int64_t)d->h_post_counts[3] > d->cand_cap) {
    // the NMS did not see every record: grow the block like lm_complete does, redo the refinement, run the NMS again
    if (d->post_retry || d->res_external || d->px_rank >= 0)
      return fail(LM_E_CAPACITY, "%d records kept, the result block holds %lld: the NMS did not see all of them", d->h_post_counts[1],
                  (long long)d->res_cap);
    CU(cudaMemcpyAsync(d->h_res, d->d_res, sizeof(lm_result_header), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    int rc = grow_and_rerun(d);
    if (rc) return rc;
    rc = lm_enqueue_post(d, d->post_iou, d->post_top_k);
    if (rc) return rc;
    d->post_retry = true;
    rc = lm_complete_post(d, out, cap, n_out, n_records);
    d->post_retry = false;
    return rc;
  }
  *n_out = n;
  if (n > cap) return fail(LM_E_CAPACITY, "%lld survivors, capacity %lld", (long long)n, (long long)cap);
  if (n > first) {
    CU(cudaMemcpyAsync(d->h_post_out + first, d->d_post_out + first, sizeof(lm_match) * (size_t)(n - first), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  if (n > 0 && out) memcpy(out, d->h_post_out, sizeof(lm_match) * (size_t)n);
  return LM_OK;
}

extern "C" int lm_match_top(lm_detector* d, const uint8_t* const* quantized, const int* rows, const int* cols, float threshold,
                            double iou_threshold, int top_k, lm_match* out, int64_t cap, int64_t* n_out, int64_t* n_records) {
  int rc = upload_quantized(d, quantized, rows, cols, false);
  if (rc) return rc;
  rc = lm_enqueue(d, threshold);
  if (rc) return rc;
  rc = lm_enqueue_post(d, iou_threshold, top_k);
  if (rc) return rc;
  return lm_complete_post(d, out, cap, n_out, n_records);
}

extern "C" int lm_match_quantized(lm_detector* d, const uint8_t* const* quantized, const int* rows, const int* cols,
                                  float threshold, lm_match* out, int64_t cap, int64_t* n_out) {
  int rc = upload_quantized(d, quantized, rows, cols, false);  // lm_run synchronises before this call returns
  if (rc) return rc;
  rc = lm_run(d, threshold);
  if (rc) return rc;
  const int64_t n = d->h_res->count;
  std::vector<lm_record> rec((size_t)n);
  int64_t got = 0;
  rc = lm_fetch_records(d, rec.data(), n, &got);
  if (rc) return rc;
  return lm_finish(d, rec.data(), got, out, cap, n_out);
}

extern "C" int lm_match_images(lm_detector* d, const uint8_t* rgb, const uint16_t* depth, int rows, int cols, const uint8_t* mask_color,
                               const uint8_t* mask_depth, float threshold, lm_match* out, int64_t cap, int64_t* n_out) {
  int rc = lm_upload_images(d, rgb, depth, rows, cols, mask_color, mask_depth);
  if (rc) return rc;
  rc = lm_run(d, threshold);
  if (rc) return rc;
  const int64_t n = d->h_res->count;
  std::vector<lm_record> rec((size_t)n);
  int64_t got = 0;
  rc = lm_fetch_records(d, rec.data(), n, &got);
  if (rc) return rc;
  return lm_finish(d, rec.data(), got, out, cap, n_out);
}

extern "C" int lm_debug_quantized(lm_detector* d, int level, int modality, uint8_t* out, int64_t cap) {
  if (!d || !out) return fail(LM_E_INVALID, "null argument");
  if (d->device < 0) return fail(LM_E_STATE, "host-only handle");
  if (!d->have_frame) return fail(LM_E_STATE, "no frame uploaded");
  if (level < 0 || level >= d->L || modality < 0 || modality >= d->M) return fail(LM_E_INVALID, "bad level/modality");
  const LevelHost& lv = d->lv[level];
  const int64_t n = (int64_t)lv.rows * lv.cols;
  if (n > cap) return fail(LM_E_CAPACITY, "need %lld bytes", (long long)n);
  CU(cudaSetDevice(d->device));
  CU(cudaMemcpyAsync(out, lv.q_src[modality], (size_t)n, cudaMemcpyDeviceToHost, d->stream));
  CU(cudaStreamSynchronize(d->stream));
  return LM_OK;
}

extern "C" int lm_debug_linear_memories(lm_detector* d, int level, int modality, uint8_t* out, int64_t cap) {
  if (!d || !out) return fail(LM_E_INVALID, "null argument");
  if (!d->have_run) return fail(LM_E_STATE, "lm_run has not been called");
  if (level < 0 || level >= d->L || modality < 0 || modality >= d->M) return fail(LM_E_INVALID, "bad level/modality");
  const LevelHost& lv = d->lv[level];
  if ((int64_t)lv.mod_stride > cap) return fail(LM_E_CAPACITY, "need %u bytes", lv.mod_stride);
  CU(cudaSetDevice(d->device));
  if (level == d->last_planes_level) {
    // the last run built this level as H-planes only (nothing reads its bytes): build the bytes now, from the frame that
    // is still bound, without touching the bit-planes
    K1Plan k;
    plan_k1(d, -1, false, k);
    const int b0 = level == d->L - 1 ? 0 : k.p.lv[level + 1].block_end;
    int rc = launch_k1(d, k, b0, k.p.lv[level].block_end - b0);
    if (rc) return rc;
    d->last_planes_level = -1;
  }
  CU(cudaMemcpyAsync(out, lv.d_lm + (size_t)modality * lv.mod_stride, lv.mod_stride, cudaMemcpyDeviceToHost, d->stream));
  CU(cudaStreamSynchronize(d->stream));
  return LM_OK;
}

extern "C" int lm_counters(lm_detector* d, int64_t* out8) {
  if (!d || !out8) return fail(LM_E_INVALID, "null argument");
  if (!d->have_run) return fail(LM_E_STATE, "lm_run has not been called");
  out8[0] = d->shard_count;
  out8[1] = d->h_res->coarse_candidates;
  out8[2] = d->alg_scan_bytes;
  out8[3] = (int64_t)(d->h_counters[0] + d->h_counters[4]) * 256;  // the reference's refinement work, whoever disposed of it
  out8[4] = d->h_res->count;
  out8[5] = (int64_t)d->h_counters[1] * 16;
  out8[6] = (int64_t)d->h_counters[4] * 256;  // ... of which: candidates the filter dropped
  out8[7] = (int64_t)d->h_counters[5] * 4;    // bytes of H-planes the filter read
  return LM_OK;
}

extern "C" int lm_set_timing(lm_detector* d, int slots) {
  if (d && d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  if (!d) return fail(LM_E_INVALID, "null detector");
  CU(cudaSetDevice(d->device));
  CU(cudaStreamSynchronize(d->stream));
  for (cudaEvent_t e : d->tev) cudaEventDestroy(e);
  d->tev.clear();
  d->timing_runs = 0;
  d->timing = slots > 0;
  for (int i = 0; i < slots * LM_TEV; ++i) {
    cudaEvent_t e;
    CU(cudaEventCreate(&e));
    d->tev.push_back(e);
  }
  return LM_OK;
}

extern "C" int lm_stage_times(lm_detector* d, float* out8) {
  if (!d || !out8) return fail(LM_E_INVALID, "null argument");
  if (!d->timing || d->timing_runs == 0) return fail(LM_E_STATE, "timing not enabled / no run recorded");
  CU(cudaSetDevice(d->device));
  CU(cudaStreamSynchronize(d->stream));
  const int64_t slots = (int64_t)d->tev.size() / LM_TEV;
  const int64_t n = std::min<int64_t>(slots, d->timing_runs);
  // events: 0 start | 1 linear memories | 2 coarse scan | 3 offsets (+ upper-level linear memories) | 4 candidate list +
  // filter planes | 5 filter | 6 exact refinement (+ collector)
  static const int from[8] = {0, 1, 2, 3, 0, 3, 4, 5}, to[8] = {1, 2, 3, 6, 6, 4, 5, 6};
  double acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  for (int64_t k = 0; k < n; ++k) {
    cudaEvent_t* ev = d->tev.data() + LM_TEV * k;
    for (int i = 0; i < 8; ++i) {
      float ms;
      CU(cudaEventElapsedTime(&ms, ev[from[i]], ev[to[i]]));
      acc[i] += ms * 1000.0;
    }
  }
  for (int i = 0; i < 8; ++i) out8[i] = (float)(acc[i] / (double)n);
  return LM_OK;
}

// ---- template extraction (Detector::addTemplate, LL.cpp:1943-1975), batched over views ---------------------------
namespace {
struct TrainBuffers {  // one chunk of views; freed when the call returns
  std::vector<void*> owned;
  ~TrainBuffers() {
    for (void* p : owned) cudaFree(p);
  }
  template <typename T>
  cudaError_t get(T** p, size_t count) {
    *p = nullptr;
    if (!count) return cudaSuccess;
    cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
    if (e == cudaSuccess) owned.push_back((void*)*p);
    return e;
  }
};
}  // namespace

// cropTemplates (LL.cpp:234-277) on one view's 2L templates: common box over all levels and modalities, origin
// rounded down to even, coordinates shifted per level; tmeta gets {width, height, first, count}.
static void crop_view(int L, const int* first, const int* count, int32_t* feats, int32_t* tmeta) {
  long long min_x = INT32_MAX, min_y = INT32_MAX, max_x = INT32_MIN, max_y = INT32_MIN;
  for (int s = 0; s < 2 * L; ++s)
    for (int i = 0; i < count[s]; ++i) {
      const int32_t* f = feats + (size_t)(first[s] + i) * 3;
      const long long x = (long long)f[0] << (s / 2), y = (long long)f[1] << (s / 2);
      min_x = std::min(min_x, x); max_x = std::max(max_x, x);
      min_y = std::min(min_y, y); max_y = std::max(max_y, y);
    }
  if (min_x % 2 == 1) min_x -= 1;
  if (min_y % 2 == 1) min_y -= 1;
  for (int s = 0; s < 2 * L; ++s) {
    const int l = s / 2;
    tmeta[s * 4 + 0] = (int32_t)((max_x - min_x) >> l);
    tmeta[s * 4 + 1] = (int32_t)((max_y - min_y) >> l);
    tmeta[s * 4 + 2] = first[s];
    tmeta[s * 4 + 3] = count[s];
    for (int i = 0; i < count[s]; ++i) {
      int32_t* f = feats + (size_t)(first[s] + i) * 3;
      f[0] -= (int32_t)(min_x >> l);
      f[1] -= (int32_t)(min_y >> l);
    }
  }
}

#define LM_TRAIN_MAX_CHUNK 512
#define LM_TRAIN_MAX_SIDE 16384

extern "C" int lm_extract_templates(lm_detector* d, int num_features, int n_views, const uint8_t* const* rgb,
                                    const uint16_t* const* depth, const uint8_t* const* masks, int rows, int cols, int32_t* ok,
                                    int32_t* tmeta, int32_t* feats) {
  if (!d || !rgb || !depth || !ok || !tmeta || !feats) return fail(LM_E_INVALID, "null argument");
  if (d->device < 0) return fail(LM_E_STATE, "host-only handle (device -1): GPU stages are unavailable");
  const int L = d->L;
  if (n_views < 0) return fail(LM_E_INVALID, "n_views = %d", n_views);
  if (num_features < 1 || (num_features >> (L - 1)) < 1)
    return fail(LM_E_INVALID, "num_features = %d: every one of the %d pyramid levels needs at least one feature (num_features >> level)",
                num_features, L);
  if (rows < 1 || cols < 1 || rows > LM_TRAIN_MAX_SIDE || cols > LM_TRAIN_MAX_SIDE)
    return fail(LM_E_INVALID, "image size %d x %d outside 1..%d", cols, rows, LM_TRAIN_MAX_SIDE);
  if (rows % (1 << (L - 1)) || cols % (1 << (L - 1)))
    return fail(LM_E_INVALID, "rows and cols must be multiples of 2^(pyramid_levels - 1) = %d for extraction on the GPU (got %d x %d)",
                1 << (L - 1), cols, rows);
  for (int v = 0; v < n_views; ++v)
    if (!rgb[v] || !depth[v]) return fail(LM_E_INVALID, "null image of view %d", v);
  if (n_views == 0) return LM_OK;
  CU(cudaSetDevice(d->device));
  cudaStream_t st = d->stream;
  if (d->upper_pending) CU(cudaStreamWaitEvent(st, d->ev_upper, 0));
  if (!d->fe_lut) {
    uint8_t lut[400];  // as in lm_upload_images
    for (int vy = 0; vy < 20; ++vy)
      for (int vx = 0; vx < 20; ++vx) {
        double a = atan2((double)(vy - 10), (double)(vx - 10)) * 180.0 / 3.14159265358979323846;
        a = fmod(a + 360.0, 360.0);
        lut[vy * 20 + vx] = (uint8_t)(1u << (((int)(fmod(a + 22.5, 360.0) / 45.0)) % 8));
      }
    CU(cudaMemcpyToSymbolAsync(c_normal_lut, lut, sizeof(lut), 0, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    d->fe_lut = true;
  }

  // layout of one view: levels l = 0..L-1 of size (rows >> l) x (cols >> l); candidate segments (level, modality)
  // with room for every pixel of their level; features in slot order with nf >> l per slot
  TrainSelect ts = {};
  ts.L = L;
  ts.nf0 = num_features;
  int64_t key_stride = 0;
  int key_off[LM_MAX_LEVELS];
  int F = 0;
  for (int l = 0; l < L; ++l) {
    ts.cols[l] = cols >> l;
    ts.npix[l] = (rows >> l) * (cols >> l);
    key_off[l] = (int)key_stride;
    key_stride += 2 * (int64_t)ts.npix[l];
    for (int m = 0; m < 2; ++m) {
      ts.first[l * 2 + m] = F;
      F += num_features >> l;
    }
  }
  ts.F = F;
  const int S = 2 * L;
  const size_t n0 = (size_t)rows * cols, n1 = L > 1 ? n0 / 4 : 0;
  const int smem = 2 * num_features * (int)sizeof(int);
  if (smem > 200 * 1024) return fail(LM_E_INVALID, "num_features = %d above the %d the selection kernel holds", num_features, 200 * 1024 / 8);
  if (smem > 48 * 1024) CU(cudaFuncSetAttribute(k_tr_select, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));

  // chunk of views resident at once: set by free device memory (half of it at most)
  const size_t per_view = n0 * (3 + 2 + 1 + 1 + 1 + 4 + 1 + 4) + n1 * (3 + 1 + 1) + (size_t)key_stride * 16 + (size_t)F * 12 + 64 + S * 16;
  size_t free_b = 0, total_b = 0;
  CU(cudaMemGetInfo(&free_b, &total_b));
  int64_t chunk = (int64_t)(free_b / 2 / per_view);
  chunk = std::min<int64_t>(std::min<int64_t>(chunk, LM_TRAIN_MAX_CHUNK), n_views);
  chunk = std::min<int64_t>(chunk, (int64_t)(INT32_MAX / key_stride));
  if (chunk < 1) return fail(LM_E_CUDA, "not enough free device memory for one view (%zu bytes)", per_view);
  const int B = (int)chunk;

  TrainBuffers tb;
  uint8_t *rgbA, *rgbB, *maskA, *maskB, *normA, *normB, *angle, *nfg, *qun, *strong, *nraw, *nq, *has_mask, *seg_fail;
  uint16_t* dep;
  int32_t *mag, *g, *d_feats, *seg_begin, *seg_end, *lcount, *area;
  unsigned long long *keys, *keys_sorted;
  CU(tb.get(&rgbA, B * n0 * 3)); CU(tb.get(&rgbB, B * n1 * 3)); CU(tb.get(&dep, B * n0));
  CU(tb.get(&maskA, B * n0)); CU(tb.get(&maskB, B * n1)); CU(tb.get(&normA, B * n0)); CU(tb.get(&normB, B * n1));
  CU(tb.get(&angle, B * n0)); CU(tb.get(&mag, B * n0)); CU(tb.get(&nfg, B * n0)); CU(tb.get(&g, B * n0));
  CU(tb.get(&qun, n0)); CU(tb.get(&strong, n0)); CU(tb.get(&nraw, n0)); CU(tb.get(&nq, n0));
  CU(tb.get(&has_mask, (size_t)B)); CU(tb.get(&seg_fail, (size_t)B * S));
  CU(tb.get(&seg_begin, (size_t)B * S)); CU(tb.get(&seg_end, (size_t)B * S));
  CU(tb.get(&lcount, (size_t)B * L * 8)); CU(tb.get(&area, (size_t)B * L));
  CU(tb.get(&keys, (size_t)B * key_stride)); CU(tb.get(&keys_sorted, (size_t)B * key_stride));
  CU(tb.get(&d_feats, (size_t)B * F * 3));
  std::vector<int32_t> h_begin((size_t)B * S);
  for (int v = 0; v < B; ++v)
    for (int l = 0; l < L; ++l)
      for (int m = 0; m < 2; ++m) h_begin[(size_t)v * S + l * 2 + m] = (int32_t)(v * key_stride + key_off[l] + m * (int64_t)ts.npix[l]);
  CU(cudaMemcpyAsync(seg_begin, h_begin.data(), h_begin.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  size_t sort_bytes = 0;
  CU(cub::DeviceSegmentedSort::SortKeys(nullptr, sort_bytes, keys, keys_sorted, (int)(B * key_stride), B * S, seg_begin, seg_end, st));
  void* sort_tmp = nullptr;
  CU(tb.get((uint8_t**)&sort_tmp, sort_bytes));
  std::vector<uint8_t> h_has(B), h_fail((size_t)B * S);

  auto grid2 = [](int w, int h, int z) { return dim3((unsigned)((w + 31) / 32), (unsigned)((h + 7) / 8), (unsigned)z); };
  for (int v0 = 0; v0 < n_views; v0 += B) {
    const int nb = std::min(B, n_views - v0);
    for (int v = 0; v < nb; ++v) {
      const uint8_t* mk = masks ? masks[v0 + v] : nullptr;
      h_has[v] = mk != nullptr;
      CU(cudaMemcpyAsync(rgbA + v * n0 * 3, rgb[v0 + v], n0 * 3, cudaMemcpyHostToDevice, st));
      CU(cudaMemcpyAsync(dep + v * n0, depth[v0 + v], n0 * 2, cudaMemcpyHostToDevice, st));
      if (mk) CU(cudaMemcpyAsync(maskA + v * n0, mk, n0, cudaMemcpyHostToDevice, st));
    }
    CU(cudaMemcpyAsync(has_mask, h_has.data(), nb, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(seg_end, seg_begin, (size_t)nb * S * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    CU(cudaMemsetAsync(lcount, 0, (size_t)nb * L * 8 * sizeof(int32_t), st));
    CU(cudaMemsetAsync(area, 0, (size_t)nb * L * sizeof(int32_t), st));
    for (int l = 0; l < L; ++l) {
      const int H = rows >> l, W = cols >> l;
      // level l lives in the A buffers for even l and in the B buffers for odd l (per-view strides n0 / n1)
      uint8_t* rgb_l = (l & 1) ? rgbB : rgbA;
      uint8_t* norm_l = (l & 1) ? normB : normA;
      uint8_t* mask_l = (l & 1) ? maskB : maskA;
      const size_t s_l = (l & 1) ? n1 : n0;
      const size_t s_u = (l & 1) ? n0 : n1;  // stride of level l - 1
      for (int v = 0; v < nb; ++v) {
        if (l > 0) {  // ColorGradientPyramid::pyrDown / DepthNormalPyramid::pyrDown (LL.cpp:557-567, 861-879)
          const uint8_t* rgb_u = ((l & 1) ? rgbA : rgbB) + v * s_u * 3;
          const uint8_t* norm_u = ((l & 1) ? normA : normB) + v * s_u;
          CU(launch_pdl(k_fe_pyrdown, grid2(W, H, 1), dim3(256), 0, st, rgb_u, H * 2, W * 2, rgb_l + v * s_l * 3, H, W));
          CU(launch_pdl(k_fe_decimate, grid2(W, H, 1), dim3(256), 0, st, norm_u, W * 2, norm_l + v * s_l, H, W, (const uint8_t*)nullptr,
                        (uint8_t*)nullptr));
          d->launches += 2;
          if (h_has[v]) {
            const uint8_t* mask_u = ((l & 1) ? maskA : maskB) + v * s_u;
            CU(launch_pdl(k_fe_decimate, grid2(W, H, 1), dim3(256), 0, st, mask_u, W * 2, mask_l + v * s_l, H, W, (const uint8_t*)nullptr,
                          (uint8_t*)nullptr));
            ++d->launches;
          }
        }
        // colour labels WITHOUT the mask (pyr.angle) and the squared magnitude
        CU(launch_pdl(k_fe_gradient, grid2(W, H, 1), dim3(FE_TW, FE_TH), 0, st, (const uint8_t*)(rgb_l + v * s_l * 3), H, W, 100, qun, strong,
                      mag + v * n0));
        CU(launch_pdl(k_fe_hysteresis, grid2(W, H, 1), dim3(256), 0, st, (const uint8_t*)qun, (const uint8_t*)strong, (const uint8_t*)nullptr,
                      H, W, angle + v * n0));
        d->launches += 2;
        if (l == 0) {
          CU(launch_pdl(k_fe_normals, grid2(W, H, 1), dim3(256), 0, st, (const uint16_t*)(dep + v * n0), H, W, 2000, 50, nraw));
          CU(launch_pdl(k_fe_median, grid2(W, H, 1), dim3(256), 0, st, (const uint8_t*)nraw, (const uint8_t*)nullptr, H, W, norm_l + v * n0, nq));
          d->launches += 2;
        }
      }
      CU(launch_pdl(k_tr_prep, grid2(W, H, nb), dim3(256), 0, st, H, W, l, L, (const uint8_t*)angle, (const int32_t*)mag, n0,
                    (const uint8_t*)norm_l, (const uint8_t*)mask_l, s_l, (const uint8_t*)has_mask, keys, seg_end, nfg, area));
      CU(launch_pdl(k_tr_coldist, dim3((unsigned)((W + 127) / 128), 1, (unsigned)nb), dim3(128), 0, st, H, W, (const uint8_t*)nfg, n0, g));
      CU(launch_pdl(k_tr_normcand, grid2(W, H, nb), dim3(256), 0, st, H, W, l, L, 2 >> l, (const uint8_t*)nfg, (const int*)g, n0, keys,
                    seg_end, lcount));
      d->launches += 3;
    }
    CU(launch_pdl(k_tr_normscore, dim3(16, (unsigned)(nb * L)), dim3(256), 0, st, keys, (const int*)seg_begin, (const int*)seg_end,
                  (const int*)lcount));
    ++d->launches;
    CU(cub::DeviceSegmentedSort::SortKeys(sort_tmp, sort_bytes, keys, keys_sorted, (int)(nb * key_stride), nb * S, seg_begin, seg_end, st));
    CU(launch_pdl(k_tr_select, dim3((unsigned)(nb * S)), dim3(32), (size_t)smem, st, ts, (const unsigned long long*)keys_sorted,
                  (const int*)seg_begin, (const int*)seg_end, (const uint8_t*)has_mask, (const int*)area, d_feats, seg_fail));
    ++d->launches;
    CU(cudaMemcpyAsync(feats + (size_t)v0 * F * 3, d_feats, (size_t)nb * F * 3 * sizeof(int32_t), cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h_fail.data(), seg_fail, (size_t)nb * S, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    int count[2 * LM_MAX_LEVELS];
    for (int s = 0; s < S; ++s) count[s] = num_features >> (s / 2);
    for (int v = 0; v < nb; ++v) {
      bool good = true;
      for (int s = 0; s < S; ++s) good = good && !h_fail[(size_t)v * S + s];
      ok[v0 + v] = good ? 1 : 0;
      int32_t* tm = tmeta + (size_t)(v0 + v) * S * 4;
      int32_t* fv = feats + (size_t)(v0 + v) * F * 3;
      if (good) crop_view(L, ts.first, count, fv, tm);
      else {
        memset(tm, 0, (size_t)S * 4 * sizeof(int32_t));
        memset(fv, 0, (size_t)F * 3 * sizeof(int32_t));
      }
    }
  }
  return LM_OK;
}
