"""ctypes binding of the C-ABI shared library (include/linemod_b200.h).

Fails loudly when the library is missing or cannot be loaded: there is no CPU / PyTorch fallback
for the hot path.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# LINEMOD_B200_LIB: another build of the same library (A/B runs of compile-time variants); never a different backend
LIB_PATH = os.environ.get("LINEMOD_B200_LIB") or os.path.join(_HERE, "csrc", "liblinemod_b200.so")

LM_OK, LM_E_INVALID, LM_E_CUDA, LM_E_STATE, LM_E_CAPACITY = 0, -1, -2, -3, -4
SHARD_CONTIGUOUS, SHARD_INTERLEAVED = 0, 1

MATCH_DTYPE = np.dtype([("x", "<i4"), ("y", "<i4"), ("similarity", "<f4"), ("class_index", "<i4"), ("template_id", "<i4")])
RECORD_DTYPE = np.dtype([("x", "<i2"), ("y", "<i2"), ("similarity", "<f4"), ("work", "<i4"), ("seq", "<i4")])
HEADER_DTYPE = np.dtype([("count", "<i4"), ("coarse_candidates", "<i4"), ("capacity", "<i4"), ("shard", "<i4")])

# every symbol include/linemod_b200.h declares (tests check the .so exports all of them)
PEER_HANDLE_BYTES = 64

SYMBOLS = [
    "lm_last_error", "lm_create", "lm_destroy", "lm_load_bank", "lm_select", "lm_select_layout", "lm_shard_range", "lm_prepare",
    "lm_upload_quantized", "lm_upload_images", "lm_match_images", "lm_debug_quantized", "lm_bind_quantized_device", "lm_run", "lm_enqueue", "lm_complete", "lm_set_result_buffer", "lm_device_result", "lm_fetch_records",
    "lm_finish", "lm_match_quantized", "lm_debug_linear_memories", "lm_counters", "lm_set_timing",
    "lm_stage_times", "lm_stream", "lm_launch_count",
    "lm_set_boxes", "lm_enqueue_post", "lm_complete_post", "lm_match_top",
    "lm_peer_export", "lm_peer_base", "lm_peer_connect", "lm_peer_connect_local", "lm_peer_disconnect",
    "lm_extract_templates",
    "lm_icp_create", "lm_icp_destroy", "lm_icp_process", "lm_icp_process_batch", "lm_icp_last_stats", "lm_icp_launch_count", "lm_icp_set_use_scene_cloud",
]

_lib = None


class LinemodLibraryError(RuntimeError):
    pass


def load():
    """Load liblinemod_b200.so (built in-tree by `make -C 6dpose_b200/csrc` / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LinemodLibraryError(
            "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a).  There is no CPU fallback for the LINEMOD hot path." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    c_int, c_i64, c_f, vp = ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p
    i32p = ctypes.POINTER(ctypes.c_int32)
    u8pp = ctypes.POINTER(ctypes.POINTER(ctypes.c_uint8))
    L.lm_last_error.restype = ctypes.c_char_p
    L.lm_create.argtypes = [c_int, c_int, ctypes.POINTER(c_int), ctypes.POINTER(vp)]
    L.lm_destroy.argtypes = [vp]
    L.lm_destroy.restype = None
    L.lm_load_bank.argtypes = [vp, c_int, i32p, c_int, i32p, i32p, c_i64]
    L.lm_select.argtypes = [vp, i32p, c_int, c_int, c_int]
    L.lm_select_layout.argtypes = [vp, i32p, c_int, c_int, c_int, c_int]
    L.lm_prepare.argtypes = [vp]
    L.lm_shard_range.argtypes = [vp, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]
    L.lm_upload_quantized.argtypes = [vp, u8pp, ctypes.POINTER(c_int), ctypes.POINTER(c_int)]
    u8p_ = ctypes.POINTER(ctypes.c_uint8)
    L.lm_upload_images.argtypes = [vp, u8p_, ctypes.POINTER(ctypes.c_uint16), c_int, c_int, u8p_, u8p_]
    L.lm_match_images.argtypes = [vp, u8p_, ctypes.POINTER(ctypes.c_uint16), c_int, c_int, u8p_, u8p_, c_f, vp, c_i64,
                                  ctypes.POINTER(c_i64)]
    L.lm_debug_quantized.argtypes = [vp, c_int, c_int, u8p_, c_i64]
    L.lm_bind_quantized_device.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(c_int), ctypes.POINTER(c_int)]
    L.lm_run.argtypes = [vp, c_f]
    L.lm_enqueue.argtypes = [vp, c_f]
    L.lm_complete.argtypes = [vp]
    L.lm_set_result_buffer.argtypes = [vp, vp, c_i64]
    L.lm_set_boxes.argtypes = [vp, i32p, c_i64]
    L.lm_enqueue_post.argtypes = [vp, ctypes.c_double, c_int]
    L.lm_complete_post.argtypes = [vp, vp, c_i64, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]
    L.lm_match_top.argtypes = [vp, u8pp, ctypes.POINTER(c_int), ctypes.POINTER(c_int), c_f, ctypes.c_double, c_int, vp, c_i64,
                               ctypes.POINTER(c_i64), ctypes.POINTER(c_i64)]
    L.lm_peer_export.argtypes = [vp, c_int, c_i64, u8p_]
    L.lm_peer_base.argtypes = [vp, ctypes.POINTER(vp)]
    L.lm_peer_connect.argtypes = [vp, c_int, c_int, u8p_]
    L.lm_peer_connect_local.argtypes = [vp, c_int, c_int, ctypes.POINTER(vp)]
    L.lm_peer_disconnect.argtypes = [vp]
    L.lm_device_result.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(c_i64)]
    L.lm_fetch_records.argtypes = [vp, vp, c_i64, ctypes.POINTER(c_i64)]
    L.lm_finish.argtypes = [vp, vp, c_i64, vp, c_i64, ctypes.POINTER(c_i64)]
    L.lm_match_quantized.argtypes = [vp, u8pp, ctypes.POINTER(c_int), ctypes.POINTER(c_int), c_f, vp, c_i64,
                                     ctypes.POINTER(c_i64)]
    L.lm_debug_linear_memories.argtypes = [vp, c_int, c_int, ctypes.POINTER(ctypes.c_uint8), c_i64]
    L.lm_counters.argtypes = [vp, ctypes.POINTER(c_i64)]
    L.lm_set_timing.argtypes = [vp, c_int]
    L.lm_stage_times.argtypes = [vp, ctypes.POINTER(c_f)]
    L.lm_stream.argtypes = [vp]
    L.lm_stream.restype = vp
    L.lm_launch_count.argtypes = [vp]
    L.lm_launch_count.restype = c_i64
    f32p, f64p = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_double)
    u16p = ctypes.POINTER(ctypes.c_uint16)
    L.lm_extract_templates.argtypes = [vp, c_int, c_int, u8pp, ctypes.POINTER(u16p), u8pp, c_int, c_int, i32p, i32p, i32p]
    L.lm_icp_create.argtypes = [c_int, ctypes.POINTER(vp)]
    L.lm_icp_destroy.argtypes = [vp]
    L.lm_icp_destroy.restype = None
    L.lm_icp_process.argtypes = [vp, u16p, c_int, c_int, u16p, c_int, c_int, f32p, f32p, f32p, f32p, c_int, c_int, c_int,
                                 f64p, f64p, f32p]
    L.lm_icp_process_batch.argtypes = [vp, c_int, u16p, c_int, c_int, ctypes.POINTER(u16p), c_int, c_int, f32p, f32p, f32p, f32p,
                                       i32p, c_int, f64p, f64p, f32p]
    L.lm_icp_last_stats.argtypes = [vp, f64p]
    L.lm_icp_set_use_scene_cloud.argtypes = [vp, c_int]
    L.lm_icp_launch_count.argtypes = [vp]
    L.lm_icp_launch_count.restype = c_i64
    for name in SYMBOLS:
        getattr(L, name)  # AttributeError if the library does not export a declared symbol
    _lib = L
    return L


def check(rc):
    if rc == LM_OK:
        return
    msg = load().lm_last_error().decode("utf-8", "replace")
    if rc == LM_E_INVALID:
        raise RuntimeError(msg)  # the reference raises cv::Exception -> RuntimeError through pybind11
    raise LinemodLibraryError("linemod_b200 error %d: %s" % (rc, msg))


class NativeDetector:
    """Thin RAII wrapper over the lm_detector handle."""

    def __init__(self, T, device=0):
        L = load()
        self._L = L
        self.T = [int(t) for t in T]
        self.levels = len(self.T)
        arr = (ctypes.c_int * self.levels)(*self.T)
        h = ctypes.c_void_p()
        check(L.lm_create(int(device), self.levels, arr, ctypes.byref(h)))
        self._h = h
        self._keep = None

    def close(self):
        if getattr(self, "_h", None):
            self._L.lm_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @staticmethod
    def _i32(a):
        return a.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))

    def load_bank(self, packed, slots):
        cb = np.ascontiguousarray(packed["class_begin"], np.int32)
        tm = np.ascontiguousarray(packed["tmeta"], np.int32)
        ft = np.ascontiguousarray(packed["feats"], np.int32)
        check(self._L.lm_load_bank(self._h, len(cb) - 1, self._i32(cb), int(slots), self._i32(tm), self._i32(ft),
                                   int(ft.shape[0])))

    def select(self, class_indices=None, shard_index=0, shard_count=1, layout=SHARD_CONTIGUOUS):
        """layout: SHARD_CONTIGUOUS (blocks of the sequence) or SHARD_INTERLEAVED (rank r takes r, r+N, ...)."""
        if class_indices is None:
            check(self._L.lm_select_layout(self._h, None, -1, int(shard_index), int(shard_count), int(layout)))
        else:
            a = np.ascontiguousarray(class_indices, np.int32)
            check(self._L.lm_select_layout(self._h, self._i32(a), int(a.shape[0]), int(shard_index), int(shard_count), int(layout)))

    def prepare(self):
        check(self._L.lm_prepare(self._h))

    def shard_range(self):
        b, c = ctypes.c_int64(), ctypes.c_int64()
        check(self._L.lm_shard_range(self._h, ctypes.byref(b), ctypes.byref(c)))
        return b.value, c.value

    def _frame_args(self, quantized):
        qs = []
        rows, cols = [], []
        for lvl in quantized:
            if len(lvl) != 2:
                raise RuntimeError("sources.size() == modalities.size()")
            rows.append(lvl[0].shape[0])
            cols.append(lvl[0].shape[1])
            for q in lvl:
                if q.dtype != np.uint8 or q.ndim != 2 or q.shape != lvl[0].shape:
                    raise TypeError("quantized images must be uint8 HxW, same size per level")
                qs.append(np.ascontiguousarray(q))
        if len(quantized) != self.levels:
            raise RuntimeError("expected %d pyramid levels, got %d" % (self.levels, len(quantized)))
        ptrs = (ctypes.POINTER(ctypes.c_uint8) * len(qs))(*[q.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)) for q in qs])
        r = (ctypes.c_int * len(rows))(*rows)
        c = (ctypes.c_int * len(cols))(*cols)
        return qs, ptrs, r, c

    def upload_quantized(self, quantized):
        qs, ptrs, r, c = self._frame_args(quantized)
        check(self._L.lm_upload_quantized(self._h, ptrs, r, c))

    @staticmethod
    def _image_args(rgb, depth, masks):
        rgb = np.ascontiguousarray(rgb)
        depth = np.ascontiguousarray(depth)
        if rgb.dtype != np.uint8 or rgb.ndim != 3 or rgb.shape[2] != 3:
            raise TypeError("sources[0] must be a uint8 HxWx3 colour image")
        if depth.dtype != np.uint16 or depth.shape != rgb.shape[:2]:
            raise TypeError("sources[1] must be a uint16 HxW depth image of the same size")
        mk = [None, None]
        if masks:
            if len(masks) != 2:
                raise RuntimeError("masks.size() == modalities.size()")
            for i, m in enumerate(masks):
                if m is not None and np.asarray(m).size:
                    m = np.ascontiguousarray(m)
                    if m.dtype != np.uint8 or m.shape != rgb.shape[:2]:
                        raise RuntimeError("mask.size() == source.size()")
                    mk[i] = m
        u8p = ctypes.POINTER(ctypes.c_uint8)
        ptr = lambda a: a.ctypes.data_as(u8p) if a is not None else None
        return rgb, depth, mk, (ptr(rgb), depth.ctypes.data_as(ctypes.POINTER(ctypes.c_uint16)), rgb.shape[0], rgb.shape[1],
                               ptr(mk[0]), ptr(mk[1]))

    def upload_images(self, rgb, depth, masks=None):
        keep = self._image_args(rgb, depth, masks)
        check(self._L.lm_upload_images(self._h, *keep[3]))

    def match_images(self, rgb, depth, masks, threshold):
        keep = self._image_args(rgb, depth, masks)
        cap = 1 << 12
        while True:
            out = np.empty(cap, MATCH_DTYPE)
            n = ctypes.c_int64()
            rc = self._L.lm_match_images(self._h, *keep[3], ctypes.c_float(threshold), out.ctypes.data_as(ctypes.c_void_p), cap,
                                         ctypes.byref(n))
            if rc == LM_E_CAPACITY:
                cap = int(n.value)
                continue
            check(rc)
            return out[:n.value].copy()

    def quantized(self, level, modality, shape):
        out = np.zeros(shape, np.uint8)
        check(self._L.lm_debug_quantized(self._h, level, modality, out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)), out.size))
        return out

    def bind_quantized_device(self, ptrs, rows, cols):
        """ptrs: device addresses (ints) index level*2+modality; rows/cols per level."""
        p = (ctypes.c_void_p * len(ptrs))(*[int(x) for x in ptrs])
        r = (ctypes.c_int * len(rows))(*[int(x) for x in rows])
        c = (ctypes.c_int * len(cols))(*[int(x) for x in cols])
        check(self._L.lm_bind_quantized_device(self._h, p, r, c))

    @staticmethod
    def bind_args(ptrs, rows, cols):
        """The ctypes arrays of bind_quantized_device, built once for a frame that is bound many times."""
        return ((ctypes.c_void_p * len(ptrs))(*[int(x) for x in ptrs]), (ctypes.c_int * len(rows))(*[int(x) for x in rows]),
                (ctypes.c_int * len(cols))(*[int(x) for x in cols]))

    def bind_quantized_device_args(self, args):
        check(self._L.lm_bind_quantized_device(self._h, args[0], args[1], args[2]))

    def run(self, threshold):
        check(self._L.lm_run(self._h, ctypes.c_float(threshold)))

    def enqueue(self, threshold):
        check(self._L.lm_enqueue(self._h, ctypes.c_float(threshold)))

    def complete(self):
        check(self._L.lm_complete(self._h))

    def fetch_records(self):
        cap = 1 << 12
        while True:
            out = np.empty(cap, RECORD_DTYPE)
            n = ctypes.c_int64()
            rc = self._L.lm_fetch_records(self._h, out.ctypes.data_as(ctypes.c_void_p), cap, ctypes.byref(n))
            if rc == LM_E_CAPACITY:
                cap = int(n.value)
                continue
            check(rc)
            return out[:n.value].copy()

    def set_result_buffer(self, device_ptr, capacity_records):
        check(self._L.lm_set_result_buffer(self._h, ctypes.c_void_p(device_ptr) if device_ptr else None, int(capacity_records)))

    # ---- multi-GPU exchange fused into the refinement kernel (include/linemod_b200.h, lm_peer_*) ----
    def peer_export(self, world, capacity_records=8192):
        """Allocate this rank's exchange buffer; returns its CUDA IPC handle (bytes)."""
        h = (ctypes.c_uint8 * PEER_HANDLE_BYTES)()
        check(self._L.lm_peer_export(self._h, int(world), int(capacity_records), h))
        return bytes(h)

    def peer_base(self):
        b = ctypes.c_void_p()
        check(self._L.lm_peer_base(self._h, ctypes.byref(b)))
        return b.value

    def peer_connect(self, rank, world, handles):
        """handles: list of `world` IPC handles (bytes), index = rank (own entry ignored)."""
        blob = b"".join(bytes(h) for h in handles)
        if len(blob) != world * PEER_HANDLE_BYTES:
            raise ValueError("need %d handles of %d bytes" % (world, PEER_HANDLE_BYTES))
        buf = (ctypes.c_uint8 * len(blob)).from_buffer_copy(blob)
        check(self._L.lm_peer_connect(self._h, int(rank), int(world), buf))

    def peer_connect_local(self, rank, world, bases):
        arr = (ctypes.c_void_p * world)(*[int(b) for b in bases])
        check(self._L.lm_peer_connect_local(self._h, int(rank), int(world), arr))

    def peer_disconnect(self):
        check(self._L.lm_peer_disconnect(self._h))

    def device_result(self):
        p, cap = ctypes.c_void_p(), ctypes.c_int64()
        check(self._L.lm_device_result(self._h, ctypes.byref(p), ctypes.byref(cap)))
        return p.value, cap.value

    def finish(self, records):
        records = np.ascontiguousarray(records, RECORD_DTYPE)
        cap = max(int(records.shape[0]), 1)
        out = np.zeros(cap, MATCH_DTYPE)
        n = ctypes.c_int64()
        check(self._L.lm_finish(self._h, records.ctypes.data_as(ctypes.c_void_p), int(records.shape[0]),
                                out.ctypes.data_as(ctypes.c_void_p), cap, ctypes.byref(n)))
        return out[:n.value].copy()

    def match_quantized(self, quantized, threshold):
        qs, ptrs, r, c = self._frame_args(quantized)
        cap = 1 << 12
        while True:
            out = np.empty(cap, MATCH_DTYPE)
            n = ctypes.c_int64()
            rc = self._L.lm_match_quantized(self._h, ptrs, r, c, ctypes.c_float(threshold),
                                            out.ctypes.data_as(ctypes.c_void_p), cap, ctypes.byref(n))
            if rc == LM_E_CAPACITY:
                cap = int(n.value)
                continue
            check(rc)
            return out[:n.value].copy()

    # ---- post-match stage on the device: greedy NMS + top-k (include/linemod_b200.h, lm_*_post) ----
    def set_boxes(self, wh):
        if wh is None:
            check(self._L.lm_set_boxes(self._h, None, 0))
            return
        wh = np.ascontiguousarray(wh, np.int32).reshape(-1, 2)
        check(self._L.lm_set_boxes(self._h, self._i32(wh), wh.shape[0]))

    def enqueue_post(self, iou_threshold=0.5, top_k=3):
        check(self._L.lm_enqueue_post(self._h, float(iou_threshold), int(top_k)))

    def complete_post(self):
        out = np.empty(1024, MATCH_DTYPE)
        n, nrec = ctypes.c_int64(), ctypes.c_int64()
        check(self._L.lm_complete_post(self._h, out.ctypes.data_as(ctypes.c_void_p), out.shape[0], ctypes.byref(n),
                                       ctypes.byref(nrec)))
        return out[:n.value].copy(), int(nrec.value)

    def match_top(self, quantized, threshold, iou_threshold=0.5, top_k=3):
        qs, ptrs, r, c = self._frame_args(quantized)
        out = np.empty(1024, MATCH_DTYPE)
        n, nrec = ctypes.c_int64(), ctypes.c_int64()
        check(self._L.lm_match_top(self._h, ptrs, r, c, ctypes.c_float(threshold), float(iou_threshold), int(top_k),
                                   out.ctypes.data_as(ctypes.c_void_p), out.shape[0], ctypes.byref(n), ctypes.byref(nrec)))
        return out[:n.value].copy(), int(nrec.value)

    def linear_memories(self, level, modality, shape):
        out = np.zeros(shape, np.uint8)
        check(self._L.lm_debug_linear_memories(self._h, level, modality, out.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8)),
                                               out.size))
        return out

    def counters(self):
        a = (ctypes.c_int64 * 8)()
        check(self._L.lm_counters(self._h, a))
        keys = ["templates", "coarse_candidates", "scan_bytes", "refine_bytes", "kept", "refine_bytes_read",
                "filter_dropped_bytes", "filter_bytes_read"]
        return dict(zip(keys, [int(v) for v in a]))

    def set_timing(self, slots):
        check(self._L.lm_set_timing(self._h, int(slots)))

    def stage_times_us(self):
        a = (ctypes.c_float * 8)()
        check(self._L.lm_stage_times(self._h, a))
        keys = ["linear_memories", "coarse_scan", "offsets", "refine", "total", "refine_prep", "refine_filter", "refine_exact"]
        return dict(zip(keys, [float(v) for v in a]))

    # ---- template extraction on the device (include/linemod_b200.h, lm_extract_templates) ----
    def extract_templates(self, num_features, rgbs, depths, masks):
        """Detector::addTemplate's extraction for n views of one size (uint8 HxWx3, uint16 HxW, uint8 HxW or None;
        the caller checks dtypes and shapes).  Returns (ok bool [n], tmeta int32 [n, 2L, 4] = width, height, first,
        count after cropTemplates, feats int32 [n, F, 3] = x, y, label with F = sum_l 2 * (num_features >> l))."""
        n = len(rgbs)
        rows, cols = (rgbs[0].shape[:2] if n else (0, 0))
        F = sum(2 * (int(num_features) >> l) for l in range(self.levels))
        ok = np.zeros(n, np.int32)
        tmeta = np.zeros((n, 2 * self.levels, 4), np.int32)
        feats = np.zeros((n, F, 3), np.int32)
        u8p, u16p = ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(ctypes.c_uint16)
        rp = (u8p * max(n, 1))(*[a.ctypes.data_as(u8p) for a in rgbs])
        dp = (u16p * max(n, 1))(*[a.ctypes.data_as(u16p) for a in depths])
        mp = None
        if any(m is not None for m in masks):
            mp = (u8p * max(n, 1))(*[m.ctypes.data_as(u8p) if m is not None else None for m in masks])
        check(self._L.lm_extract_templates(self._h, int(num_features), n, rp, dp, mp, int(rows), int(cols), self._i32(ok),
                                           self._i32(tmeta), self._i32(feats)))
        return ok.astype(bool), tmeta, feats

    def stream(self):
        return self._L.lm_stream(self._h)

    def launch_count(self):
        return int(self._L.lm_launch_count(self._h))


class NativeIcp:
    """RAII wrapper over the lm_icp handle (poseRefine compute)."""

    def __init__(self, device=0):
        L = load()
        self._L = L
        h = ctypes.c_void_p()
        check(L.lm_icp_create(int(device), ctypes.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self._L.lm_icp_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def process_batch(self, scene_depth, model_depths, sceneK, modelKs, Rs, ts, detect_xy, max_iterations=30):
        """scene u16 HxW; model_depths list of u16 HxW (same size); modelKs/Rs [n,3,3] f32; ts [n,3] f32;
        detect_xy [n,2] int.  Returns (R [n,3,3] f64, t [n,3] f64 mm, residual [n] f32)."""
        n = len(model_depths)
        scene = np.ascontiguousarray(scene_depth, np.uint16)
        models = [np.ascontiguousarray(m, np.uint16) for m in model_depths]
        for m in models:
            if m.shape != models[0].shape:
                raise TypeError("model depth images must share one size")
        u16p = ctypes.POINTER(ctypes.c_uint16)
        f32p, f64p = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_double)
        mp = (u16p * max(n, 1))(*[m.ctypes.data_as(u16p) for m in models])
        sK = np.ascontiguousarray(sceneK, np.float32).reshape(9)
        mK = np.ascontiguousarray(modelKs, np.float32).reshape(n, 9)
        R = np.ascontiguousarray(Rs, np.float32).reshape(n, 9)
        t = np.ascontiguousarray(ts, np.float32).reshape(n, 3)
        xy = np.ascontiguousarray(detect_xy, np.int32).reshape(n, 2)
        Ro = np.full((n, 3, 3), np.nan, np.float64)
        to = np.full((n, 3), np.nan, np.float64)
        res = np.zeros(n, np.float32)
        mrows, mcols = (models[0].shape if n else (1, 1))
        check(self._L.lm_icp_process_batch(self._h, n, scene.ctypes.data_as(u16p), scene.shape[0], scene.shape[1], mp, mrows, mcols,
                                           sK.ctypes.data_as(f32p), mK.ctypes.data_as(f32p), R.ctypes.data_as(f32p),
                                           t.ctypes.data_as(f32p), xy.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                           int(max_iterations), Ro.ctypes.data_as(f64p), to.ctypes.data_as(f64p),
                                           res.ctypes.data_as(f32p)))
        return Ro, to, res

    def set_use_scene_cloud(self, on):
        check(self._L.lm_icp_set_use_scene_cloud(self._h, 1 if on else 0))

    def last_stats(self):
        a = (ctypes.c_double * 4)()
        check(self._L.lm_icp_last_stats(self._h, a))
        return dict(points=int(a[0]), iterations=int(a[1]), rmse=float(a[2]), kernel_us=float(a[3]))

    def launch_count(self):
        return int(self._L.lm_icp_launch_count(self._h))
