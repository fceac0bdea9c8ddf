"""cofusion_b200 -- Python harness around libcofusion_b200.so (the C ABI of include/cofusion_b200.h).

The product is the CUDA library; this package only loads it, declares the prototypes and gives the
tests / bench a thin object layer.  PyTorch is used by callers for device memory and streams
(`tensor.data_ptr()` is what crosses the ABI).  There is NO CPU fallback: if the extension is not
built, or no CUDA device is visible, the constructors raise.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CFB_LIB_PATH") or os.path.join(_HERE, "libcofusion_b200.so")  # (override: A/B builds in tools)
_lib = None

c_float_p = C.POINTER(C.c_float)
c_void_pp = C.POINTER(C.c_void_p)


class TrackStats(C.Structure):
    _fields_ = [("lastICPError", C.c_float), ("lastICPCount", C.c_float), ("lastRGBError", C.c_float),
                ("lastRGBCount", C.c_float), ("lastSO3Error", C.c_float), ("lastSO3Count", C.c_float),
                ("lastA", C.c_double * 36), ("lastb", C.c_double * 6), ("so3_iterations", C.c_int),
                ("pad_", C.c_int)]


class CfbError(RuntimeError):
    pass


def lib():
    """Load libcofusion_b200.so (raises if it has not been built -- no silent fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CfbError("libcofusion_b200.so is missing: run `python -c 'import __graft_entry__ as g; "
                           "g.build()'` (there is no CPU fallback)")
        _lib = C.CDLL(LIB_PATH)
        _lib.cfb_last_error.restype = C.c_char_p
        _lib.cfb_step_scratch_bytes.restype = C.c_size_t
    return _lib


def check(rc):
    if rc != 0:
        raise CfbError("cfb error %d: %s" % (rc, lib().cfb_last_error().decode()))


def _p(t):
    """device pointer of a torch tensor (or None)"""
    return C.c_void_p(0 if t is None else t.data_ptr())


def _f(a):
    a = np.ascontiguousarray(a, dtype=np.float32)
    return a.ctypes.data_as(c_float_p), a


def _stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Odometry:
    """cfb_odom_* = RGBDOdometry (Core/Utils/RGBDOdometry.h). Inputs are torch CUDA tensors."""

    def __init__(self, W, H, K, dist_thresh=0.10, angle_thresh=float(np.sin(np.deg2rad(20.0)))):
        fx, fy, cx, cy = K
        self.W, self.H, self.K = W, H, K
        self._h = C.c_void_p()
        check(lib().cfb_odom_create(W, H, C.c_float(cx), C.c_float(cy), C.c_float(fx), C.c_float(fy),
                                    C.c_float(dist_thresh), C.c_float(angle_thresh), C.byref(self._h)))

    def __del__(self):
        if getattr(self, "_h", None) and self._h.value and _lib is not None:
            _lib.cfb_odom_destroy(self._h)
            self._h = C.c_void_p()

    def init_icp(self, depth_pyr, cutoff):
        ptrs = (C.c_void_p * 3)(*[d.data_ptr() for d in depth_pyr])
        pitch = (C.c_size_t * 3)(*[d.stride(0) * 4 for d in depth_pyr])
        check(lib().cfb_odom_init_icp(self._h, ptrs, pitch, C.c_float(cutoff), _stream()))

    def init_icp_model(self, v4, n4, cutoff, pose):
        pp, keep = _f(pose)
        check(lib().cfb_odom_init_icp_model(self._h, _p(v4), _p(n4), C.c_float(cutoff), pp, _stream()))

    def init_rgb_model(self, img):
        check(lib().cfb_odom_init_rgb_model(self._h, _p(img), C.c_size_t(img.stride(0)), img.shape[2], _stream()))

    def init_rgb(self, img):
        check(lib().cfb_odom_init_rgb(self._h, _p(img), C.c_size_t(img.stride(0)), img.shape[2], _stream()))

    def init_first_rgb(self, img):
        check(lib().cfb_odom_init_first_rgb(self._h, _p(img), C.c_size_t(img.stride(0)), img.shape[2], _stream()))

    def track(self, pose, rgb_only=False, icp_weight=10.0, pyramid=True, fast_odom=False, so3=True,
              error_map=None, force_host_loop=False):
        """getIncrementalTransformation; pose: 4x4 camera->world (numpy) -> new 4x4 + stats."""
        pose = np.asarray(pose, dtype=np.float32)
        trans = np.ascontiguousarray(pose[:3, 3]).copy()
        rot = np.ascontiguousarray(pose[:3, :3]).copy()
        st = TrackStats()
        check(lib().cfb_odom_get_incremental_transformation(
            self._h, trans.ctypes.data_as(c_float_p), rot.ctypes.data_as(c_float_p), int(rgb_only),
            C.c_float(icp_weight), int(pyramid), int(fast_odom), int(so3), _p(error_map),
            C.c_size_t(0 if error_map is None else error_map.stride(0) * 4), int(force_host_loop), C.byref(st),
            _stream()))
        out = np.eye(4, dtype=np.float32)
        out[:3, :3] = rot
        out[:3, 3] = trans
        return out, st

    def view(self, which, level):
        """copy of an internal pyramid buffer as a numpy array"""
        import torch
        ptr, pitch = C.c_void_p(), C.c_size_t()
        check(lib().cfb_odom_view(self._h, which, level, C.byref(ptr), C.byref(pitch)))
        w, h = self.W >> level, self.H >> level
        shapes = {0: (3 * h, w, np.float32), 1: (3 * h, w, np.float32), 2: (3 * h, w, np.float32),
                  3: (3 * h, w, np.float32), 4: (h, w, np.float32), 5: (h, w, np.float32), 6: (h, w, np.uint8),
                  7: (h, w, np.uint8), 8: (h, w, np.int16), 9: (h, w, np.int16), 10: (h, w, np.uint8),
                  11: (h, w * 3, np.float32), 12: (h, w * 4, np.int32)}
        r, c, dt = shapes[which]
        out = np.empty((r, c), dtype=dt)
        torch.cuda.synchronize()
        _cudart_memcpy_d2h(out, ptr.value)
        return out


def _cudart_memcpy_d2h(dst_np, src_ptr):
    check(lib().cfb_download(dst_np.ctypes.data_as(C.c_void_p), C.c_void_p(src_ptr), C.c_size_t(dst_np.nbytes),
                             _stream()))


class TrackParams(C.Structure):
    _fields_ = [("frameToFrameRGB", C.c_int), ("rgbOnly", C.c_int), ("icpWeight", C.c_float), ("pyramid", C.c_int),
                ("fastOdom", C.c_int), ("so3", C.c_int), ("maxDepthProcessed", C.c_float), ("force_host_loop", C.c_int)]

    @staticmethod
    def default():  # CoFusion.cpp:51-60 / GUI defaults
        return TrackParams(0, 0, 10.0, 1, 0, 1, 20.0, 0)


class Context:
    """cfb_ctx_*: per-device frame state (RGB, raw/filtered depth, depth pyramid, mask)."""

    def __init__(self, W, H, K, device=0):
        fx, fy, cx, cy = K
        self.W, self.H, self.K = W, H, K
        self._h = C.c_void_p()
        check(lib().cfb_ctx_create(device, W, H, C.c_float(fx), C.c_float(fy), C.c_float(cx), C.c_float(cy),
                                   C.byref(self._h)))
        lib().cfb_ctx_stream.restype = C.c_void_p
        self.stream = lib().cfb_ctx_stream(self._h)

    def __del__(self):
        if getattr(self, "_h", None) and self._h.value and _lib is not None:
            _lib.cfb_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def upload_frame(self, rgb, depth, mask=None):
        """host numpy arrays or pinned torch tensors"""
        def hp(a):
            if a is None:
                return C.c_void_p(0)
            if hasattr(a, "data_ptr"):
                return C.c_void_p(a.data_ptr())
            return a.ctypes.data_as(C.c_void_p)
        check(lib().cfb_ctx_upload_frame(self._h, hp(rgb), hp(depth), hp(mask)))

    def set_frame_device(self, rgb, depth, mask=None):
        check(lib().cfb_ctx_set_frame_device(self._h, _p(rgb), _p(depth), _p(mask)))

    def preprocess(self, depth_cutoff):
        check(lib().cfb_ctx_preprocess(self._h, C.c_float(depth_cutoff)))

    def sync(self):
        check(lib().cfb_ctx_sync(self._h))

    def take_launch_count(self):
        return lib().cfb_ctx_take_launch_count(self._h)

    def view(self, which):
        ptr, pitch = C.c_void_p(), C.c_size_t()
        check(lib().cfb_ctx_view(self._h, which, C.byref(ptr), C.byref(pitch)))
        W, H = self.W, self.H
        shp = {0: ((H, W, 3), np.uint8), 1: ((H, W), np.float32), 2: ((H, W), np.float32),
               3: ((H // 2, W // 2), np.float32), 4: ((H // 4, W // 4), np.float32), 5: ((H, W), np.uint8)}[which]
        out = np.empty(shp[0], dtype=shp[1])
        self.sync()
        check(lib().cfb_download(out.ctypes.data_as(C.c_void_p), ptr, C.c_size_t(out.nbytes), C.c_void_p(self.stream)))
        return out


class Model:
    """cfb_model_*: Core/Model/Model.h without OpenGL."""

    def __init__(self, ctx, model_id=0, conf_threshold=10.0, max_surfels=1 << 20, enable_fill_in=True):
        self.ctx = ctx
        self._h = C.c_void_p()
        check(lib().cfb_model_create(ctx._h, model_id, C.c_float(conf_threshold), max_surfels, int(enable_fill_in),
                                     C.byref(self._h)))
        lib().cfb_model_compute_fusion_weight.restype = C.c_float

    def __del__(self):
        if getattr(self, "_h", None) and self._h.value and _lib is not None:
            _lib.cfb_model_destroy(self._h)
            self._h = C.c_void_p()

    @property
    def pose(self):
        p = np.zeros(16, np.float32)
        check(lib().cfb_model_get_pose(self._h, p.ctypes.data_as(c_float_p)))
        return p.reshape(4, 4)

    def override_pose(self, pose):
        pp, keep = _f(np.asarray(pose, np.float32).reshape(16))
        check(lib().cfb_model_override_pose(self._h, pp))

    def set_confidence_threshold(self, v):
        check(lib().cfb_model_set_confidence_threshold(self._h, C.c_float(v)))

    def info(self):
        """(id, confidence threshold, max depth)"""
        i, c, d = C.c_uint(0), C.c_float(0), C.c_float(0)
        check(lib().cfb_model_get_info(self._h, C.byref(i), C.byref(c), C.byref(d)))
        return i.value, c.value, d.value

    def set_max_depth(self, v):
        check(lib().cfb_model_set_max_depth(self._h, C.c_float(v)))

    def set_prediction(self, v4, n4, img):
        dev = hasattr(v4, "data_ptr")
        if dev:
            check(lib().cfb_model_set_prediction(self._h, _p(v4), _p(n4), _p(img), img.shape[2], 1))
        else:
            v4 = np.ascontiguousarray(v4, np.float32)
            n4 = np.ascontiguousarray(n4, np.float32)
            img = np.ascontiguousarray(img, np.uint8)
            check(lib().cfb_model_set_prediction(self._h, v4.ctypes.data_as(C.c_void_p), n4.ctypes.data_as(C.c_void_p),
                                                 img.ctypes.data_as(C.c_void_p), img.shape[2], 0))
            self.ctx.sync()

    def init_first_rgb(self):
        check(lib().cfb_model_init_first_rgb(self._h))

    def perform_tracking(self, params=None):
        params = params or TrackParams.default()
        pose = np.zeros(16, np.float32)
        st = TrackStats()
        check(lib().cfb_model_perform_tracking(self._h, C.byref(params), pose.ctypes.data_as(c_float_p), C.byref(st)))
        return pose.reshape(4, 4), st

    def odometry_view(self, which, level):
        """numpy copy of one of the tracker's internal pyramid buffers (see cfb_odom_view)"""
        lib().cfb_model_odometry.restype = C.c_void_p
        o = Odometry.__new__(Odometry)
        o.W, o.H, o.K = self.ctx.W, self.ctx.H, self.ctx.K
        o._h = C.c_void_p(lib().cfb_model_odometry(self._h))
        o.__class__ = type("BorrowedOdometry", (Odometry,), {"__del__": lambda self_: None})
        self.ctx.sync()
        return o.view(which, level)

    def initialise(self, time, max_depth=20.0):
        check(lib().cfb_model_initialise(self._h, int(time), C.c_float(max_depth)))

    def predict_indices(self, time, depth_cutoff=20.0, time_delta=200):
        check(lib().cfb_model_predict_indices(self._h, int(time), C.c_float(depth_cutoff), int(time_delta)))

    def fuse(self, time, depth_cutoff=20.0, weight_multiplier=1.0):
        check(lib().cfb_model_fuse(self._h, int(time), C.c_float(depth_cutoff), C.c_float(weight_multiplier)))

    def clean(self, time, time_delta=200, depth_cutoff=20.0, outlier_coefficient=3.0):
        check(lib().cfb_model_clean(self._h, int(time), int(time_delta), C.c_float(depth_cutoff),
                                    C.c_float(outlier_coefficient)))

    def combined_predict(self, depth_cutoff, time, max_time, time_delta=200):
        check(lib().cfb_model_combined_predict(self._h, C.c_float(depth_cutoff), int(time), int(max_time),
                                               int(time_delta)))

    def perform_fill_in(self, frame_to_frame_rgb=False, lost=False):
        check(lib().cfb_model_perform_fill_in(self._h, int(frame_to_frame_rgb), int(lost)))

    def fusion_weight(self, mult=1.0):
        return float(lib().cfb_model_compute_fusion_weight(self._h, C.c_float(mult)))

    def download_map(self):
        n = C.c_uint(0)
        check(lib().cfb_model_last_count(self._h, C.byref(n)))
        out = np.zeros((n.value, 12), np.float32)
        if n.value:
            check(lib().cfb_model_download_map(self._h, out.ctypes.data_as(c_float_p), C.c_size_t(n.value), C.byref(n)))
        return out

    def upload_map(self, surfels):
        s = np.ascontiguousarray(surfels, np.float32)
        check(lib().cfb_model_upload_map(self._h, s.ctypes.data_as(c_float_p), s.shape[0]))

    def last_count(self):
        n = C.c_uint(0)
        check(lib().cfb_model_last_count(self._h, C.byref(n)))
        return n.value

    VIEWS = {0: (4, np.float32), 1: (4, np.float32), 2: (4, np.uint8), 3: (1, np.float32), 4: (1, np.uint32),
             5: (4, np.float32), 6: (4, np.float32), 7: (4, np.float32), 8: (4, np.uint8), 9: (4, np.float32),
             10: (4, np.float32), 11: (1, np.uint16), 12: (4, np.uint8), 13: (4, np.float32), 14: (4, np.float32)}

    def view_ptr(self, which):
        """raw device pointer of a model buffer (see cfb_model_view)"""
        ptr, pitch = C.c_void_p(), C.c_size_t()
        check(lib().cfb_model_view(self._h, which, C.byref(ptr), C.byref(pitch)))
        return ptr.value

    def view(self, which, n_unstable=0):
        ptr, pitch = C.c_void_p(), C.c_size_t()
        check(lib().cfb_model_view(self._h, which, C.byref(ptr), C.byref(pitch)))
        W, H = self.ctx.W, self.ctx.H
        if which == 15:
            out = np.empty((n_unstable, 12), np.float32)
        else:
            ch, dt = self.VIEWS[which]
            out = np.empty((H, W, ch) if ch > 1 else (H, W), dtype=dt)
        self.ctx.sync()
        if out.nbytes:
            check(lib().cfb_download(out.ctypes.data_as(C.c_void_p), ptr, C.c_size_t(out.nbytes),
                                     C.c_void_p(self.ctx.stream)))
        return out


class SegParams(C.Structure):  # cfb_seg_params
    _fields_ = [("crfIterations", C.c_int), ("scaleFeaturesRGB", C.c_float), ("scaleFeaturesDepth", C.c_float),
                ("scaleFeaturesPos", C.c_float), ("weightAppearance", C.c_float), ("weightSmoothness", C.c_float),
                ("unaryThresholdNew", C.c_float), ("unaryKError", C.c_float), ("unaryWeightError", C.c_float),
                ("maxRelSizeNew", C.c_float), ("minRelSizeNew", C.c_float)]

    @staticmethod
    def default():
        p = SegParams()
        lib().cfb_seg_default_params(C.byref(p))
        return p


class ModelData(C.Structure):  # cfb_model_data
    _fields_ = [("id", C.c_uint), ("superPixelCount", C.c_uint), ("avgConfidence", C.c_float),
                ("depthMean", C.c_float), ("depthStd", C.c_float), ("top", C.c_ushort), ("right", C.c_ushort),
                ("bottom", C.c_ushort), ("left", C.c_ushort)]

    def astuple(self):
        return (self.id, self.superPixelCount, self.avgConfidence, self.depthMean, self.depthStd, self.top,
                self.right, self.bottom, self.left)


SEG_MAX_MODELS = 15


class Segmentation:
    """cfb_segmentation_*: Segmentation::performSegmentationCRF on device buffers (torch CUDA tensors)."""

    def __init__(self, W, H, device=0, _borrowed=None):
        self.W, self.H, self.N = W, H, (W // 16) * (H // 16)
        self._owned = _borrowed is None
        self._h = C.c_void_p()
        if _borrowed is None:
            check(lib().cfb_segmentation_create(device, W, H, C.byref(self._h)))
        else:
            self._h = _borrowed
        self.num_labels = 0
        self.num_models = 0

    def __del__(self):
        if getattr(self, "_owned", False) and self._h.value and _lib is not None:
            _lib.cfb_segmentation_destroy(self._h)
            self._h = C.c_void_p()

    def slic(self, rgb):
        check(lib().cfb_segmentation_slic(self._h, _p(rgb), _stream()))
        return self.view(0)

    def perform_crf(self, rgb, depth, model_ids, icp_errors, vert_confs, next_model_id, allow_new, params=None):
        """All image arguments are CUDA tensors.  Returns (fullSeg u8 HxW tensor, [ModelData], hasNew)."""
        import torch
        n = len(model_ids)
        prm = params or SegParams.default()
        ids = (C.c_ubyte * n)(*model_ids)
        dp = lambda t: t.data_ptr() if hasattr(t, "data_ptr") else int(t)  # tensors or raw device pointers
        icp = (C.c_void_p * n)(*[dp(t) for t in icp_errors])
        vc = (C.c_void_p * n)(*[dp(t) for t in vert_confs])
        full = torch.empty((self.H, self.W), dtype=torch.uint8, device=rgb.device)
        md = (ModelData * (n + 1))()
        cnt, has_new = C.c_int(0), C.c_int(0)
        check(lib().cfb_segmentation_perform_crf(self._h, _p(rgb), _p(depth), n, ids, icp, vc,
                                                 C.c_ubyte(next_model_id), int(bool(allow_new)), C.byref(prm),
                                                 _p(full), md, C.byref(cnt), C.byref(has_new), _stream()))
        self.num_models, self.num_labels = n, n + int(bool(allow_new))
        return full, [md[i] for i in range(cnt.value)], bool(has_new.value)

    def view(self, which):
        """0 SLIC labels, 1 counts, 2 unary, 3 low-res map, 4 low-res maps, 5 Q (numpy copies)"""
        ptr, nbytes = C.c_void_p(), C.c_size_t()
        check(lib().cfb_segmentation_view(self._h, which, C.byref(ptr), C.byref(nbytes)))
        dt = {0: np.int32, 1: np.uint32, 2: np.float32, 3: np.uint8, 4: np.float32, 5: np.float32}[which]
        out = np.empty(nbytes.value // np.dtype(dt).itemsize, dt)
        _cudart_memcpy_d2h(out, ptr.value)
        if which == 0:
            return out.reshape(self.H, self.W)
        if which in (2, 5):
            return out.reshape(self.N, -1)
        if which == 4:
            return out.reshape(-1, self.N)
        return out


class CoFusionParams(C.Structure):
    _fields_ = [("timeDelta", C.c_int), ("depthCutoff", C.c_float), ("maxDepthProcessed", C.c_float),
                ("icpWeight", C.c_float), ("pyramid", C.c_int), ("fastOdom", C.c_int), ("so3", C.c_int),
                ("frameToFrameRGB", C.c_int), ("rgbOnly", C.c_int), ("confGlobalInit", C.c_float),
                ("confObjectInit", C.c_float), ("outlierCoefficient", C.c_float), ("maxSurfels", C.c_uint),
                ("predictBeforeFuse", C.c_int), ("enableMultipleModels", C.c_int),
                ("modelSpawnOffset", C.c_uint), ("seg", SegParams)]

    @staticmethod
    def default(max_surfels=1 << 21):
        p = CoFusionParams()
        lib().cfb_cofusion_default_params(C.byref(p))
        p.maxSurfels = max_surfels
        return p


def nccl_unique_id():
    """128-byte NCCL unique id (rank 0 creates it, the application distributes it)"""
    buf = (C.c_ubyte * 128)()
    check(lib().cfb_nccl_unique_id(buf))
    return bytes(buf)


def shard_owner(index, world):
    """rank that owns the model at list position `index` of a scene sharded over `world` ranks (shard.cuh)"""
    return index % world if world > 0 else 0


class Frame(C.Structure):  # cfb_frame
    _fields_ = [("rgb", C.c_void_p), ("depth", C.c_void_p), ("depth_u16", C.c_void_p), ("depth_scale", C.c_float),
                ("flip_colors", C.c_int), ("mask", C.c_void_p), ("device_ptrs", C.c_int), ("timestamp", C.c_int64)]


class _Borrowed:
    pass


class CoFusion:
    """cfb_cofusion_*: CoFusion::processFrame for the models of one device."""

    def __init__(self, W, H, K, params=None, device=0):
        fx, fy, cx, cy = K
        self.W, self.H, self.K = W, H, K
        self.params = params or CoFusionParams.default()
        self._h = C.c_void_p()
        check(lib().cfb_cofusion_create(device, W, H, C.c_float(fx), C.c_float(fy), C.c_float(cx), C.c_float(cy),
                                        C.byref(self.params), C.byref(self._h)))
        lib().cfb_cofusion_model.restype = C.c_void_p
        lib().cfb_cofusion_ctx.restype = C.c_void_p
        lib().cfb_ctx_stream.restype = C.c_void_p
        self.ctx = Context.__new__(Context)
        self.ctx.W, self.ctx.H, self.ctx.K = W, H, K
        self._ctx_h = C.c_void_p(lib().cfb_cofusion_ctx(self._h))
        self.ctx._h = self._ctx_h  # borrowed (BorrowedContext has no __del__): never destroyed from Python
        self.ctx.__class__ = type("BorrowedContext", (Context,), {"__del__": lambda self_: None})
        self.ctx.stream = lib().cfb_ctx_stream(self._ctx_h)
        self.ctx.sync = lambda: check(lib().cfb_ctx_sync(self._ctx_h))
        self.ctx.take_launch_count = lambda: lib().cfb_ctx_take_launch_count(self._ctx_h)

    def __del__(self):
        if getattr(self, "_h", None) and self._h.value and _lib is not None:
            _lib.cfb_cofusion_destroy(self._h)
            self._h = C.c_void_p()

    def _checked(self, a, dtype, shape, what):
        """dtype / shape / contiguity of an image crossing the ABI (raw pointers carry none of it)"""
        if a is None:
            return None
        if hasattr(a, "data_ptr"):  # torch tensor (CUDA, or pinned / pageable host)
            import torch
            want = {np.uint8: torch.uint8, np.float32: torch.float32, np.uint16: getattr(torch, "uint16", None)}[dtype]
            ok_dtype = a.dtype == want or (dtype is np.uint16 and a.dtype == torch.int16)
            if not ok_dtype or a.numel() != int(np.prod(shape)) or not a.is_contiguous():
                raise CfbError("%s: expected contiguous %s%s, got %s %s" % (what, np.dtype(dtype).name, shape, a.dtype, tuple(a.shape)))
            return a
        a = np.asarray(a)
        if a.dtype != dtype or a.size != int(np.prod(shape)):
            raise CfbError("%s: expected %s%s, got %s %s" % (what, np.dtype(dtype).name, shape, a.dtype, a.shape))
        return np.ascontiguousarray(a)

    @staticmethod
    def _ptr(a):
        if a is None:
            return C.c_void_p(0)
        if hasattr(a, "data_ptr"):
            return C.c_void_p(a.data_ptr())
        return a.ctypes.data_as(C.c_void_p)

    def shard_init(self, rank, world, unique_id):
        """collective: join the object-sharded job (one process per GPU); unique_id = nccl_unique_id() of rank 0"""
        buf = (C.c_ubyte * 128).from_buffer_copy(bytes(unique_id))
        check(lib().cfb_cofusion_shard_init(self._h, int(rank), int(world), buf))
        self.rank, self.world = rank, world

    def process_frame(self, rgb, depth, mask=None, weight_multiplier=1.0):
        """rgb/depth/mask: host numpy arrays, pinned torch tensors, or CUDA torch tensors (None on the ranks of a
        sharded job that are not the root: the frame arrives by broadcast)"""
        dev = hasattr(rgb, "is_cuda") and rgb.is_cuda
        rgb = self._checked(rgb, np.uint8, (self.H, self.W, 3), "rgb")
        depth = self._checked(depth, np.float32, (self.H, self.W), "depth")
        mask = self._checked(mask, np.uint8, (self.H, self.W), "mask")
        check(lib().cfb_cofusion_process_frame(self._h, self._ptr(rgb), self._ptr(depth), self._ptr(mask), int(dev),
                                               C.c_float(weight_multiplier)))

    def process_frame_ex(self, rgb, depth=None, depth_u16=None, depth_scale=0.001, flip_colors=False, mask=None,
                         in_pose=None, bootstrap=False, timestamp=0, weight_multiplier=1.0):
        """cfb_cofusion_process_frame_ex: CoFusion::processFrame(frame, inPose, weightMultiplier, bootstrap) with the
        log readers' conversions (u16 depth x scale, BGR flip) done on the device"""
        dev = hasattr(rgb, "is_cuda") and rgb.is_cuda
        fr = Frame()
        rgb = self._checked(rgb, np.uint8, (self.H, self.W, 3), "rgb")
        depth = self._checked(depth, np.float32, (self.H, self.W), "depth")
        depth_u16 = self._checked(depth_u16, np.uint16, (self.H, self.W), "depth_u16")
        mask = self._checked(mask, np.uint8, (self.H, self.W), "mask")
        fr.rgb, fr.depth, fr.depth_u16, fr.mask = (self._ptr(x).value for x in (rgb, depth, depth_u16, mask))
        fr.depth_scale, fr.flip_colors, fr.device_ptrs, fr.timestamp = depth_scale, int(flip_colors), int(dev), int(timestamp)
        pp = None
        if in_pose is not None:
            pa = np.ascontiguousarray(in_pose, np.float32).reshape(16)
            pp = pa.ctypes.data_as(c_float_p)
        check(lib().cfb_cofusion_process_frame_ex(self._h, C.byref(fr), pp, C.c_float(weight_multiplier), int(bool(bootstrap))))

    def enable_pose_logging(self, on=True):
        check(lib().cfb_cofusion_enable_pose_logging(self._h, int(bool(on))))

    def pose_log(self, index):
        n = C.c_int(0)
        check(lib().cfb_cofusion_pose_log(self._h, int(index), None, None, 0, C.byref(n)))
        ts = np.zeros(n.value, np.int64)
        p7 = np.zeros((n.value, 7), np.float32)
        if n.value:
            check(lib().cfb_cofusion_pose_log(self._h, int(index), ts.ctypes.data_as(C.c_void_p), p7.ctypes.data_as(C.c_void_p),
                                              n.value, C.byref(n)))
        return ts, p7

    def export_poses(self, directory):
        check(lib().cfb_cofusion_export_poses(self._h, str(directory).encode()))

    def save_ply(self, directory):
        check(lib().cfb_cofusion_save_ply(self._h, str(directory).encode()))

    def spawn_object_model(self, model_id, pose=None):
        pp = None
        if pose is not None:
            pa = np.ascontiguousarray(pose, np.float32).reshape(16)
            pp = pa.ctypes.data_as(c_float_p)
        check(lib().cfb_cofusion_spawn_object_model(self._h, int(model_id), pp))

    @property
    def num_models(self):
        return lib().cfb_cofusion_num_models(self._h)

    @property
    def tick(self):
        return lib().cfb_cofusion_tick(self._h)

    def model(self, index=0):
        m = Model.__new__(Model)
        m.ctx = self.ctx
        m._h = C.c_void_p(lib().cfb_cofusion_model(self._h, int(index)))
        m.__class__ = type("BorrowedModel", (Model,), {"__del__": lambda self_: None})
        lib().cfb_model_compute_fusion_weight.restype = C.c_float
        return m

    def pose(self, index=0):
        return self.model(index).pose

    def last_stats(self, index=0):
        st = TrackStats()
        check(lib().cfb_cofusion_last_stats(self._h, int(index), C.byref(st)))
        return st

    def ctx_view_mask(self):
        """textures[MASK]: the label image the fuse / clean stage of the last frame used (HxW u8)"""
        return self.ctx.view(5)

    def last_segmentation(self):
        """([ModelData], hasNewLabel, spawned_id or -1, deactivated) of the last frame"""
        md = (ModelData * (SEG_MAX_MODELS + 1))()
        cnt, hn, sp, de = C.c_int(0), C.c_int(0), C.c_int(-1), C.c_int(0)
        check(lib().cfb_cofusion_last_segmentation(self._h, md, C.byref(cnt), C.byref(hn), C.byref(sp), C.byref(de)))
        return [md[i] for i in range(cnt.value)], bool(hn.value), sp.value, de.value

    def set_batched_tracking(self, on):
        check(lib().cfb_cofusion_set_batched_tracking(self._h, int(bool(on))))

    @property
    def num_inactive_models(self):
        return lib().cfb_cofusion_num_inactive_models(self._h)

    def segmentation(self):
        lib().cfb_cofusion_segmentation.restype = C.c_void_p
        h = lib().cfb_cofusion_segmentation(self._h)
        return Segmentation(self.W, self.H, _borrowed=C.c_void_p(h)) if h else None
