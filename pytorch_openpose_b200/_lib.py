"""ctypes binding of libopenpose_b200.so (C ABI: include/openpose_b200.h).

This is the binding a maintainer of the reference would add next to src/body.py / src/hand.py (see
INTEGRATION.md).  There is no CPU fallback: if the shared library is missing or no sm_100 GPU is visible the
import / first call fails loudly."""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int64, c_uint8, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libopenpose_b200.so")

OPB_OK = 0
OPB_ERR_INVALID = -1
OPB_ERR_CUDA = -2
OPB_ERR_MISSING_LAYER = -3
OPB_ERR_CAPACITY = -4
OPB_ERR_SUBSET_INDEX = -5
OPB_ERR_NO_DEVICE = -6
NET_BODY, NET_HAND = 0, 1
JPEG_FALLBACK, JPEG_CORRUPT = 1, 2

# name -> (restype, argtypes); every symbol include/openpose_b200.h declares
SIGNATURES = {
    "opb_abi_version": (c_int, []),
    "opb_last_error": (c_char_p, []),
    "opb_context_create": (c_int, [c_int, POINTER(c_void_p)]),
    "opb_context_destroy": (c_int, [c_void_p]),
    "opb_context_synchronize": (c_int, [c_void_p]),
    "opb_context_launch_count": (c_int, [c_void_p, POINTER(c_int64)]),
    "opb_net_create": (c_int, [c_void_p, c_int, POINTER(c_void_p)]),
    "opb_net_load_layer": (c_int, [c_void_p, c_char_p, c_void_p, c_void_p, c_int, c_int, c_int]),
    "opb_net_finalize": (c_int, [c_void_p]),
    "opb_net_destroy": (c_int, [c_void_p]),
    "opb_net_layer_count": (c_int, [c_int]),
    "opb_net_layer_info": (c_int, [c_int, c_int, POINTER(c_char_p), POINTER(c_int), POINTER(c_int), POINTER(c_int),
                                   POINTER(c_int)]),
    "opb_session_create": (c_int, [c_void_p, POINTER(c_void_p)]),
    "opb_session_destroy": (c_int, [c_void_p]),
    "opb_session_set_profiling": (c_int, [c_void_p, c_int]),
    "opb_session_profile_count": (c_int, [c_void_p]),
    "opb_session_profile_get": (c_int, [c_void_p, c_int, POINTER(c_char_p), POINTER(c_float), POINTER(c_double)]),
    "opb_session_progress": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int), POINTER(c_char_p), POINTER(c_char_p)]),
    "opb_session_mark": (c_int, [c_void_p, c_int]),
    "opb_session_elapsed": (c_int, [c_void_p, c_int, c_void_p, c_int, POINTER(c_float)]),
    "opb_session_graph_stats": (c_int, [c_void_p, POINTER(ctypes.c_longlong), POINTER(ctypes.c_longlong)]),
    "opb_body_submit": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, POINTER(c_double), c_int]),
    "opb_body_wait": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int)]),
    "opb_body_fetch": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int]),
    "opb_body_submit_batch": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, POINTER(c_double), c_int]),
    "opb_body_wait_batch": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "opb_body_fetch_frame": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int]),
    "opb_hand_submit": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, POINTER(c_double), c_int]),
    "opb_hand_submit_ragged": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, POINTER(c_double), c_int]),
    "opb_hand_wait": (c_int, [c_void_p, c_void_p]),
    "opb_pose_submit_batch": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, POINTER(c_double), c_int,
                                      POINTER(c_double), c_int, c_void_p]),
    "opb_pose_wait": (c_int, [c_void_p, c_void_p, POINTER(c_int)]),
    "opb_pose_select": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "opb_pose_every_submit": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, POINTER(c_double), c_int,
                                      POINTER(c_double), c_int]),
    "opb_pose_every_wait": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int)]),
    "opb_pose_every_fetch": (c_int, [c_void_p, c_void_p, c_int]),
    "opb_pose_every_select": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "opb_tracker_create": (c_int, [c_void_p, c_int, c_double, c_int, POINTER(c_void_p)]),
    "opb_tracker_destroy": (c_int, [c_void_p]),
    "opb_tracker_reset": (c_int, [c_void_p]),
    "opb_tracker_state": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "opb_pose_every_wait_tracked": (c_int, [c_void_p, c_void_p, c_int, POINTER(c_int), POINTER(c_int)]),
    "opb_pose_every_fetch_ids": (c_int, [c_void_p, c_void_p, c_int]),
    "opb_tracker_link_host": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "opb_body_maps": (c_int, [c_void_p, c_void_p, c_void_p]),
    "opb_hand_maps": (c_int, [c_void_p, c_void_p]),
    "opb_batch_body_submit": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_double]),
    "opb_batch_hand_submit": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int]),
    "opb_batch_body_submit_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_double]),
    "opb_batch_hand_submit_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int]),
    "opb_batch_maps": (c_int, [c_void_p, c_void_p]),
    "opb_batch_debug_input": (c_int, [c_void_p, c_void_p]),
    "opb_hand_track_submit": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int]),
    "opb_hand_track_wait": (c_int, [c_void_p, c_void_p]),
    "opb_hand_track_crops": (c_int, [c_void_p, c_void_p]),
    "opb_hand_track_boxes": (c_int, [c_void_p, c_int, c_int, c_void_p]),
    "opb_debug_hand_track_taps": (c_int, [c_int, c_int, c_void_p, c_void_p]),
    "opb_batch_pose_submit": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_double, c_int]),
    "opb_batch_pose_wait": (c_int, [c_void_p, c_void_p, c_void_p, POINTER(c_int)]),
    "opb_batch_pose_every_submit": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_double, c_int]),
    "opb_batch_pose_every_select": (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_void_p,
                                            c_void_p]),
    "opb_scale_dims": (c_int, [c_int, c_int, c_double, POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "opb_preprocess": (c_int, [c_void_p, c_void_p, c_int, c_int, c_double, c_void_p]),
    "opb_net_forward": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "opb_upsample_avg": (c_int, [c_void_p, POINTER(c_void_p), POINTER(c_double), c_int, c_int, c_int, c_int, c_int,
                                 c_void_p]),
    "opb_find_peaks": (c_int, [c_void_p, c_void_p, c_int, c_int, c_double, c_void_p, c_int, POINTER(c_int),
                               POINTER(c_int)]),
    "opb_find_peaks_blurred": (c_int, [c_void_p, c_void_p, c_int, c_int, c_double, c_void_p, c_int, POINTER(c_int),
                               POINTER(c_int)]),
    "opb_group_limbs": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, POINTER(c_int), c_double, c_void_p, c_int,
                                POINTER(c_int), c_void_p, c_int, POINTER(c_int)]),
    "opb_hand_peaks": (c_int, [c_void_p, c_void_p, c_int, c_int, c_double, c_void_p]),
    "opb_hand_debug_post": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                    c_void_p, c_void_p, c_void_p]),
    "opb_debug_pairwise_sum": (c_int, [c_void_p, ctypes.c_longlong, c_int, POINTER(c_double)]),
    "opb_bench_grouping": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, POINTER(c_float), POINTER(c_int),
                                   POINTER(c_int)]),
    "opb_smooth_debug": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "opb_wide_pool_weights": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "opb_debug_resize_taps": (c_int, [c_int, c_int, ctypes.c_double, c_void_p, c_void_p]),
    "opb_debug_composite_taps": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p]),
    "opb_debug_resize_dsize": (c_int, [c_int, ctypes.c_double]),
    "opb_debug_batch_resize_taps": (c_int, [c_int, c_int, ctypes.c_double, c_void_p, c_void_p]),
    "opb_debug_batch_composite_taps": (c_int, [c_int, c_int, c_int, c_void_p, c_void_p]),
    "opb_debug_pair_tiles": (c_int, [c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "opb_net_debug_plan": (c_int, [c_void_p, c_int, c_void_p, POINTER(c_int)]),
    "opb_net_debug_set_input": (c_int, [c_void_p, c_int, c_void_p]),
    "opb_net_debug_info": (c_int, [c_void_p, c_int, c_void_p]),
    "opb_net_debug_step": (c_int, [c_void_p, c_int, c_void_p]),
    "opb_net_debug_read": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p]),
    "opb_net_debug_run": (c_int, [c_void_p]),
    "opb_body_debug_post_dims": (c_int, [c_int, c_int, POINTER(c_double), c_int, c_int, c_void_p, POINTER(c_int)]),
    "opb_body_debug_post_submit": (c_int, [c_void_p, c_int, c_int, c_int, POINTER(c_double), c_int, c_int,
                                           POINTER(c_void_p), POINTER(c_void_p)]),
    "opb_body_debug_part_begin": (c_int, [c_void_p, c_int, c_void_p]),
    "opb_jpeg_submit": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, POINTER(c_void_p),
                                POINTER(c_int), POINTER(c_int)]),
    "opb_jpeg_upload": (c_int, [c_void_p, c_int, c_void_p]),
    "opb_jpeg_fetch": (c_int, [c_void_p, c_void_p]),
    "opb_jpeg_status": (c_int, [c_void_p, c_void_p]),
    "opb_jpeg_decode_host": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, POINTER(c_int), POINTER(c_int),
                                     POINTER(c_int)]),
    "opb_conv2d": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int,
                           c_int, c_int, c_void_p, c_int]),
}

_lib = None


class OpbError(RuntimeError):
    def __init__(self, code, message):
        super().__init__("libopenpose_b200 error %d: %s" % (code, message))
        self.code = code


def lib():
    """The loaded library (loads on first use).  Raises ImportError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s not found: build it with `python -m pytorch_openpose_b200.build` "
                              "(there is no CPU fallback)" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError here == header/library mismatch
            fn.restype = res
            fn.argtypes = args
        if L.opb_abi_version() != 1:
            raise ImportError("libopenpose_b200 ABI version mismatch")
        _lib = L
    return _lib


def check(rc):
    """Translate a return code into the exception the reference would raise at that point."""
    if rc == OPB_OK:
        return
    msg = lib().opb_last_error().decode("utf-8", "replace")
    if rc == OPB_ERR_MISSING_LAYER:
        raise KeyError(msg)                 # util.transfer: model_weights[missing key], src/util.py:39
    if rc == OPB_ERR_SUBSET_INDEX:
        raise IndexError(msg)               # src/body.py:173
    raise OpbError(rc, msg)


_contexts = {}


def context(device=None):
    """One library context per GPU of this process."""
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0")) if "OPB_DEVICE" not in os.environ else int(os.environ["OPB_DEVICE"])
        try:
            import torch
            if torch.cuda.is_available() and "OPB_DEVICE" not in os.environ:
                device = torch.cuda.current_device()
        except Exception:
            pass
    if device not in _contexts:
        h = c_void_p()
        check(lib().opb_context_create(int(device), ctypes.byref(h)))
        _contexts[device] = h
    return _contexts[device]


def launch_count(device=None):
    n = c_int64()
    check(lib().opb_context_launch_count(context(device), ctypes.byref(n)))
    return n.value


def layer_table(kind):
    """[(name, cout, cin, k, relu)] of the architecture, as the library expects it."""
    L = lib()
    out = []
    for i in range(L.opb_net_layer_count(kind)):
        name, co, ci, k, relu = c_char_p(), c_int(), c_int(), c_int(), c_int()
        check(L.opb_net_layer_info(kind, i, ctypes.byref(name), ctypes.byref(co), ctypes.byref(ci), ctypes.byref(k),
                                   ctypes.byref(relu)))
        out.append((name.value.decode(), co.value, ci.value, k.value, bool(relu.value)))
    return out


class Net(object):
    """Device weights of one CNN, built from a caffe-keyed flat state dict (the reference checkpoint format)."""

    def __init__(self, kind, weights, device=None):
        import numpy as np
        L = lib()
        self.kind = kind
        self.ctx = context(device)
        self.handle = c_void_p()
        check(L.opb_net_create(self.ctx, kind, ctypes.byref(self.handle)))
        for name, cout, cin, k, _ in layer_table(kind):
            w = weights[name + ".weight"]          # KeyError on a missing layer, like util.transfer
            b = weights[name + ".bias"]
            w = np.ascontiguousarray(_to_numpy(w), dtype=np.float32)
            b = np.ascontiguousarray(_to_numpy(b), dtype=np.float32)
            if w.shape != (cout, cin, k, k) or b.shape != (cout,):
                raise RuntimeError("size mismatch for %s: checkpoint %s vs model %s" % (name, w.shape, (cout, cin, k, k)))
            check(L.opb_net_load_layer(self.handle, name.encode(), w.ctypes.data, b.ctypes.data, cout, cin, k))
        check(L.opb_net_finalize(self.handle))

    def session(self):
        return Session(self)

    def __del__(self):
        try:
            if self.handle:
                lib().opb_net_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class Session(object):
    def __init__(self, net):
        self.net = net
        self.handle = c_void_p()
        check(lib().opb_session_create(net.handle, ctypes.byref(self.handle)))

    def set_profiling(self, on):
        check(lib().opb_session_set_profiling(self.handle, int(on)))

    def profile(self):
        """[(mark name, ms since previous mark, algorithmic GFLOP)] of the last profiled frame."""
        L = lib()
        out = []
        for i in range(L.opb_session_profile_count(self.handle)):
            name, ms, gf = c_char_p(), c_float(), c_double()
            check(L.opb_session_profile_get(self.handle, i, ctypes.byref(name), ctypes.byref(ms), ctypes.byref(gf)))
            out.append((name.value.decode(), ms.value, gf.value))
        return out

    def progress(self):
        """(index of the last completed profile mark, total marks, its name, name of the next one) -- debugging."""
        d, t, a, b = c_int(), c_int(), c_char_p(), c_char_p()
        check(lib().opb_session_progress(self.handle, ctypes.byref(d), ctypes.byref(t), ctypes.byref(a), ctypes.byref(b)))
        return d.value, t.value, (a.value or b"").decode(), (b.value or b"").decode()

    def mark(self, slot):
        check(lib().opb_session_mark(self.handle, slot))

    def elapsed_ms(self, slot_a, other, slot_b):
        ms = c_float()
        check(lib().opb_session_elapsed(self.handle, slot_a, other.handle, slot_b, ctypes.byref(ms)))
        return ms.value

    def __del__(self):
        try:
            if self.handle:
                lib().opb_session_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class Tracker(object):
    """Person tracks of one video on the device (opb_tracker_*): the rule of `motion.PersonLinker`, bit for bit."""

    def __init__(self, ctx, max_gap, max_dist, min_joints=3):
        self.handle = c_void_p()
        check(lib().opb_tracker_create(ctx, int(max_gap), float(max_dist), int(min_joints), ctypes.byref(self.handle)))

    def reset(self):
        check(lib().opb_tracker_reset(self.handle))

    def state(self):
        """(live tracks, next id, frames linked so far)."""
        live, nxt, frame = c_int(), c_int(), c_int()
        check(lib().opb_tracker_state(self.handle, ctypes.byref(live), ctypes.byref(nxt), ctypes.byref(frame)))
        return live.value, nxt.value, frame.value

    def link_host(self, frames):
        """frames: a list of (P_f, 60, 3) float64 record arrays -> list of (P_f,) int track ids, linked on the device."""
        import numpy as np
        counts = np.array([len(r) for r in frames], dtype=np.int32)
        records = np.ascontiguousarray(np.concatenate([np.asarray(r, dtype=np.float64).reshape(-1, 60, 3) for r in frames])
                                       if len(frames) else np.zeros((0, 60, 3)))
        ids = np.empty(len(records), dtype=np.int32)
        check(lib().opb_tracker_link_host(self.handle, records.ctypes.data, counts.ctypes.data, len(counts), ids.ctypes.data))
        return np.split(ids.astype(np.int64), np.cumsum(counts)[:-1]) if len(counts) else []

    def __del__(self):
        try:
            if self.handle:
                lib().opb_tracker_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


def _to_numpy(t):
    if hasattr(t, "detach"):
        return t.detach().cpu().numpy()
    return t


def scales_array(scale_search):
    arr = (c_double * len(scale_search))(*[float(s) for s in scale_search])
    return arr, len(scale_search)
