"""ctypes binding of libb200pose.so (include/b200pose.h).  Loading is lazy; every failure is loud."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200POSE_LIB selects another build of the same library (tools/variants.py: compile-time tuning variants); there is
# still no fallback of any kind - a missing file is an error.
LIB_PATH = os.environ.get("B200POSE_LIB") or os.path.join(_HERE, "libb200pose.so")
_lib = None

c_float_p = ctypes.POINTER(ctypes.c_float)
NUM_TENSORS = 184
HUMAN_FLOATS = 73
MODE_BF16, MODE_FP32, MODE_BF16X3 = 0, 1, 2
MODES = {"bf16": MODE_BF16, "fp32": MODE_FP32, "bf16x3": MODE_BF16X3}
PREPROCESS = {"rtpose": 1, "vgg": 2, "inception": 3, "ssd": 4}      # get_outputs' `preprocess` names


class B200PoseError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200PoseError("%s is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(there is no CPU/PyTorch fallback for this path)" % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, ci, cl, cf = ctypes.c_void_p, ctypes.c_int, ctypes.c_long, ctypes.c_float
    sig = {
        "b200pose_last_error": ([], ctypes.c_char_p),
        "b200pose_version": ([], ci),
        "b200pose_launch_count": ([], cl),
        "b200pose_net_create": ([ctypes.POINTER(vp), ci], ci),
        "b200pose_net_destroy": ([vp], None),
        "b200pose_net_tensor_shape": ([ci, ctypes.POINTER(cl)], ci),
        "b200pose_net_set_tensor": ([vp, ci, vp, cl], ci),
        "b200pose_net_finalize": ([vp], ci),
        "b200pose_net_forward": ([vp, vp, ci, ci, ci, ci, ci, ctypes.POINTER(vp), ci, vp], ci),
        "b200pose_net_forward_u8": ([vp, vp, ci, ci, ci, ci, ci, ctypes.POINTER(vp), ci, vp], ci),
        "b200pose_net_set_preprocess": ([vp, ci], ci),
        "b200pose_net_forward_u8_ragged": ([vp, vp, ci, ci, ci, ci, vp, vp, ci, ctypes.POINTER(vp), ci, vp], ci),
        "b200pose_infer_raw_u8_ragged": ([vp, vp, vp, ci, ci, vp, vp, ci, ci, ci, cf, vp], ci),
        "b200pose_ragged_layout": ([ci, vp, vp, ci, ci, vp, vp, vp, ctypes.POINTER(ci), ctypes.POINTER(ci)], ci),
        "b200pose_net_profile": ([vp, vp, vp, ci, vp], ci),
        "b200pose_net_last_maps": ([vp, ctypes.POINTER(vp), ctypes.POINTER(vp), ctypes.POINTER(ci), ctypes.POINTER(ci),
                                    ctypes.POINTER(ci)], ci),
        "b200pose_post_create": ([ctypes.POINTER(vp), ci, ci, ci, ci], ci),
        "b200pose_post_destroy": ([vp], None),
        "b200pose_post_run": ([vp, vp, vp, ci, ci, ci, ci, ci, cf, vp], ci),
        "b200pose_post_sync": ([vp], ci),
        "b200pose_post_last_ticket": ([vp], cl),
        "b200pose_post_select": ([vp, cl], ci),
        "b200pose_post_debug": ([vp, vp, ci, ci], ci),
        "b200pose_post_status_accum": ([vp, ci], ci),
        "b200pose_post_debug_sort": ([vp, vp, ci, vp], ci),
        "b200pose_post_num_humans": ([vp, ci], ci),
        "b200pose_post_status": ([vp, ci], ci),
        "b200pose_post_get_humans": ([vp, ci, vp, ci], ci),
        "b200pose_post_get_peaks": ([vp, ci, vp, ci], ci),
        "b200pose_infer": ([vp, vp, vp, ci, ci, ci, ci, ci, cf, vp], ci),
        "b200pose_infer_u8": ([vp, vp, vp, ci, ci, ci, ci, ci, cf, vp], ci),
        "b200pose_flip_merge": ([vp, vp, vp, vp, vp, ci, ci, ci, ci, ci, vp, vp, vp], ci),
        "b200pose_infer_flip": ([vp, vp, vp, ci, ci, ci, ci, ci, cf, vp], ci),
        "b200pose_infer_u8_flip": ([vp, vp, vp, ci, ci, ci, ci, ci, cf, vp], ci),
        "b200pose_crop_geometry": ([ci, ci, ci, ci, ctypes.POINTER(ctypes.c_double)] + [ctypes.POINTER(ci)] * 4, ci),
        "b200pose_net_crop_with_factor": ([vp, vp, ci, ci, ci, ci, ci, ci, vp, ci, vp], ci),
        "b200pose_infer_raw_u8": ([vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, cf, ci, vp], ci),
        "b200pose_infer_raw_u8_multiscale": ([vp, vp, vp, ci, ci, ci, ci, ci, ci, ctypes.POINTER(ctypes.c_double), ci, ci, cf,
                                              ci, vp], ci),
        "process_paf": ([ci, ci, ci, vp, ci, ci, ci, vp, ci, ci, ci, vp], ci),
        "get_num_humans": ([], ci),
        "get_part_cid": ([ci, ci], ci),
        "get_score": ([ci], cf),
        "get_part_x": ([ci], ci),
        "get_part_y": ([ci], ci),
        "get_part_score": ([ci], cf),
    }
    for name, (args, res) in sig.items():
        fn = getattr(L, name)     # AttributeError here = the library does not export what include/b200pose.h declares
        fn.argtypes = args
        fn.restype = res
    _lib = L
    return L


EXPORTED = ["b200pose_last_error", "b200pose_version", "b200pose_launch_count", "b200pose_net_create",
            "b200pose_net_destroy", "b200pose_net_tensor_shape", "b200pose_net_set_tensor", "b200pose_net_finalize",
            "b200pose_net_forward", "b200pose_net_forward_u8", "b200pose_net_set_preprocess", "b200pose_net_profile", "b200pose_net_last_maps", "b200pose_post_create", "b200pose_post_destroy",
            "b200pose_post_run", "b200pose_post_sync", "b200pose_post_last_ticket", "b200pose_post_select", "b200pose_post_debug", "b200pose_post_debug_sort", "b200pose_post_status_accum", "b200pose_post_num_humans", "b200pose_post_status",
            "b200pose_post_get_humans", "b200pose_post_get_peaks", "b200pose_infer", "b200pose_infer_u8", "b200pose_flip_merge", "b200pose_infer_flip",
            "b200pose_infer_u8_flip", "b200pose_crop_geometry", "b200pose_net_crop_with_factor",
            "b200pose_infer_raw_u8", "b200pose_infer_raw_u8_multiscale", "b200pose_net_forward_u8_ragged",
            "b200pose_infer_raw_u8_ragged", "b200pose_ragged_layout", "process_paf", "get_num_humans",
            "get_part_cid", "get_score", "get_part_x", "get_part_y", "get_part_score"]


def check(rc, what=""):
    if rc != 0:
        msg = lib().b200pose_last_error()
        raise B200PoseError("%s failed (rc=%d): %s" % (what or "b200pose call", rc, msg.decode() if msg else "?"))


def crop_geometry(src_h, src_w, dest_size=368, factor=8):
    """(im_scale, (res_h, res_w), (pad_h, pad_w)) exactly as crop_with_factor (im_transform.py:119-134) computes them.
    Host arithmetic only, but it lives in the library so that there is one implementation."""
    sc = ctypes.c_double()
    v = [ctypes.c_int() for _ in range(4)]
    check(lib().b200pose_crop_geometry(int(src_h), int(src_w), int(dest_size), int(factor), ctypes.byref(sc),
                                       *[ctypes.byref(x) for x in v]), "b200pose_crop_geometry")
    return sc.value, (v[0].value, v[1].value), (v[2].value, v[3].value)


def ragged_layout(src_sizes, dest_size=368, factor=8):
    """Layout of a ragged batch of raw frames [(src_h, src_w), ...] packed back to back, as b200pose_infer_raw_u8_ragged
    computes it: (byte offset of each frame, [(pad_h, pad_w)] per frame, (canvas_h, canvas_w)).  Host arithmetic only."""
    n = len(src_sizes)
    sh = (ctypes.c_int * max(n, 1))(*[int(h) for h, _ in src_sizes])
    sw = (ctypes.c_int * max(n, 1))(*[int(w) for _, w in src_sizes])
    off = (ctypes.c_long * max(n, 1))()
    ph, pw = (ctypes.c_int * max(n, 1))(), (ctypes.c_int * max(n, 1))()
    ch, cw = ctypes.c_int(), ctypes.c_int()
    check(lib().b200pose_ragged_layout(n, sh, sw, int(dest_size), int(factor), off, ph, pw, ctypes.byref(ch),
                                       ctypes.byref(cw)), "b200pose_ragged_layout")
    return list(off[:n]), list(zip(ph[:n], pw[:n])), (ch.value, cw.value)


def launch_count():
    return int(lib().b200pose_launch_count())
