"""ctypes binding of libtfrpn_cuda.so (include/tfrpn.h).  No fallback: if the shared library is
missing or no CUDA device is present, importing / calling raises."""
import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# TFRPN_LIB_PATH: a debug build of the same library (tools/phase_times.py); the product path is the in-tree .so
LIB_PATH = os.environ.get("TFRPN_LIB_PATH") or os.path.join(_HERE, "_lib", "libtfrpn_cuda.so")


class AnchorCfg(C.Structure):
    _fields_ = [("img_h", C.c_int32), ("img_w", C.c_int32), ("fm_h", C.c_int32), ("fm_w", C.c_int32),
                ("n_scales", C.c_int32), ("n_ratios", C.c_int32),
                ("scales", C.c_double * 8), ("ratios", C.c_double * 8)]


class TargetCfg(C.Structure):
    _fields_ = [("pos_iou_threshold", C.c_float), ("neg_iou_threshold", C.c_float),
                ("total_pos", C.c_int32), ("total_neg", C.c_int32), ("variances", C.c_float * 4),
                ("seed", C.c_uint64), ("offset", C.c_uint64), ("image_offset", C.c_int32),
                ("reserved", C.c_int32)]


class TargetDebug(C.Structure):
    _fields_ = [("argmax_row", C.c_void_p), ("argmax_col", C.c_void_p), ("max_iou", C.c_void_p),
                ("pos_pre", C.c_void_p), ("neg_pre", C.c_void_p), ("pos_count", C.c_void_p),
                ("neg_count", C.c_void_p)]


class NmsCfg(C.Structure):
    _fields_ = [("max_output_size_per_class", C.c_int32), ("max_total_size", C.c_int32),
                ("iou_threshold", C.c_float), ("score_threshold", C.c_float),
                ("pad_per_class", C.c_int32), ("clip_boxes", C.c_int32), ("pre_nms_topn", C.c_int32)]


class ProposalCfg(C.Structure):
    _fields_ = [("variances", C.c_float * 4), ("pre_nms_topn", C.c_int32), ("post_nms_topn", C.c_int32),
                ("nms_iou_threshold", C.c_float), ("clip", C.c_int32)]


class LossOut(C.Structure):
    _fields_ = [("reg_loss", C.c_float), ("cls_loss", C.c_float), ("n_pos", C.c_int32), ("n_cls", C.c_int32)]


class RecallCfg(C.Structure):
    _fields_ = [("n_thresholds", C.c_int32), ("thresholds", C.c_float * 16), ("n_limits", C.c_int32),
                ("limits", C.c_int32 * 8), ("matching", C.c_int32), ("reserved", C.c_int32)]


class MapCfg(C.Structure):
    _fields_ = [("protocol", C.c_int32), ("num_classes", C.c_int32), ("n_thresholds", C.c_int32),
                ("thresholds", C.c_float * 16), ("max_dets", C.c_int32), ("reserved", C.c_int32)]


class MapState(C.Structure):
    _fields_ = [("records", C.c_void_p), ("capacity", C.c_int64), ("cursor", C.c_void_p), ("n_gt", C.c_void_p),
                ("overflow", C.c_void_p)]


class RoiTargetCfg(C.Structure):
    _fields_ = [("num_classes", C.c_int32), ("total_pos", C.c_int32), ("total_neg", C.c_int32),
                ("fg_iou_threshold", C.c_float), ("bg_iou_high", C.c_float), ("bg_iou_low", C.c_float),
                ("variances", C.c_float * 4), ("append_gt", C.c_int32), ("image_offset", C.c_int32),
                ("seed", C.c_uint64), ("offset", C.c_uint64)]


class StepBuffers(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("gt_boxes", "gt_labels", "rpn_reg", "rpn_cls", "deltas", "labels",
                                          "out_boxes", "out_scores", "valid", "keep_idx")]


P = C.c_void_p
I = C.c_int
KERNEL_IDS = 13  # TFRPN_K_COUNT of include/tfrpn.h
# name -> (restype, argtypes); must list every symbol include/tfrpn.h declares
PROTOTYPES = {
    "tfrpn_version": (I, []),
    "tfrpn_last_error": (C.c_char_p, []),
    "tfrpn_create": (I, [C.POINTER(P), I]),
    "tfrpn_destroy": (I, [P]),
    "tfrpn_reserve": (I, [P, I, I, I, I]),
    "tfrpn_workspace_bytes": (C.c_size_t, [I, I, I, I]),
    "tfrpn_launch_count": (C.c_uint64, []),
    "tfrpn_profile_enable": (I, [P, I]),
    "tfrpn_profile_read": (I, [P, I, C.POINTER(C.c_double), C.POINTER(I)]),
    "tfrpn_kernel_name": (C.c_char_p, [I]),
    "tfrpn_base_anchors_host": (I, [C.POINTER(AnchorCfg), P]),
    "tfrpn_anchors": (I, [C.POINTER(AnchorCfg), P, P]),
    "tfrpn_iou_map": (I, [P, I, P, I, I, I, P, P]),
    "tfrpn_selftest_division": (I, [C.c_uint64, C.c_uint64, P, P]),
    "tfrpn_encode_deltas": (I, [P, I, P, I, I, P, P]),
    "tfrpn_decode": (I, [P, I, P, P, I, I, I, P, P]),
    "tfrpn_decode_anchor_cfg": (I, [C.POINTER(AnchorCfg), P, P, I, I, P, P]),
    "tfrpn_scale_boxes": (I, [P, C.c_int64, C.c_float, C.c_float, I, P, P]),
    "tfrpn_rpn_targets": (I, [P, P, P, P, I, I, I, C.POINTER(TargetCfg), P, P, C.POINTER(TargetDebug), P]),
    "tfrpn_rpn_targets_compact": (I, [P, P, P, P, I, I, I, C.POINTER(TargetCfg), P, P, P, P]),
    "tfrpn_expand_targets_host": (I, [P, P, I, I, I, P, I, P]),
    "tfrpn_roi_targets": (I, [P, P, P, P, P, I, I, I, C.POINTER(RoiTargetCfg), P, P, P, P, P, P, P, P]),
    "tfrpn_select_mask": (I, [P, P, P, I, I, I, C.c_uint64, C.c_uint64, I, I, P, P]),
    "tfrpn_rpn_losses": (I, [P, P, P, P, P, I, I, C.c_float, P, P, P, P]),
    "tfrpn_topk": (I, [P, P, I, I, I, P, P, P, I, P, P]),
    "tfrpn_predict_topk": (I, [P, P, P, P, I, I, I, P, I, P, P, P, P]),
    "tfrpn_pad_gt": (I, [P, P, P, P, I, I, I, P, P, P]),
    "tfrpn_nms": (I, [P, P, P, I, I, C.POINTER(NmsCfg), P, P, P, P, P, P]),
    "tfrpn_proposals": (I, [P, P, P, P, I, I, C.POINTER(ProposalCfg), P, P, P, P, P]),
    "tfrpn_proposals_anchor_cfg": (I, [P, P, P, C.POINTER(AnchorCfg), I, C.POINTER(ProposalCfg), P, P, P, P, P]),
    "tfrpn_rpn_targets_sparse": (I, [P, P, P, P, I, I, I, C.POINTER(TargetCfg), P, P, P, P]),
    "tfrpn_expand_labels_host": (I, [P, I, I, I, P, I, P]),
    "tfrpn_rpn_targets_host": (I, [P, P, P, P, I, I, I, C.POINTER(TargetCfg), P, P, P]),
    "tfrpn_proposals_host": (I, [P, P, P, P, I, I, C.POINTER(ProposalCfg), P, P, P, P, P]),
    "tfrpn_rpn_step_host": (I, [P, P, P, P, I, I, I, C.POINTER(TargetCfg), P, P, P, P, C.POINTER(ProposalCfg), P, P, P, P, P]),
    "tfrpn_pipeline_create": (I, [P, I, C.POINTER(P)]),
    "tfrpn_pipeline_submit": (I, [P, P, I, I, P, P, I, C.POINTER(TargetCfg), P, P, P, P, C.POINTER(ProposalCfg),
                                  P, P, P, P, C.POINTER(C.c_int64)]),
    "tfrpn_pipeline_acquire": (I, [P, I, I, I, I, C.POINTER(StepBuffers)]),
    "tfrpn_pipeline_submit_acquired": (I, [P, P, C.POINTER(TargetCfg), C.POINTER(ProposalCfg), C.POINTER(C.c_int64)]),
    "tfrpn_pipeline_wait": (I, [P, C.c_int64]),
    "tfrpn_pipeline_set_option": (I, [P, I, I]),
    "tfrpn_pipeline_last_copy_bytes": (I, [P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "tfrpn_pipeline_trace": (I, [P, C.c_int64, C.POINTER(C.c_float)]),
    "tfrpn_pipeline_drain": (I, [P]),
    "tfrpn_pipeline_destroy": (I, [P]),
    "tfrpn_host_alloc": (I, [C.POINTER(P), C.c_size_t]),
    "tfrpn_host_free": (I, [P]),
    "tfrpn_proposal_recall": (I, [P, P, P, P, P, I, I, I, C.POINTER(RecallCfg), P, P, P]),
    "tfrpn_nms_multiclass": (I, [P, P, I, P, I, I, I, C.POINTER(NmsCfg), P, P, P, P, P, P]),
    "tfrpn_nms_multiclass_workspace_bytes": (C.c_size_t, [I, I, I, C.POINTER(NmsCfg)]),
    "tfrpn_reserve_nms_multiclass": (I, [P, I, I, I, C.POINTER(NmsCfg)]),
    "tfrpn_map_update": (I, [P, P, P, P, P, P, P, P, I, I, I, C.POINTER(MapCfg), C.POINTER(MapState), P]),
    "tfrpn_map_compute": (I, [P, C.POINTER(MapCfg), C.POINTER(MapState), P, P, P]),
    "tfrpn_map_workspace_bytes": (C.c_size_t, [C.c_int64, I]),
}

_lib = None
_lock = threading.Lock()


class TfrpnError(RuntimeError):
    pass


def load():
    """Load libtfrpn_cuda.so (once).  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise ImportError(
                    "libtfrpn_cuda.so not found at %s -- build it with `python -c 'import __graft_entry__ as g; "
                    "g.build()'` or `make -C tf-rpn_b200/csrc`.  tfrpn has no CPU fallback." % LIB_PATH)
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in PROTOTYPES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


_STATUS = {-1: ValueError, -2: ValueError, -3: TfrpnError, -4: TfrpnError, -5: NotImplementedError}


def check(rc):
    if rc != 0:
        msg = load().tfrpn_last_error().decode("utf-8", "replace")
        raise _STATUS.get(rc, TfrpnError)("tfrpn status %d: %s" % (rc, msg))


_handles = threading.local()


def handle(device_index):
    """One handle per (thread, device): the C handle is single-threaded by contract."""
    cache = getattr(_handles, "cache", None)
    if cache is None:
        cache = _handles.cache = {}
    h = cache.get(device_index)
    if h is None:
        out = P()
        check(load().tfrpn_create(C.byref(out), int(device_index)))
        h = cache[device_index] = out
    return h


def launch_count():
    return int(load().tfrpn_launch_count())
