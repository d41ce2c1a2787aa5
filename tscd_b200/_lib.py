"""ctypes binding of libtscd_b200.so (the C-ABI declared in include/tscd_b200.h).

There is deliberately no fallback: if the CUDA library is missing or a call fails, a RuntimeError is
raised.  Nothing here imports ``oracle``.
"""
import ctypes as C
import os

from .build import LIB_PATH

TSCD_F32, TSCD_F16, TSCD_BF16 = 0, 1, 2
MAX_LEVELS = 3
_ERR = {-1: "invalid argument", -2: "unsupported configuration", -3: "capacity exceeded", -4: "CUDA error",
        -5: "frame-store slot out of range or never written"}
TSCD_ERR_CAPACITY, TSCD_ERR_FRAME_SLOT = -3, -5


class View(C.Structure):
    _fields_ = [("ptr", C.c_void_p * MAX_LEVELS), ("frame_stride", C.c_int64 * MAX_LEVELS),
                ("anchor_stride", C.c_int64 * MAX_LEVELS), ("chan_stride", C.c_int64 * MAX_LEVELS)]


class Anchors(C.Structure):
    _fields_ = [("num_levels", C.c_int32), ("level_h", C.c_int32 * MAX_LEVELS), ("level_w", C.c_int32 * MAX_LEVELS),
                ("level_stride", C.c_int32 * MAX_LEVELS), ("level_start", C.c_int32 * (MAX_LEVELS + 1))]


class SelectArgs(C.Structure):
    _fields_ = [("mode", C.c_int32), ("num_frames", C.c_int32), ("num_classes", C.c_int32), ("head_dtype", C.c_int32),
                ("apply_sigmoid", C.c_int32), ("apply_decode", C.c_int32), ("pre_k", C.c_int32),
                ("conf_thresh", C.c_float), ("minimal_limit", C.c_int32), ("maximal_limit", C.c_int32),
                ("cand_cap", C.c_int32), ("anchors", Anchors), ("reg", View), ("obj", View), ("cls", View),
                ("cand_idx", C.c_void_p), ("cand_box", C.c_void_p), ("cand_score", C.c_void_p),
                ("cand_cls", C.c_void_p), ("cand_count", C.c_void_p),
                ("ws_conf", C.c_void_p), ("ws_cls", C.c_void_p), ("ws_pitch", C.c_int32), ("status", C.c_void_p),
                ("cand_rank", C.c_void_p)]


class PackHeadArgs(C.Structure):
    _fields_ = [("num_frames", C.c_int32), ("num_classes", C.c_int32), ("head_dtype", C.c_int32), ("row_pitch", C.c_int32),
                ("obj_pitch", C.c_int64), ("anchors", Anchors), ("reg", View), ("obj", View), ("cls", View),
                ("rows", C.c_void_p), ("obj_plane", C.c_void_p)]


class NmsArgs(C.Structure):
    _fields_ = [("num_frames", C.c_int32), ("cand_cap", C.c_int32), ("max_keep", C.c_int32), ("iou_thresh", C.c_float),
                ("box", C.c_void_p), ("score", C.c_void_p), ("cls", C.c_void_p), ("count", C.c_void_p),
                ("keep", C.c_void_p), ("keep_count", C.c_void_p), ("status", C.c_void_p),
                ("ws", C.c_void_p), ("ws_bytes", C.c_int64), ("strict_keep", C.c_int32), ("rank", C.c_void_p)]


class GatherArgs(C.Structure):
    _fields_ = [("num_frames", C.c_int32), ("num_classes", C.c_int32), ("head_dtype", C.c_int32),
                ("apply_sigmoid", C.c_int32), ("apply_decode", C.c_int32), ("cand_cap", C.c_int32),
                ("max_keep", C.c_int32), ("use_keep", C.c_int32), ("feat_dim", C.c_int32), ("feat_dtype", C.c_int32),
                ("bank_dtype", C.c_int32), ("anchors", Anchors), ("reg", View), ("obj", View), ("cls", View),
                ("feat_cls", View), ("feat_reg", View), ("feat_edge", View),
                ("cand_idx", C.c_void_p), ("cand_count", C.c_void_p), ("keep", C.c_void_p), ("keep_count", C.c_void_p),
                ("sel_count", C.c_void_p), ("row_off", C.c_void_p), ("sel_idx", C.c_void_p), ("sel_rows", C.c_void_p),
                ("bank_cls", C.c_void_p), ("bank_reg", C.c_void_p), ("bank_edge", C.c_void_p),
                ("bank_score", C.c_void_p), ("bank_fg", C.c_void_p), ("bank_box", C.c_void_p)]


class LinearArgs(C.Structure):
    _fields_ = [("M", C.c_int32), ("N", C.c_int32), ("K", C.c_int32), ("dtype", C.c_int32),
                ("x", C.c_void_p), ("ldx", C.c_int64), ("w", C.c_void_p), ("ldw", C.c_int64),
                ("bias", C.c_void_p), ("m_dev", C.c_void_p), ("out16", C.c_void_p), ("ld16", C.c_int32),
                ("out32", C.c_void_p), ("ld32", C.c_int32)]


class AttnLayout(C.Structure):
    _fields_ = [("B", C.c_int32), ("F", C.c_int32), ("L", C.c_int32), ("self_attn", C.c_int32), ("dtype", C.c_int32),
                ("row_cap", C.c_int32), ("nk_pitch", C.c_int32), ("row_off", C.c_void_p), ("lrow_off", C.c_void_p)]


class AttnPrepArgs(C.Structure):
    _fields_ = [("lay", AttnLayout), ("scale", C.c_float), ("qkv_cls", C.c_void_p), ("qkv_reg", C.c_void_p),
                ("ld_qkv", C.c_int32), ("key_score", C.c_void_p),
                ("qn_cls", C.c_void_p), ("kn_cls", C.c_void_p), ("vn_cls", C.c_void_p),
                ("qn_reg", C.c_void_p), ("kn_reg", C.c_void_p), ("vn_reg", C.c_void_p),
                ("vt_cls", C.c_void_p), ("vt_reg", C.c_void_p), ("xori_cls", C.c_void_p), ("xori_reg", C.c_void_p),
                ("ld_xori", C.c_int32), ("row_frame", C.c_void_p)]


class QkvProjectArgs(C.Structure):
    _fields_ = [("lay", AttnLayout), ("rows", C.c_int32), ("m_dev", C.c_void_p), ("x", C.c_void_p), ("ldx", C.c_int64),
                ("w", C.c_void_p), ("row_meta", C.c_void_p), ("key_score", C.c_void_p), ("scale", C.c_float),
                ("qn", C.c_void_p), ("kn", C.c_void_p), ("vn", C.c_void_p), ("vt", C.c_void_p), ("xori", C.c_void_p),
                ("ld_xori", C.c_int32)]


class AttnRowmetaArgs(C.Structure):
    _fields_ = [("lay", AttnLayout), ("row_frame", C.c_void_p), ("row_meta", C.c_void_p), ("vt_cls", C.c_void_p),
                ("vt_reg", C.c_void_p)]


class AttnPvArgs(C.Structure):
    _fields_ = [("lay", AttnLayout), ("qn_cls", C.c_void_p), ("kn_cls", C.c_void_p), ("qn_reg", C.c_void_p),
                ("kn_reg", C.c_void_p), ("vt_cls", C.c_void_p), ("vt_reg", C.c_void_p), ("row_frame", C.c_void_p),
                ("need_reg", C.c_int32), ("x_cls", C.c_void_p), ("x_reg", C.c_void_p), ("ld_x", C.c_int32),
                ("stats", C.c_void_p), ("max_logit", C.c_float)]


class AttnRound2Args(C.Structure):
    _fields_ = [("lay", AttnLayout), ("qn_cls", C.c_void_p), ("kn_cls", C.c_void_p), ("qn_reg", C.c_void_p),
                ("kn_reg", C.c_void_p), ("vn_cls", C.c_void_p), ("vn_reg", C.c_void_p), ("vt", C.c_void_p),
                ("row_frame", C.c_void_p), ("stats", C.c_void_p), ("use_obj_mask", C.c_int32),
                ("sim_thresh", C.c_float), ("conf_sim_thresh", C.c_float), ("out", C.c_void_p), ("ld_out", C.c_int32),
                ("w_out", C.c_void_p), ("w_in", C.c_void_p)]


class TransposeArgs(C.Structure):
    _fields_ = [("lay", AttnLayout), ("width", C.c_int32), ("x", C.c_void_p), ("ld_x", C.c_int32), ("xt", C.c_void_p)]


def _fields(spec):
    """'name:type' list -> ctypes fields; types: i=int32, f=float, p=pointer."""
    m = {"i": C.c_int32, "f": C.c_float, "p": C.c_void_p}
    return [(x.split(":")[0], m[x.split(":")[1]]) for x in spec.split()]


class CafmPrepArgs(C.Structure):
    _fields_ = _fields("B:i F:i L:i D:i bank_dtype:i row_off:p lrow_off:p bank_reg:p bank_edge:p time_emb:p se_w1:p "
                       "se_w2:p emb_reg:p emb_cls:p feat:p edge:p feat16:p kin16:p kin:p norm_reg:p norm_cls:p emb_dtype:i")


class CafmChainArgs(C.Structure):
    _fields_ = _fields("B:i F:i L:i D:i kmax:i out_dtype:i row_off:p lrow_off:p resume:p feat:p edge:p kin:p kproj:p "
                       "vproj:p kproj16:p vproj16:p wq16:p bank_reg:p bank_edge:p time_emb:p emb_reg:p emb_cls:p norm_reg:p norm_cls:p wq_t:p se_w1:p se_w2:p ln_w:p "
                       "ln_b:p dec_w:p dec_b:p st_n:p st_out:p st_edge:p st_reg:p st_cls:p st_nreg:p st_ncls:p "
                       "st_time:p sc_qin:p sc_q:p sc_k:p ref_n:p lap_col:p lap_row:p out16:p out32:p perm:p status:p emb_dtype:i slot:p")


class CafmWideArgs(C.Structure):
    _fields_ = [("base", CafmChainArgs)] + _fields("qin16:p attn:p q_beg:p q_end:p kv_beg:p kv_end:p ctl:p perm_s:p prow_s:p ord_prev:p "
                                                   "n_prev:p last_l0:p")


class FrameFlashArgs(C.Structure):
    _fields_ = _fields("num_items:i heads:i head_dim:i dtype:i max_q:i q_beg:p q_end:p kv_beg:p kv_end:p q:p ldq:i k:p ldk:i v:p ldv:i "
                       "out:p ldo:i")


class EdgePatchesArgs(C.Structure):
    _fields_ = [("num_frames", C.c_int32), ("max_keep", C.c_int32), ("feat_dtype", C.c_int32), ("op_dtype", C.c_int32),
                ("anchors", Anchors), ("feat_reg", View), ("sel_idx", C.c_void_p), ("sel_count", C.c_void_p), ("row_off", C.c_void_p),
                ("seg_base", C.c_int32 * MAX_LEVELS), ("seg_cap", C.c_int32 * MAX_LEVELS), ("level_count", C.c_void_p),
                ("slot", C.c_void_p), ("patches", C.c_void_p), ("hf", C.c_void_p), ("status", C.c_void_p)]


class EdgeCombineArgs(C.Structure):
    _fields_ = _fields("rows_cap:i op_dtype:i total_rows:p slot:p content:p hf_out:p bank_edge:p")


class CafmCostArgs(C.Structure):
    _fields_ = _fields("B:i L:i D:i kmax:i lrow_off:p resume:p st_n:p emb_reg:p emb_cls:p norm_reg:p norm_cls:p "
                       "st_reg:p st_cls:p st_nreg:p st_ncls:p cost:p ref_n:p emb_dtype:i emb_reg16:p emb_cls16:p emb16_dtype:i slot:p")


class CafmLapArgs(C.Structure):
    _fields_ = _fields("num_frames:i kmax:i lrow_off:p ref_n:p cost:p lap_col:p lap_row:p")


class LocalOffsetsArgs(C.Structure):
    _fields_ = _fields("B:i F:i L:i sel_count:p lrow_off:p")


class FrameAttentionArgs(C.Structure):
    _fields_ = _fields("num_frames:i heads:i head_dim:i in_dtype:i lrow_off:p q:p ldq:i k:p ldk:i v:p ldv:i out:p ldo:i")


class ResidualLn2Args(C.Structure):
    _fields_ = _fields("rows_cap:i dim:i n_rows:p x:p r:p w_a:p b_a:p w_b:p b_b:p out_dtype:i out16:p out32:p head_w:p head_b:p head_out:p")


class FinalExpandArgs(C.Structure):
    _fields_ = _fields("B:i F:i L:i num_classes:i max_keep:i conf_thre:f xform_clip:f sel_count:p sel_rows:p lrow_off:p "
                       "cls_logits:p ld_cls:i obj_logits:p ld_obj:i reg_deltas:p ld_reg:i "
                       "r_box:p r_score:p r_cls:p r_obj:p r_cscore:p r_count:p "
                       "o_box:p o_score:p o_cls:p o_obj:p o_cscore:p o_count:p")


class FinalRowsArgs(C.Structure):
    _fields_ = _fields("num_frames:i cand_cap:i keep_cap:i box:p obj:p cscore:p cls:p keep:p keep_count:p rows:p")


class BankPackArgs(C.Structure):
    _fields_ = _fields("n_local_frames:i n_global_frames:i kmax:i dtype:i sel_count:p row_off:p bank_cls:p bank_reg:p bank_score:p send:p")


class BankUnpackArgs(C.Structure):
    _fields_ = [("world", C.c_int32), ("n_local_frames", C.c_int32), ("n_global_frames", C.c_int32), ("kmax", C.c_int32),
                ("dtype", C.c_int32), ("rank_bytes", C.c_int64), ("recv", C.c_void_p), ("sel_count", C.c_void_p),
                ("row_off", C.c_void_p), ("bank_cls", C.c_void_p), ("bank_reg", C.c_void_p), ("bank_edge", C.c_void_p),
                ("bank_score", C.c_void_p), ("v_count", C.c_void_p), ("v_row_off", C.c_void_p), ("v_bank_cls", C.c_void_p),
                ("v_bank_reg", C.c_void_p), ("v_bank_edge", C.c_void_p), ("v_bank_score", C.c_void_p)]


class FrameStoreC(C.Structure):
    _fields_ = _fields("frames:i kmax:i num_classes:i dtype:i count:p status:p bank_cls:p bank_reg:p bank_edge:p bank_score:p "
                       "sel_idx:p sel_rows:p")


class FrameScatterArgs(C.Structure):
    _fields_ = [("store", FrameStoreC)] + _fields("num_frames:i frame_slots:p sel_count:p row_off:p sel_idx:p sel_rows:p bank_cls:p "
                                                  "bank_reg:p bank_edge:p bank_score:p status:p slot_error:p")


class ClipAssembleArgs(C.Structure):
    _fields_ = [("store", FrameStoreC), ("B", C.c_int32), ("F", C.c_int32), ("L", C.c_int32), ("row_cap", C.c_int64)] + \
        _fields("clip_slots:p sel_count:p row_off:p bank_cls:p bank_reg:p bank_edge:p bank_score:p sel_idx:p sel_rows:p status:p")


class PackDetectionsArgs(C.Structure):
    _fields_ = _fields("num_frames:i cap:i rows:p count:p scale:p offsets:p packed:p")


class PackRowsArgs(C.Structure):
    _fields_ = _fields("num_frames:i cap:i rows:p count:p offsets:p packed:p")


class ReppLinkArgs(C.Structure):
    _fields_ = [("num_frames", C.c_int32), ("max_det", C.c_int32), ("distance_func", C.c_int32), ("clf_mode", C.c_int32),
                ("clf_thr", C.c_double), ("coef", C.c_double * 4), ("intercept", C.c_double),
                ("frame_off", C.c_void_p), ("bbox", C.c_void_p), ("center", C.c_void_p), ("score", C.c_void_p), ("cls", C.c_void_p),
                ("pairs", C.c_void_p), ("pair_count", C.c_void_p), ("ws_dist", C.c_void_p), ("ws_idx", C.c_void_p),
                ("ws_pitch", C.c_int32), ("status", C.c_void_p)]


_lib = None

# every symbol include/tscd_b200.h declares: (name, restype, argtypes)
SYMBOLS = [
    ("tscd_version", C.c_char_p, []),
    ("tscd_device_ok", C.c_int, []),
    ("tscd_last_cuda_error", C.c_char_p, []),
    ("tscd_select", C.c_int, [C.POINTER(SelectArgs), C.c_void_p]),
    ("tscd_pack_head", C.c_int, [C.POINTER(PackHeadArgs), C.c_void_p]),
    ("tscd_debug_select_keys", C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    ("tscd_nms", C.c_int, [C.POINTER(NmsArgs), C.c_void_p]),
    ("tscd_nms_workspace_bytes", C.c_int64, [C.c_int32, C.c_int32]),
    ("tscd_gather", C.c_int, [C.POINTER(GatherArgs), C.c_void_p]),
    ("tscd_local_offsets", C.c_int, [C.POINTER(LocalOffsetsArgs), C.c_void_p]),
    ("tscd_linear", C.c_int, [C.POINTER(LinearArgs), C.c_void_p]),
    ("tscd_attn_prep", C.c_int, [C.POINTER(AttnPrepArgs), C.c_void_p]),
    ("tscd_qkv_project", C.c_int, [C.POINTER(QkvProjectArgs), C.c_void_p]),
    ("tscd_attn_rowmeta", C.c_int, [C.POINTER(AttnRowmetaArgs), C.c_void_p]),
    ("tscd_attn_pv", C.c_int, [C.POINTER(AttnPvArgs), C.c_void_p]),
    ("tscd_attn_round2", C.c_int, [C.POINTER(AttnRound2Args), C.c_void_p]),
    ("tscd_transpose_clip", C.c_int, [C.POINTER(TransposeArgs), C.c_void_p]),
    ("tscd_cafm_prep", C.c_int, [C.POINTER(CafmPrepArgs), C.c_void_p]),
    ("tscd_cafm_cost", C.c_int, [C.POINTER(CafmCostArgs), C.c_void_p]),
    ("tscd_cafm_lap", C.c_int, [C.POINTER(CafmLapArgs), C.c_void_p]),
    ("tscd_debug_chain_clocks", C.c_int, [C.POINTER(C.c_longlong), C.c_int]),
    ("tscd_cafm_chain", C.c_int, [C.POINTER(CafmChainArgs), C.c_void_p]),
    ("tscd_cafm_wide", C.c_int, [C.POINTER(CafmWideArgs), C.c_int, C.c_int, C.c_void_p]),
    ("tscd_frame_flash", C.c_int, [C.POINTER(FrameFlashArgs), C.c_void_p]),
    ("tscd_edge_patches", C.c_int, [C.POINTER(EdgePatchesArgs), C.c_void_p]),
    ("tscd_edge_combine", C.c_int, [C.POINTER(EdgeCombineArgs), C.c_void_p]),
    ("tscd_frame_attention", C.c_int, [C.POINTER(FrameAttentionArgs), C.c_void_p]),
    ("tscd_residual_ln2", C.c_int, [C.POINTER(ResidualLn2Args), C.c_void_p]),
    ("tscd_final_expand", C.c_int, [C.POINTER(FinalExpandArgs), C.c_void_p]),
    ("tscd_final_rows", C.c_int, [C.POINTER(FinalRowsArgs), C.c_void_p]),
    ("tscd_pack_detections", C.c_int, [C.POINTER(PackDetectionsArgs), C.c_void_p]),
    ("tscd_pack_rows", C.c_int, [C.POINTER(PackRowsArgs), C.c_void_p]),
    ("tscd_repp_link", C.c_int, [C.POINTER(ReppLinkArgs), C.c_void_p]),
    ("tscd_bank_pack_bytes", C.c_int64, [C.c_int32, C.c_int32]),
    ("tscd_bank_pack", C.c_int, [C.POINTER(BankPackArgs), C.c_void_p]),
    ("tscd_bank_unpack", C.c_int, [C.POINTER(BankUnpackArgs), C.c_void_p]),
    ("tscd_frame_scatter", C.c_int, [C.POINTER(FrameScatterArgs), C.c_void_p]),
    ("tscd_clip_assemble", C.c_int, [C.POINTER(ClipAssembleArgs), C.c_void_p]),
]


def lib():
    """Load the shared library (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: run `python -m tscd_b200.build` (or __graft_entry__.build()). "
                "tscd_b200 has no CPU or PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, res, args in SYMBOLS:
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


# kernels launched per C-ABI call (for the bench's `gpu_launches` claim)
_DEBUG_SYNC = os.environ.get("TSCD_DEBUG_SYNC", "0") == "1"
KERNELS_PER_CALL = {"tscd_gather": 2, "tscd_nms_large": 3, "tscd_bank_unpack": 2, "tscd_clip_assemble": 2, "tscd_pack_detections": 2, "tscd_pack_rows": 2, "tscd_cafm_wide_p1": 2}
launch_count = 0
# optional per-entry-point CUDA-event timing: {"names": set or None (= all), "events": {name: [(start, end), ...]}}
profile = None


def check(rc, what):
    global launch_count
    if rc != 0:
        detail = lib().tscd_last_cuda_error().decode() if rc == -4 else ""
        raise RuntimeError(f"{what} failed: {_ERR.get(rc, rc)} (code {rc}) {detail}")
    launch_count += KERNELS_PER_CALL.get(what, 1)
    if _DEBUG_SYNC:                      # TSCD_DEBUG_SYNC=1: localise asynchronous kernel faults
        import torch
        try:
            torch.cuda.synchronize()
        except Exception as e:           # noqa: BLE001
            raise RuntimeError(f"{what}: asynchronous CUDA failure: {e}") from e


class timed:
    """Context manager: brackets one C-ABI call with CUDA events on the current stream when profiling is on."""

    def __init__(self, name, tag=None):
        self.on = profile is not None and (profile["names"] is None or name in profile["names"])
        self.name = name if tag is None else f"{name}:{tag}"

    def __enter__(self):
        if self.on:
            import torch
            self.s = torch.cuda.Event(enable_timing=True)
            self.e = torch.cuda.Event(enable_timing=True)
            self.s.record()
        return self

    def __exit__(self, *exc):
        if self.on:
            self.e.record()
            profile["events"].setdefault(self.name, []).append((self.s, self.e))
        return False
