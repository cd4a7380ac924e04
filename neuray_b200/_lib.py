"""ctypes binding of libneuray_b200.so (C-ABI declared in include/neuray_b200.h).

The library is the product: if it is missing the import of this module still succeeds (so that CPU-only host
logic can be imported), but the first call that needs it raises -- there is no PyTorch or CPU fallback.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# NEURAY_B200_LIB: development switch to load another in-tree build of the same library (A/B runs of kernel variants)
LIB_PATH = os.environ.get("NEURAY_B200_LIB") or os.path.join(_HERE, "libneuray_b200.so")

ABI_VERSION = 6
NR_POINT_REC = 20
NR_MAX_VIEWS = 32
NR_MAX_SAMPLES = 256


class NrWeightLayout(C.Structure):
    _names = ("total_point total_ray dd_head dd_head_stride dd_l0_w dd_l0_b dd_l1_w dd_l1_b dd_l2_w dd_l2_b "
              "grp_b pe0_w pe0_b pe1_w pe1_b rd0_w rd0_b rd1_w rd1_b nf0_w nf0_b nf1_w nf1_b grp_b_size "
              "hoist_w hoist_b base0_w base1_w base1_b "
              "grp_d1 vis0_w vis0_b vis1_w vis1_b vis1l_w vis1l_b v20_w v20_b v21_w v21_b rgb0_w rgb0_b rgb1_w rgb1_b "
              "rgb2_w rgb2_b grp_d1_size grp_d2 geo0_w geo0_b geo1_w geo1_b grp_d2_size "
              "wq wk wv wfc ln_w ln_b og0_w og0_b og1_w og1_b").split()
    _fields_ = [(n, C.c_int32) for n in _names]


class NrPassParams(C.Structure):
    _fields_ = [
        ("coords", C.c_void_p), ("que_depth", C.c_void_p), ("que_cam", C.c_void_p),
        ("rn", C.c_int32), ("dn", C.c_int32),
        ("feat", C.c_void_p), ("rgb", C.c_void_p), ("view_params", C.c_void_p),
        ("rfn", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("fh", C.c_int32), ("fw", C.c_int32),
        ("w_point", C.c_void_p), ("w_ray", C.c_void_p), ("pos_enc", C.c_void_p),
        ("use_vis", C.c_int32), ("var_bias", C.c_float),
        ("ray_mask_view_num", C.c_int32), ("ray_mask_point_num", C.c_int32),
        ("point_rec", C.c_void_p),
        ("pixel_colors", C.c_void_p), ("hit_prob", C.c_void_p), ("render_depth", C.c_void_p), ("ray_mask", C.c_void_p),
        ("fine_dn", C.c_int32), ("fine_use_all", C.c_int32), ("fine_u", C.c_void_p), ("fine_u_stride", C.c_int32),
        ("fine_depth", C.c_void_p),
        ("w_tc", C.c_void_p),
    ]


class NrLinear(C.Structure):
    _fields_ = [("w", C.c_void_p), ("b", C.c_void_p)]


class NrPassWeights(C.Structure):
    _fields_ = [("dist_decoder", NrLinear * 3 * 4), ("prob_embed", NrLinear * 2), ("ray_dir_fc", NrLinear * 2),
                ("neuray_fc", NrLinear * 2), ("base_fc", NrLinear * 2), ("vis_fc", NrLinear * 2), ("vis_fc2", NrLinear * 2),
                ("rgb_fc", NrLinear * 3), ("geometry_fc", NrLinear * 2), ("out_geometry_fc", NrLinear * 2),
                ("w_qs", C.c_void_p), ("w_ks", C.c_void_p), ("w_vs", C.c_void_p), ("attn_fc", C.c_void_p),
                ("layer_norm_w", C.c_void_p), ("layer_norm_b", C.c_void_p)]


class NrTcLayout(C.Structure):
    _fields_ = [(n, C.c_int32) for n in "total stage head0 pe0 pe1 b0 b1 v01 v2r rd1 hst g0".split()]


# name -> (restype, argtypes); mirrors include/neuray_b200.h one to one (tests/test_abi.py checks the header against this)
_vp, _i, _f = C.c_void_p, C.c_int, C.c_float
SIGNATURES = {
    "nr_abi_version": (C.c_int, []),
    "nr_last_error": (C.c_char_p, []),
    "nr_weight_layout": (C.c_int, [C.POINTER(NrWeightLayout)]),
    "nr_tc_layout": (C.c_int, [C.POINTER(NrTcLayout)]),
    "nr_pack_weights": (C.c_int, [C.POINTER(NrPassWeights), _vp, _vp, _vp, _vp]),
    "nr_camera_blocks": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp]),
    "nr_pack_feature_maps": (C.c_int, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "nr_render_pass_fwd": (C.c_int, [C.POINTER(NrPassParams), _vp]),
    "nr_point_kernel": (C.c_int, [C.POINTER(NrPassParams), _vp]),
    "nr_ray_kernel": (C.c_int, [C.POINTER(NrPassParams), _vp]),
    "nr_point_kernel_debug": (C.c_int, [C.POINTER(NrPassParams), _vp, _vp]),
    "nr_point_kernel_timing": (C.c_int, [C.POINTER(NrPassParams), _vp, _vp]),
    "nr_sample_depth": (C.c_int, [_vp, _i, _i, _vp, _vp, _vp, _vp]),
    "nr_coords2rays": (C.c_int, [_vp, _vp, _i, _vp, _vp, _vp]),
    "nr_depth2points": (C.c_int, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "nr_depth2dists": (C.c_int, [_vp, _i, _i, _vp, _vp]),
    "nr_depth2inv_dists": (C.c_int, [_vp, _vp, _i, _i, _vp, _vp]),
    "nr_alpha_values2hit_prob": (C.c_int, [_vp, _i, _i, _vp, _vp]),
    "nr_project_points": (C.c_int, [_vp, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "nr_interpolate_feats": (C.c_int, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _f, _i, _i, _vp, _vp]),
    "nr_interpolate_feats_bwd": (C.c_int, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _f, _i, _i, _vp, _vp]),
    "nr_sample_fine_depth": (C.c_int, [_vp, _vp, _vp, _i, _i, _i, _vp, _i, _i, _i, _vp, _vp]),
    "nr_diff_feats": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "nr_tc_selftest": (C.c_int, [_vp, _vp, _vp, _i, _i, _i, _vp]),
    "nr_render_pass_bwd": (C.c_int, [_vp, _vp, _vp]),
    "nr_bwd_slot": (C.c_int, [C.c_char_p]),
    "nr_tape_gemms": (C.c_int, [_vp, _i, _vp, _vp, C.c_longlong, _vp, _vp, C.c_longlong, _vp, _vp]),
    "nr_self_hit_prob": (C.c_int, [_vp, _vp]),
    "nr_encoder_layout": (C.c_int, [_vp]),
    "nr_image_encoder_pack": (C.c_int, [_vp, _i, _vp, _vp]),
    "nr_vis_encoder_pack": (C.c_int, [_vp, _i, _vp, _vp]),
    "nr_image_encoder_dims": (C.c_int, [_i, _i, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "nr_image_encoder_workspace": (C.c_longlong, [_i, _i, _i]),
    "nr_vis_encoder_workspace": (C.c_longlong, [_i, _i, _i]),
    "nr_image_encoder_fwd": (C.c_int, [_vp, _vp, _i, _i, _i, _vp, _i, _i, _i, _vp, C.c_longlong, _vp]),
    "nr_vis_encoder_fwd": (C.c_int, [_vp, _vp, _i, _i, _i, _i, _vp, C.c_longlong, _vp]),
    "nr_conv2d_nhwc": (C.c_int, [_vp, _vp]),
    "nr_conv_pack_weight": (C.c_int, [_vp, _i, _i, _i, _i, _vp, _vp]),
    "nr_instance_norm_act": (C.c_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    "nr_nchw_to_nhwc": (C.c_int, [_vp, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    "nr_nhwc_to_nchw": (C.c_int, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "nr_extract_depth": (C.c_int, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    "nr_depth_init_dims": (C.c_int, [_i, _i, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "nr_depth_init_workspace": (C.c_longlong, [_i, _i, _i]),
    "nr_depth_init_pack": (C.c_int, [_vp, _i, _vp, _vp]),
    "nr_depth_init_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp, _i, _i, _i, _vp, C.c_longlong, _vp]),
    "nr_mvsnet_layout": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_longlong)]),
    "nr_mvsnet_pack": (C.c_int, [_vp, _i, _vp, _vp]),
    "nr_mvsnet_dims": (C.c_int, [_i, _i, _i, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "nr_mvsnet_workspace": (C.c_longlong, [_vp]),
    "nr_mvsnet_fwd": (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_longlong, _vp]),
    "nr_cost_volume_head_layout": (C.c_int, [_i, C.POINTER(C.c_int), C.POINTER(C.c_longlong)]),
    "nr_cost_volume_head_pack": (C.c_int, [_i, _vp, _i, _vp, _vp]),
    "nr_cost_volume_head_workspace": (C.c_longlong, [_i, _i, _i, _i]),
    "nr_cost_volume_head_fwd": (C.c_int, [_i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _i, _i, _i, _vp, C.c_longlong, _vp]),
    "nr_depth_mean": (C.c_int, [_vp, _vp]),
    "nr_render_loss": (C.c_int, [_vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "nr_depth_loss": (C.c_int, [_vp, _vp]),
    "nr_consistency_loss": (C.c_int, [_vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp]),
}


class NrMvsIn(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in "ref_imgs src_imgs ref_Ks ref_poses src_Ks src_poses depth_range nn_ids".split()] + \
               [(n, C.c_int32) for n in "rfn sn nn h w dn is_train".split()]


class NrDepthMeanParams(C.Structure):
    _fields_ = [("map", C.c_void_p), ("coords", C.c_void_p), ("w_point", C.c_void_p * 2)] + \
               [(n, C.c_int32) for n in "rfn pn h w fh fw".split()] + \
               [("mean", C.c_void_p * 2), ("d_mean", C.c_void_p * 2), ("d_w_point", C.c_void_p * 2), ("d_map", C.c_void_p)]


class NrDepthLossParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in "depth_pr coords true_depth aug_depth depth_range".split()] + \
               [(n, C.c_int32) for n in "rfn pn h w loss_type".split()] + [("beta", C.c_float), ("correct_thresh", C.c_float)] + \
               [("loss", C.c_void_p), ("g", C.c_void_p), ("d_depth_pr", C.c_void_p)]


class NrEncoderLayout(C.Structure):
    _fields_ = [("image_tensors", C.c_int32), ("vis_tensors", C.c_int32), ("image_packed_floats", C.c_int64), ("vis_packed_floats", C.c_int64),
                ("depth_init_tensors", C.c_int32), ("reserved", C.c_int32), ("depth_init_packed_floats", C.c_int64)]


class NrConv2d(C.Structure):
    _fields_ = [("x", C.c_void_p), ("w_packed", C.c_void_p), ("bias", C.c_void_p), ("res", C.c_void_p), ("y", C.c_void_p), ("stats", C.c_void_p)] + \
               [(n, C.c_int32) for n in "n h w cin cout ks stride reflect x_stride x_off y_stride y_off res_stride res_off tf32x1 pad bm".split()]


class NrSelfParams(C.Structure):
    _fields_ = [("map", C.c_void_p), ("coords", C.c_void_p), ("que_depth", C.c_void_p), ("w_point", C.c_void_p),
                ("rn", C.c_int32), ("dn", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("fh", C.c_int32), ("fw", C.c_int32),
                ("use_vis", C.c_int32), ("depth_range", C.c_void_p), ("var_bias", C.c_float),
                ("hit", C.c_void_p), ("d_hit", C.c_void_p), ("d_w_point", C.c_void_p), ("d_map", C.c_void_p)]


class NrGemmDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in "g_tape g_slot n_out x_tape x_slot n_in out_off reserved".split()]


class NrBwdParams(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in "d_pixel_colors d_hit_prob d_render_depth tape_row grad_row tape_point grad_point d_feat".split()]


_slot_cache = {}


def bwd_slot(name):
    """Slot number on the backward tapes (csrc/nr_train_math.cuh)."""
    if name not in _slot_cache:
        v = lib().nr_bwd_slot(name.encode())
        if v < 0:
            raise NeurayB200Error(f"unknown tape slot {name}")
        _slot_cache[name] = v
    return _slot_cache[name]

_lib = None
_layout = None

# bookkeeping for bench.py: number of CUDA kernels this package launched, and (when PROFILE is a list) CUDA-event
# pairs around every point-kernel launch, recorded on the launching stream
LAUNCHES = 0
PROFILE = None


class NeurayB200Error(RuntimeError):
    pass


def lib():
    """The loaded library; raises if it has not been built (python -m neuray_b200.build)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NeurayB200Error(
                f"{LIB_PATH} not found: build the CUDA extension with `python -m neuray_b200.build` "
                "(there is no CPU / PyTorch fallback for the rendering path)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        if handle.nr_abi_version() != ABI_VERSION:
            raise NeurayB200Error("libneuray_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().nr_last_error()
        raise NeurayB200Error(f"{what} failed (code {rc}): {msg.decode() if msg else ''}")


def weight_layout():
    global _layout
    if _layout is None:
        lay = NrWeightLayout()
        check(lib().nr_weight_layout(C.byref(lay)), "nr_weight_layout")
        _layout = lay
    return _layout


def tc_layout():
    lay = NrTcLayout()
    check(lib().nr_tc_layout(C.byref(lay)), "nr_tc_layout")
    return lay


def ptr(t):
    """Device pointer of a contiguous fp32/uint8 CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise NeurayB200Error("neuray_b200 ops need CUDA tensors (no CPU fallback)")
    if not t.is_contiguous():
        raise NeurayB200Error("neuray_b200 ops need contiguous tensors")
    return t.data_ptr()


def stream_of(t):
    import torch
    return torch.cuda.current_stream(t.device).cuda_stream


def on_device(t):
    """Context that makes t's device the current CUDA device: the library launches on the current device of the calling
    thread, so every entry point of the package wraps its launches in this."""
    import torch
    if not t.is_cuda:
        raise NeurayB200Error("neuray_b200 ops need CUDA tensors (no CPU fallback)")
    return torch.cuda.device(t.device)


def call(name, *args, on, kernels=1, stream=None, what=None):
    """Enqueues the library entry point `name`(*args, stream) on the device of tensor `on`.  The stream is the current
    stream of that device unless `stream` is given (a backward that must follow the stream its forward ran on).  Raises
    NeurayB200Error on a nonzero return and adds `kernels`, the number of kernels the entry point launches, to LAUNCHES."""
    global LAUNCHES
    with on_device(on):
        check(getattr(lib(), name)(*args, stream_of(on) if stream is None else stream), what or name)
    LAUNCHES += kernels


def f32(t):
    """t as a contiguous fp32 tensor outside autograd (t itself, detached, when it already is one)."""
    return t.detach().contiguous().float()


# Grow-only device workspaces, reused across passes, chunks and frames.  The C-ABI never allocates (the caller owns the
# workspace); taking hundreds of MB of point records and tapes per pass from torch's caching allocator every time fragmented
# it and cost cudaMalloc calls in steady state.  Work is stream-ordered on the caller's stream; using one buffer from
# several streams at once is not supported.  Each key is its own buffer: buffers whose keys differ can be live together.
_WORKSPACES = {}


def workspace(key, numel, dev, dtype):
    """The first `numel` elements of the (key, dev) workspace, grown (never shrunk) to fit."""
    import torch
    k = (key, str(dev))
    buf = _WORKSPACES.get(k)
    if buf is None or buf.numel() < numel:
        buf = None                     # the old buffer is freed before the larger one is allocated
        _WORKSPACES.pop(k, None)
        buf = _WORKSPACES[k] = torch.empty(numel, dtype=dtype, device=dev)
    return buf[:numel]
