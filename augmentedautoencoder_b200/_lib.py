"""ctypes binding of libaae_b200.so (the C ABI declared in include/aae_b200.h).  Fails loudly: no fallback."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libaae_b200.so")
HEADER_PATH = os.path.join(_HERE, "..", "include", "aae_b200.h")

AAE_MAX_LAYERS = 8
PREC_FP32_SIMT = 0
PREC_TC_SPLIT = 1
RENDER_VIEW_FLOATS = 64
RENDER_BEHIND_CAMERA, RENDER_EMPTY, RENDER_BAD_CROP = 1, 2, 4


class AaeError(RuntimeError):
    pass


class NetCfg(C.Structure):
    _fields_ = [("in_h", C.c_int32), ("in_w", C.c_int32), ("in_c", C.c_int32), ("num_layers", C.c_int32),
                ("filters", C.c_int32 * AAE_MAX_LAYERS), ("strides", C.c_int32 * AAE_MAX_LAYERS),
                ("kernel_size", C.c_int32), ("latent", C.c_int32), ("max_batch", C.c_int32), ("precision", C.c_int32)]


_P = C.c_void_p
_I = C.c_int
_L = C.c_int64
_F = C.c_float
_SIGS = {
    "aae_version": (_I, []),
    "aae_last_error_string": (C.c_char_p, []),
    "aae_device_supported": (_I, [_I]),
    "aae_launch_count": (_L, []),
    "aae_encoder_create": (_I, [_I, C.POINTER(NetCfg), C.POINTER(_P)]),
    "aae_encoder_destroy": (_I, [_P]),
    "aae_encoder_set_weights": (_I, [_P, _I, _P, _P, _P]),
    "aae_encoder_get_weights": (_I, [_P, _I, _P, _P, _P]),
    "aae_encoder_forward_u8": (_I, [_P, _P, _I, _P, _P]),
    "aae_encoder_forward_f32": (_I, [_P, _P, _I, _P, _P]),
    "aae_encoder_range_status": (_I, [_P, _P]),
    "aae_encoder_range_word": (_I, [_P, C.POINTER(_P)]),
    "aae_encoder_activation": (_I, [_P, _I, C.POINTER(_P), C.POINTER(_L)]),
    "aae_encoder_profile": (_I, [_P, _I, _P, _I]),
    "aae_codebook_profile": (_I, [_P, _I, _P, _I]),
    "aae_codebook_create": (_I, [_I, _P, _L, _I, _I, _L, _I, _I, C.POINTER(_P)]),
    "aae_codebook_destroy": (_I, [_P]),
    "aae_l2_normalize": (_I, [_P, _I, _I, _P, _P]),
    "aae_codebook_match": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "aae_codebook_cosine": (_I, [_P, _P, _I, _P, _P]),
    "aae_topk_merge": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "aae_topk_merge_packed": (_I, [_P, _I, _I, _I, _P, _P, _P]),
    "aae_codebook_rows": (_L, [_P]),
    "aae_launch_floor_probe": (_I, [_I, _I, _P]),
    "aae_decoder_create": (_I, [_I, C.POINTER(NetCfg), C.POINTER(_P)]),
    "aae_decoder_destroy": (_I, [_P]),
    "aae_decoder_set_weights": (_I, [_P, _I, _P, _P, _P]),
    "aae_decoder_get_weights": (_I, [_P, _I, _P, _P, _P]),
    "aae_decoder_forward": (_I, [_P, _P, _I, _P, _P]),
    "aae_decoder_range_status": (_I, [_P, _P]),
    "aae_bootstrap_l2_loss": (_I, [_P, _P, _I, _I, _I, _P, _P, _P]),
    "aae_trainer_create": (_I, [_P, _P, _I, _F, _F, _F, _F, C.POINTER(_P)]),
    "aae_trainer_destroy": (_I, [_P]),
    "aae_train_step": (_I, [_P, _P, _P, _I, _P, _P]),
    "aae_trainer_forward_backward": (_I, [_P, _P, _P, _I, _P, _P]),
    "aae_trainer_get_grads": (_I, [_P, _I, _I, _P, _P, _P]),
    "aae_trainer_global_step": (_L, [_P]),
    "aae_trainer_profile": (_I, [_P, _I, _P, _I]),
    "aae_trainer_get_state": (_I, [_P, _I, _I, _P, _P, _P, _P, _P]),
    "aae_trainer_set_state": (_I, [_P, _I, _I, _P, _P, _P, _P, _P]),
    "aae_trainer_set_global_step": (_I, [_P, _L]),
    "aae_extract_square_patches": (_I, [_P, _I, _I, _P, _I, _F, _I, _P, _P]),
    "aae_augment_batch": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P]),
    "aae_mesh_create": (_I, [_I, _P, _L, _P, _L, C.POINTER(_P)]),
    "aae_mesh_destroy": (_I, [_P]),
    "aae_render_workspace_bytes": (_L, [_P, _I, _I, _I]),
    "aae_render_frames": (_I, [_P, _P, _I, _I, _I, _F, _F, _P, _L, _P, _P, _P, _P, _P]),
    "aae_render_crops": (_I, [_P, _P, _I, _I, _I, _F, _F, _P, C.c_double, _I, _I, _P, _P, _P, _L, _P, _P, _P, _P, _P, _P]),
}

_lib = None


def lib():
    """The loaded library.  Raises AaeError if it has not been built (python __graft_entry__.py / build_ext.py)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise AaeError(f"{LIB_PATH} is missing: build it with `python -m augmentedautoencoder_b200.build_ext` "
                           "(there is no CPU or PyTorch fallback for the hot path)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(status: int, what: str = ""):
    if status != 0:
        msg = lib().aae_last_error_string().decode("utf-8", "replace")
        raise AaeError(f"{what or 'aae call'} failed (status {status}): {msg}")


def make_cfg(h, w, c, filters, strides, kernel_size, latent, max_batch, precision) -> NetCfg:
    if len(filters) != len(strides) or not 1 <= len(filters) <= AAE_MAX_LAYERS:
        raise ValueError("NUM_FILTER / STRIDES must have the same length in [1, %d]" % AAE_MAX_LAYERS)
    cfg = NetCfg()
    cfg.in_h, cfg.in_w, cfg.in_c = int(h), int(w), int(c)
    cfg.num_layers = len(filters)
    for i, (f, s) in enumerate(zip(filters, strides)):
        cfg.filters[i], cfg.strides[i] = int(f), int(s)
    cfg.kernel_size, cfg.latent, cfg.max_batch, cfg.precision = int(kernel_size), int(latent), int(max_batch), int(precision)
    return cfg


def ptr(t):
    """Device (or host) pointer of a torch tensor / numpy array as c_void_p; None -> NULL."""
    if t is None:
        return None
    if hasattr(t, "data_ptr"):
        return C.c_void_p(t.data_ptr())
    return C.c_void_p(t.ctypes.data)
