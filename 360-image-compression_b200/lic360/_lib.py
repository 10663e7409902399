"""ctypes binding of liblic360_b200.so (include/lic360_b200.h). Import fails loudly when the library is absent."""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LIC360_LIB") or os.path.join(os.path.dirname(_HERE), "lib", "liblic360_b200.so")  # override: A/B builds

if not os.path.exists(LIB_PATH):
    raise ImportError(
        "lic360: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(there is no CPU or PyTorch fallback for this path)" % LIB_PATH)

LIB = ctypes.CDLL(LIB_PATH)

_P, _I, _F, _Z, _L = ctypes.c_void_p, ctypes.c_int, ctypes.c_float, ctypes.c_size_t, ctypes.c_long

# name -> (restype, argtypes); must list every symbol include/lic360_b200.h declares (tests/test_abi.py checks it)
SIGNATURES = {
    "lic360_last_error": (ctypes.c_char_p, []),
    "lic360_version": (_I, []),
    "lic360_launch_count": (ctypes.c_longlong, []),
    "lic360_code_contex": (_I, [_I, _I, _P, _P]),
    "lic360_slab": (_I, [_P, _I, _I, _I, _I, _P, _P]),
    "lic360_cconv_wp_floats": (_Z, [_I, _I, _I, _I]),
    "lic360_cconv_wq_floats": (_Z, [_I, _I, _I, _I]),
    "lic360_cconv_pack": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "lic360_cconv_ec_forward": (_I, [_P] * 7 + [_I] * 8 + [_P]),
    "lic360_cconv_dc_forward": (_I, [_P] * 7 + [_I] * 8 + [_P, _P, _I, _P]),
    "lic360_tile_extract": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _P, _P, _I, _P, _P]),
    "lic360_tile_extract_batch": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _I, _P, _P]),
    "lic360_tile_input": (_I, [_P, _P, _I, _I, _I, _I, _F, _F, _I, _P, _P, _I, _P]),
    "lic360_tile_add": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _I, _P]),
    "lic360_gmm_table": (_I, [_P, _P, _P, _P, _I, _I, _I, _F, _I, _F, _P]),
    "lic360_entropy_table": (_I, [_P, _P, _I, _I, _I, _P]),
    "lic360_entropy_gmm_forward": (_I, [_P] * 9 + [_I, _I, _P]),
    "lic360_entropy_gmm_backward": (_I, [_P] * 5 + [_I, _I, _P]),
    "lic360_context_reshape": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "lic360_contex_shift": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "lic360_mask_constrain": (_I, [_P, _I, _I, _I, _I, _I, _P]),
    "lic360_quant_forward": (_I, [_P] * 7 + [_I] * 5 + [_P]),
    "lic360_quant_update_weight": (_I, [_P, _P, _I, _I, _F, _P]),
    "lic360_quant_backward": (_I, [_P] * 8 + [_I] * 5 + [_F, _P]),
    "lic360_dquant_forward": (_I, [_P] * 5 + [_I] * 5 + [_P]),
    "lic360_imp_map_forward": (_I, [_P] * 4 + [_I] * 5 + [_P]),
    "lic360_imp_map_init": (_I, [_P, _P, _I, _I, _F, _F, _F, _F, _P]),
    "lic360_imp_map_backward": (_I, [_P] * 6 + [_I] * 5 + [_F, _I, _P]),
    "lic360_imp2mask": (_I, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "lic360_scale": (_I, [_P, _P, _Z, _F, _F, _P]),
    "lic360_sphere_pad": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "lic360_sphere_pad_inplace": (_I, [_P, _I, _I, _I, _I, _P]),
    "lic360_sphere_pad_backward": (_I, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "lic360_sphere_trim": (_I, [_P, _I, _I, _I, _I, _P]),
    "lic360_sphere_cut_edge": (_I, [_P, _P, _I, _I, _I, _I, _I, _P]),
    "lic360_sphere_lat_scale": (_I, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "lic360_dtow": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "lic360_projects_init": (_I, [_P, _I, _I, _P, _P, _F, _P]),
    "lic360_projects_update": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "lic360_projects_forward": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "lic360_projects_backward": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P]),
    "lic360_coder_create": (_P, [ctypes.c_char_p, _F]),
    "lic360_coder_destroy": (None, [_P]),
    "lic360_coder_reset_fname": (_I, [_P, ctypes.c_char_p]),
    "lic360_coder_start_encoder": (_I, [_P]),
    "lic360_coder_end_encoder": (_I, [_P]),
    "lic360_coder_start_decoder": (_I, [_P]),
    "lic360_coder_encodes": (_I, [_P, _P, _I, _P, _P, _I]),
    "lic360_coder_decodes": (_I, [_P, _P, _I, _P, _I, _P]),
    "lic360_coder_encode_one": (_I, [_P, _P, _I, _I, _I]),
    "lic360_coder_decode_one": (_I, [_P, _P, _I, _I, _P]),
    "lic360_coder_start_encoder_mem": (_I, [_P]),
    "lic360_coder_finish_mem": (_L, [_P]),
    "lic360_coder_get_bytes": (_L, [_P, _P, _L]),
    "lic360_coder_start_decoder_mem": (_I, [_P, _P, _L]),
    "lic360_coder_encode_rows": (_I, [_P, _P, _I, _I]),
    "lic360_coder_decode_rows": (_I, [_P, _P, _I, _I, _P]),
    "lic360_codec_create": (_P, [_I, _I, _I]),
    "lic360_codec_destroy": (None, [_P]),
    "lic360_codec_set_layer": (_I, [_P, _I, _I, _P, _P, _P]),
    "lic360_codec_encode": (_I, [_P, _P, _P, _P]),
    "lic360_codec_estimate": (_I, [_P, _P, _P, _P, _P, _P, _P]),
    "lic360_codec_stream_size": (_L, [_P, _I]),
    "lic360_codec_stream_copy": (_L, [_P, _I, _P, _L]),
    "lic360_codec_decode": (_I, [_P, _P, _L, _P, _L, _P, _P]),
    "lic360_codec_last_timing": (_I, [_P, _P, _I]),
    "lic360_codec_set_mode": (_I, [_P, _I]),
    "lic360_codec_kernel_times": (_I, [_P, _I, _P, _I]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(LIB, _name)  # AttributeError here means the library is stale: rebuild
    _fn.restype = _res
    _fn.argtypes = _args


def check(status):
    if status != 0:
        msg = LIB.lic360_last_error()
        raise RuntimeError("lic360_b200 (status %d): %s" % (status, msg.decode() if msg else "unknown error"))


def ptr(t):
    return t.data_ptr()


def ptr_or_null(t):
    return None if t is None else t.data_ptr()


def cstream(t):
    """cudaStream_t of torch's current stream on the tensor's device (the reference captures it once at op
    construction, base_opt.hpp:20-23)."""
    return torch.cuda.current_stream(t.device).cuda_stream
