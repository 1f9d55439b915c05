"""ctypes binding of include/wetts_b200.h.  Fails loudly when the CUDA library is missing:
there is no CPU fallback behind this package."""
import ctypes as C
import os

_CSRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc")
LIB_PATH = os.path.join(_CSRC, "libwetts_b200.so")

MAX_UPSAMPLES, MAX_RB_KERNELS, MAX_DILATIONS = 6, 4, 4


class VitsConfig(C.Structure):
    _fields_ = [
        ("n_vocab", C.c_int32), ("n_speakers", C.c_int32), ("inter_channels", C.c_int32),
        ("hidden_channels", C.c_int32), ("filter_channels", C.c_int32), ("n_heads", C.c_int32),
        ("n_layers", C.c_int32), ("kernel_size", C.c_int32), ("gin_channels", C.c_int32),
        ("use_sdp", C.c_int32), ("resblock_type", C.c_int32), ("n_resblock_kernels", C.c_int32),
        ("resblock_kernel_sizes", C.c_int32 * MAX_RB_KERNELS),
        ("resblock_n_dilations", C.c_int32 * MAX_RB_KERNELS),
        ("resblock_dilations", (C.c_int32 * MAX_DILATIONS) * MAX_RB_KERNELS),
        ("n_upsamples", C.c_int32),
        ("upsample_rates", C.c_int32 * MAX_UPSAMPLES),
        ("upsample_kernel_sizes", C.c_int32 * MAX_UPSAMPLES),
        ("upsample_initial_channel", C.c_int32),
        ("vocoder_type", C.c_int32), ("vocos_channels", C.c_int32), ("vocos_h_channels", C.c_int32),
        ("vocos_out_channels", C.c_int32), ("vocos_num_layers", C.c_int32), ("vocos_n_fft", C.c_int32),
        ("vocos_hop_length", C.c_int32), ("flow_type", C.c_int32),
    ]


_P, _I, _F, _SZ, _I64 = C.c_void_p, C.c_int, C.c_float, C.c_size_t, C.c_int64

# name -> (restype, argtypes); must list every symbol include/wetts_b200.h declares
PROTOTYPES = {
    "wetts_last_error": (C.c_char_p, []),
    "wetts_version": (C.c_char_p, []),
    "wetts_set_option": (_I, [C.c_char_p, _I]),
    "wetts_get_option": (_I, [C.c_char_p, C.POINTER(_I)]),
    "wetts_vits_set_option": (_I, [_P, C.c_char_p, _I]),
    "wetts_vits_get_option": (_I, [_P, C.c_char_p, C.POINTER(_I)]),
    "wetts_vits_create": (_I, [C.POINTER(VitsConfig), _I, C.POINTER(_P)]),
    "wetts_vits_set_tensor": (_I, [_P, C.c_char_p, _P, C.POINTER(_I64), _I]),
    "wetts_vits_finalize": (_I, [_P]),
    "wetts_vits_destroy": (None, [_P]),
    "wetts_vits_upsample_factor": (_I, [_P]),
    "wetts_speaker_embedding": (_I, [_P, _P, _I, _P, _P]),
    "wetts_text_encoder_workspace_bytes": (_SZ, [_P, _I, _I]),
    "wetts_text_encoder_forward": (_I, [_P, _P, _P, _I, _I, _P, _P, _P, _P, _SZ, _P]),
    "wetts_duration_workspace_bytes": (_SZ, [_P, _I, _I]),
    "wetts_duration_forward": (_I, [_P, _P, _P, _P, _P, _F, _I, _I, _P, _P, _SZ, _P]),
    "wetts_length_regulate": (_I, [_P, _P, _P, _P, _F, _I, _I, _P, _P, _P, _P]),
    "wetts_expand_prior": (_I, [_P, _P, _P, _P, _P, _P, _P, _I64, _I64, _F, _I, _I, _I, _P, _P, _P, _P, _P, _P]),
    "wetts_flow_workspace_bytes": (_SZ, [_P, _I, _I]),
    "wetts_flow_reverse": (_I, [_P, _P, _P, _P, _I, _I, _P, _SZ, _P]),
    "wetts_flow_forward": (_I, [_P, _P, _P, _P, _I, _I, _P, _SZ, _P]),
    "wetts_generator_workspace_bytes": (_SZ, [_P, _I, _I]),
    "wetts_generator_forward": (_I, [_P, _P, _P, _P, _I, _I, _P, _P, _SZ, _P]),
    "wetts_generator_forward_view": (_I, [_P, _P, _I64, _I64, _P, _P, _I, _I, _P, _P, _SZ, _P]),
    "wetts_vits_infer_workspace_bytes": (_SZ, [_P, _I, _I, _I]),
    "wetts_vits_infer_durations": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _P, _P, _P, C.POINTER(_I), _P, _SZ, _P]),
    "wetts_vits_infer_synthesize": (_I, [_P, _P, _P, _P, _P, _I64, _I64, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _P, _P,
                                         _SZ, _P]),
    "wetts_vits_decoder_workspace_bytes": (_SZ, [_P, _I, _I]),
    "wetts_vits_forward_decoder": (_I, [_P, _P, _P, _I, _I, _P, _P, _SZ, _P]),
    "wetts_posterior_workspace_bytes": (_SZ, [_P, _I, _I]),
    "wetts_posterior_encoder_forward": (_I, [_P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _SZ, _P]),
    "wetts_spectrogram_workspace_bytes": (_SZ, [_P, _I, _I64]),
    "wetts_spectrogram": (_I, [_P, _P, _P, _I, _I64, _P, _P, _P, _SZ, _P]),
    "wetts_vits_voice_conversion_workspace_bytes": (_SZ, [_P, _I, _I]),
    "wetts_vits_voice_conversion": (_I, [_P, _P, _P, _P, _P, _P, _I, _I, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "wetts_audio_to_int16": (_I, [_P, _P, _I, _I64, _I, _P, _P, _P]),
    "wetts_vits_check_fault": (_I, [_P, _P, _I]),
    "wetts_vits_launch_count": (C.c_uint64, [_P]),
}

_lib = None


class WettsError(RuntimeError):
    pass


def load():
    """dlopen the engine; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise WettsError(
            f"{LIB_PATH} not found: build it with `python -m wetts_b200.build` (nvcc, sm_100a). "
            "wetts_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise WettsError(load().wetts_last_error().decode("utf-8", "replace"))
