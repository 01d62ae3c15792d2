"""ctypes binding of the C-ABI in include/sopro_b200.h (sopro_b200/lib/libsopro_b200.so).

There is NO fallback: if the shared library is missing or fails to load, importing
this module raises.  Build it with ./build.sh (or __graft_entry__.build())."""
from __future__ import annotations

import ctypes as C
import os

MAX_AR_LAYERS = 16
_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libsopro_b200.so")


class SoproError(RuntimeError):
    pass


class ArConfig(C.Structure):
    _fields_ = [
        ("d_model", C.c_int32), ("n_layers", C.c_int32), ("kernel", C.c_int32), ("n_heads", C.c_int32),
        ("vocab", C.c_int32), ("eos_id", C.c_int32),
        ("dilation", C.c_int32 * MAX_AR_LAYERS), ("has_attn", C.c_int32 * MAX_AR_LAYERS),
        ("weight_dtype", C.c_int32),
    ]


_FP = C.POINTER(C.c_float)


class ArLayerWeights(C.Structure):
    _fields_ = [(n, _FP) for n in (
        "norm_w", "glu_w", "glu_b", "dw_w", "dw_b", "ffn_norm_w", "ffn_w1", "ffn_b1", "ffn_w2", "ffn_b2",
        "nq_w", "nkv_w", "q_w", "k_w", "v_w", "o_w")] + [("gate_tanh", C.c_float)]


class ArWeights(C.Structure):
    _fields_ = [
        ("layer", ArLayerWeights * MAX_AR_LAYERS),
        ("final_norm_w", _FP), ("head_w", _FP), ("head_b", _FP), ("cb_embed", _FP),
        ("cb_embed_rows", C.c_int64), ("bos_row", C.c_int64),
    ]


class ArSampling(C.Structure):
    _fields_ = [
        ("top_p", C.c_float), ("temperature", C.c_float), ("recovery_top_p", C.c_float),
        ("recovery_temp", C.c_float), ("repetition_penalty", C.c_float),
        ("top_k", C.c_int32), ("anti_loop", C.c_int32), ("loop_streak", C.c_int32),
        ("min_gen_frames", C.c_int32), ("stop_on_first_eos", C.c_int32),
    ]


MIMI_MAX_LAYERS, MIMI_MAX_RATIOS = 16, 8


class MimiConfigC(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "hidden", "codebook_dim", "n_q", "n_sem", "vocab", "n_layers", "n_heads", "ffn", "window", "num_filters",
        "kernel", "last_kernel", "res_kernel", "compress", "n_ratios")] + [
        ("ratios", C.c_int32 * MIMI_MAX_RATIOS), ("norm_eps", C.c_float), ("rope_theta", C.c_float)]


class MimiLayerWeights(C.Structure):
    _fields_ = [(n, _FP) for n in ("ln1_w", "ln1_b", "q_w", "k_w", "v_w", "o_w", "ls1", "ln2_w", "ln2_b", "fc1_w", "fc2_w", "ls2")]


class MimiStageWeights(C.Structure):
    _fields_ = [(n, _FP) for n in ("convt_w", "convt_b", "res1_w", "res1_b", "res2_w", "res2_b")]


class MimiWeights(C.Structure):
    _fields_ = [("embed", _FP), ("sem_out_proj", _FP), ("ac_out_proj", _FP), ("upsample_w", _FP),
                ("layer", MimiLayerWeights * MIMI_MAX_LAYERS), ("conv0_w", _FP), ("conv0_b", _FP),
                ("stage", MimiStageWeights * MIMI_MAX_RATIOS), ("last_w", _FP), ("last_b", _FP)]


class MimiEncStageWeights(C.Structure):
    _fields_ = [(n, _FP) for n in ("res1_w", "res1_b", "res2_w", "res2_b", "down_w", "down_b")]


class MimiEncoderWeights(C.Structure):
    _fields_ = [("conv0_w", _FP), ("conv0_b", _FP), ("stage", MimiEncStageWeights * MIMI_MAX_RATIOS), ("last_w", _FP),
                ("last_b", _FP), ("layer", MimiLayerWeights * MIMI_MAX_LAYERS), ("downsample_w", _FP), ("sem_in_proj", _FP),
                ("ac_in_proj", _FP), ("embed", _FP)]


class SsmBlockWeights(C.Structure):
    _fields_ = [(n, C.POINTER(C.c_float)) for n in
                ("norm_w", "glu_w", "glu_b", "dw_w", "dw_b", "ffn_norm_w", "ffn_w1", "ffn_b1", "ffn_w2", "ffn_b2")]


class NarConfig(C.Structure):
    _fields_ = [("d_model", C.c_int32), ("n_layers", C.c_int32), ("kernel", C.c_int32), ("dilation", C.c_int32 * 16),
                ("n_codebooks", C.c_int32), ("codebook_size", C.c_int32), ("head_dim", C.c_int32),
                ("adapter_hidden", C.c_int32), ("n_stages", C.c_int32), ("stage_first", C.c_int32 * 8),
                ("stage_count", C.c_int32 * 8)]


class NarWeights(C.Structure):
    _fields_ = [("block", SsmBlockWeights * 16)] + [(n, C.POINTER(C.c_float)) for n in
                ("norm_w", "pre_w", "pre_b", "stage_emb", "adapter_norm_w", "adapter_w0", "adapter_b0", "adapter_w2", "adapter_b2")] + [
        ("head_w", C.POINTER(C.c_float) * 64), ("head_b", C.POINTER(C.c_float) * 64), ("head_id_emb", C.POINTER(C.c_float) * 8),
        ("mix", C.POINTER(C.c_float) * 8), ("prev_cb_weights", C.POINTER(C.c_float)), ("cb_embed", C.POINTER(C.c_float))]


class PrefillConfig(C.Structure):
    _fields_ = [("d_model", C.c_int32), ("n_layers_text", C.c_int32), ("text_kernel", C.c_int32), ("text_vocab", C.c_int32),
                ("sv_dim", C.c_int32), ("ref_layers", C.c_int32), ("ref_heads", C.c_int32), ("ref_gmax", C.c_float),
                ("max_text_len", C.c_int32), ("max_frames_pos", C.c_int32)]


class PrefillRefLayer(C.Structure):
    _fields_ = [("nq_w", C.POINTER(C.c_float)), ("q_w", C.POINTER(C.c_float)), ("o_w", C.POINTER(C.c_float)), ("gate", C.c_float)]


class PrefillWeights(C.Structure):
    _fields_ = [("text_emb", C.POINTER(C.c_float)), ("text_pos", C.POINTER(C.c_float)), ("frame_pos", C.POINTER(C.c_float)),
                ("text_block", SsmBlockWeights * 16), ("text_norm_w", C.POINTER(C.c_float)),
                ("film_w0", C.POINTER(C.c_float)), ("film_b0", C.POINTER(C.c_float)), ("film_w2", C.POINTER(C.c_float)),
                ("film_b2", C.POINTER(C.c_float)), ("film_norm_w", C.POINTER(C.c_float)), ("film_norm_b", C.POINTER(C.c_float)),
                ("ref_layer", PrefillRefLayer * 8), ("cond_norm_w", C.POINTER(C.c_float))]


class RefPrepConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("d_model", "sv_embed_dim", "sv_dim", "n_codebooks", "codebook_size", "sv_kernel",
                                         "ref_enc_layers", "ref_enc_kernel", "ref_layers", "ref_heads")]


class RefPrepKvLayer(C.Structure):
    _fields_ = [(n, C.POINTER(C.c_float)) for n in ("nkv_w", "k_w", "v_w")]


class RefPrepWeights(C.Structure):
    _fields_ = [(n, C.POINTER(C.c_float)) for n in ("sv_emb", "sv_cb_weights", "sv_dw0_w", "sv_dw0_b", "sv_dw1_w", "sv_dw1_b",
                                                    "pool_w0", "pool_b0", "pool_w2")] + [("pool_b2", C.c_float)] + [
        (n, C.POINTER(C.c_float)) for n in ("proj_w", "proj_b", "cb_embed", "ref_cb_weights")] + [
        ("ref_block", SsmBlockWeights * 16), ("ref_norm_w", C.POINTER(C.c_float)), ("layer", RefPrepKvLayer * 8)]


# every symbol include/sopro_b200.h declares: name -> (restype, argtypes)
_VP, _I, _I32P = C.c_void_p, C.c_int, C.POINTER(C.c_int32)
SYMBOLS = {
    "sopro_last_error": (C.c_char_p, []),
    "sopro_version": (C.c_char_p, []),
    "sopro_engine_create": (_I, [C.POINTER(ArConfig), C.POINTER(ArWeights), _I, C.POINTER(_VP)]),
    "sopro_engine_destroy": (_I, [_VP]),
    "sopro_engine_step_weight_bytes": (C.c_int64, [_VP]),
    "sopro_engine_num_sms": (_I, [_VP]),
    "sopro_ar_session_create": (_I, [_VP, _I, _I, _I, C.POINTER(_VP)]),
    "sopro_ar_session_destroy": (_I, [_VP]),
    "sopro_ar_session_set_team": (_I, [_VP, _I]),
    "sopro_ar_session_set_contraction": (_I, [_VP, _I]),
    "sopro_ar_begin": (_I, [_VP, _I, _I, _VP, _VP, _I, _I32P, _VP, _I, C.POINTER(ArSampling), _VP]),
    "sopro_ar_run": (_I, [_VP, _I, _VP]),
    "sopro_ar_outputs": (_I, [_VP, C.POINTER(_VP), C.POINTER(_VP), C.POINTER(_VP)]),
    "sopro_ar_read": (_I, [_VP, _VP, _VP, _VP, _VP]),
    "sopro_ar_position": (_I, [_VP]),
    "sopro_ar_generate_host": (_I, [_VP, _I, _I, _VP, _VP, _I, _I32P, _VP, _I, C.POINTER(ArSampling), _VP, _VP, _VP]),
    "sopro_ar_set_forced_tokens": (_I, [_VP, _VP]),
    "sopro_ar_set_trace": (_I, [_VP, _VP, _VP]),
    "sopro_ar_set_timing": (_I, [_VP, _VP, _I]),
    "sopro_ar_debug_sampled": (_I, [_VP, _VP, _VP]),
    "sopro_ar_debug_kv": (_I, [_VP, _VP, _VP, _VP]),
    "sopro_noise_create": (_I, [C.c_uint64, _VP]),
    "sopro_noise_rows": (_I, [_VP, _I, _I, _I, _VP]),
    "sopro_noise_destroy": (_I, [_VP]),
    "sopro_debug_pack_umma": (_I, [_VP, _I, _I, _I, _I, _VP, C.c_int64]),
    "sopro_debug_pack_w6": (_I, [_VP, _I, _I, _VP]),
    "sopro_debug_sample": (_I, [_VP, _I, _VP, _I, _VP, _I, _VP, _I, _I, _VP]),
    "sopro_mimi_create": (_I, [C.POINTER(MimiConfigC), C.POINTER(MimiWeights), _I, C.POINTER(_VP)]),
    "sopro_mimi_destroy": (_I, [_VP]),
    "sopro_mimi_samples_per_frame": (C.c_int64, [_VP]),
    "sopro_mimi_decode": (_I, [_VP, _VP, _I, _I, _VP, _VP]),
    "sopro_mimi_decode_host": (_I, [_VP, _VP, _I, _I, _VP, _VP]),
    "sopro_mimi_set_precision": (_I, [_VP, _I]),
    "sopro_mimi_set_graphs": (_I, [_VP, _I]),
    "sopro_mimi_check": (_I, [_VP, _VP]),
    "sopro_mimi_stream_create": (_I, [_VP, _I, C.POINTER(_VP)]),
    "sopro_mimi_stream_destroy": (_I, [_VP]),
    "sopro_mimi_stream_reset": (_I, [_VP, _VP]),
    "sopro_mimi_stream_frames": (C.c_int64, [_VP]),
    "sopro_mimi_decode_step": (_I, [_VP, _VP, _I, _VP, _VP]),
    "sopro_mimi_decode_step_host": (_I, [_VP, _VP, _I, _VP, _VP]),
    "sopro_mimi_encoder_create": (_I, [C.POINTER(MimiConfigC), C.POINTER(MimiEncoderWeights), _I, C.POINTER(_VP)]),
    "sopro_mimi_encoder_destroy": (_I, [_VP]),
    "sopro_mimi_encoded_frames": (C.c_int64, [_VP, C.c_int64]),
    "sopro_mimi_encode": (_I, [_VP, _VP, C.c_int64, _VP, _VP, _VP]),
    "sopro_mimi_encode_host": (_I, [_VP, _VP, C.c_int64, _VP, _VP, _VP]),
    "sopro_nar_create": (_I, [_VP, _VP, _I, C.POINTER(_VP)]),
    "sopro_nar_destroy": (_I, [_VP]),
    "sopro_nar_set_forced": (_I, [_VP, _VP]),
    "sopro_nar_set_contraction": (_I, [_VP, _I]),
    "sopro_nar_set_graphs": (_I, [_VP, _I]),
    "sopro_nar_refine": (_I, [_VP, _VP, C.c_int64, _VP, _VP, _I, _I, _VP, _VP]),
    "sopro_prefill_create": (_I, [_VP, _VP, _I, C.POINTER(_VP)]),
    "sopro_prefill_destroy": (_I, [_VP]),
    "sopro_refprep_create": (_I, [C.POINTER(RefPrepConfig), C.POINTER(RefPrepWeights), _I, C.POINTER(_VP)]),
    "sopro_refprep_destroy": (_I, [_VP]),
    "sopro_refprep_run": (_I, [_VP, _VP, _I, _VP, _VP, _VP, _VP, _VP]),
    "sopro_refprep_check": (_I, [_VP, _VP]),
    "sopro_prefill_run": (_I, [_VP, _VP, _VP, _I, _I, _VP, _I, _VP, _VP, _I, C.c_float, _I, _VP, _VP, _VP, _VP]),
    "sopro_prefill_run_voices": (_I, [_VP, _VP, _VP, _I, _I, _VP, _I, _VP, _VP, _VP, _VP, C.c_float, _I, _VP, _VP, _VP, _VP]),
    "sopro_debug_tc_gemm": (_I, [_VP, _I, C.c_int64, _I, _I, _I, _I, _VP, _I, _VP, _I, _I, _VP, _VP, _VP, _VP, _I, _VP]),
}

_lib = None


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SoproError(
            f"{LIB_PATH} not found: the CUDA extension is not built (run ./build.sh). "
            "sopro_b200 has no CPU or PyTorch fallback for the hot path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != 0:
        msg = load().sopro_last_error()
        raise SoproError(f"sopro_b200 error {rc}: {msg.decode() if msg else '?'}")
