"""ctypes binding of libavc_b200.so (include/avc_b200.h).  Fails loudly: no CPU fallback."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import os

_HERE = Path(__file__).resolve().parent
# AVC_LIB selects another build of the same library (instrumented / experimental builds made by scripts/); never a fallback
LIB_PATH = Path(os.environ["AVC_LIB"]).resolve() if os.environ.get("AVC_LIB") else _HERE / "libavc_b200.so"

AVC_MAX_BLOCKS = 8


class EncoderDesc(C.Structure):
    _fields_ = [("c_in", C.c_int32), ("c_h", C.c_int32), ("c_out", C.c_int32), ("kernel_size", C.c_int32),
                ("bank_size", C.c_int32), ("c_bank", C.c_int32), ("n_conv_blocks", C.c_int32),
                ("n_dense_blocks", C.c_int32), ("subsample", C.c_int32 * AVC_MAX_BLOCKS), ("neg_slope", C.c_float)]


class DecoderDesc(C.Structure):
    _fields_ = [("c_in", C.c_int32), ("c_cond", C.c_int32), ("c_h", C.c_int32), ("c_out", C.c_int32),
                ("kernel_size", C.c_int32), ("n_conv_blocks", C.c_int32), ("upsample", C.c_int32 * AVC_MAX_BLOCKS),
                ("neg_slope", C.c_float)]


class ModelDesc(C.Structure):
    _fields_ = [("speaker", EncoderDesc), ("content", EncoderDesc), ("decoder", DecoderDesc)]


class WeightView(C.Structure):
    _fields_ = [("name", C.c_char_p), ("data", C.c_void_p), ("ndim", C.c_int32), ("shape", C.c_int64 * 4)]


class HeaderArgs(C.Structure):
    _fields_ = [
        ("source", C.c_void_p), ("src_stride", C.c_int64 * 3), ("B", C.c_int32), ("T", C.c_int32),
        ("target", C.c_void_p), ("tgt_stride", C.c_int64 * 3), ("T_tgt", C.c_int32),
        ("header0", C.c_void_p), ("hdr_stride", C.c_int64 * 2),
        ("header_out", C.c_void_p), ("out_stride", C.c_int64 * 2),
        ("loss_out", C.c_void_p), ("grad_out", C.c_void_p),
        ("eps", C.c_float), ("lam", C.c_float), ("lr", C.c_float), ("n_iters", C.c_int32),
        ("inv_norm", C.c_double), ("use_graph", C.c_int32),
    ]


class SpkGradArgs(C.Structure):
    _fields_ = [
        ("perturbed", C.c_void_p), ("p_stride", C.c_int64 * 3), ("B", C.c_int32), ("T", C.c_int32),
        ("source", C.c_void_p), ("s_stride", C.c_int64 * 3),
        ("target", C.c_void_p), ("t_stride", C.c_int64 * 3), ("T_tgt", C.c_int32),
        ("grad_out", C.c_void_p), ("g_stride", C.c_int64 * 3),
        ("loss_out", C.c_void_p),
        ("lam", C.c_float), ("inv_norm", C.c_double), ("use_graph", C.c_int32),
    ]


class PmTrainerArgs(C.Structure):
    _fields_ = [
        ("B", C.c_int32), ("F", C.c_int32), ("T", C.c_int32), ("future_steps", C.c_int32),
        ("eps1", C.c_float), ("eps2", C.c_float), ("eps3", C.c_float), ("lam", C.c_float),
        ("beta1", C.c_float), ("beta2", C.c_float), ("adam_eps", C.c_float), ("inv_norm", C.c_double),
    ]


class AudioDesc(C.Structure):
    _fields_ = [("sample_rate", C.c_int32), ("n_fft", C.c_int32), ("hop_length", C.c_int32), ("win_length", C.c_int32),
                ("n_mels", C.c_int32), ("preemph", C.c_float), ("ref_db", C.c_float), ("max_db", C.c_float)]


# int (*avc_allreduce_fn)(void* ctx, float* comm, int64_t n_floats, void* stream)
ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p)


class AttackArgs(C.Structure):
    _fields_ = [
        ("vc_tgt", C.c_void_p), ("tgt_stride", C.c_int64 * 3), ("B", C.c_int32), ("T_tgt", C.c_int32),
        ("adv_tgt", C.c_void_p), ("adv_stride", C.c_int64 * 3), ("T_adv", C.c_int32),
        ("vc_src", C.c_void_p), ("src_stride", C.c_int64 * 3), ("T_src", C.c_int32),
        ("w0", C.c_void_p), ("w0_stride", C.c_int64 * 3),
        ("adv_out", C.c_void_p), ("out_stride", C.c_int64 * 3),
        ("loss_out", C.c_void_p), ("grad_out", C.c_void_p),
        ("eps", C.c_float), ("n_iters", C.c_int32), ("inv_norm", C.c_double), ("use_graph", C.c_int32),
    ]


class AttackVarlenArgs(C.Structure):
    _fields_ = [
        ("vc_tgt", C.c_void_p), ("w0", C.c_void_p), ("adv_out", C.c_void_p), ("grad_out", C.c_void_p),
        ("frames_host", C.POINTER(C.c_int32)), ("B", C.c_int32),
        ("adv_tgt", C.c_void_p), ("adv_stride", C.c_int64 * 3), ("T_adv", C.c_int32),
        ("vc_src", C.c_void_p), ("src_stride", C.c_int64 * 3), ("T_src", C.c_int32),
        ("loss_out", C.c_void_p), ("eps", C.c_float), ("n_iters", C.c_int32), ("inv_norm", C.c_double), ("use_graph", C.c_int32),
    ]


EXPORTS = [
    "avc_create", "avc_destroy", "avc_last_error", "avc_load_weights", "avc_emb_attack", "avc_e2e_attack",
    "avc_fb_attack", "avc_attack_varlen", "avc_speaker_encoder", "avc_inference", "avc_decoder_frames", "avc_conv1d_fwd",
    "avc_conv1d_dgrad", "avc_conv1d_wgrad", "avc_conv1d_wgrad_ex", "avc_instnorm_adain_act_fwd", "avc_instnorm_adain_act_bwd", "avc_adam_tanh_step",
    "avc_unit_timing", "avc_unit_last_ms",
    "avc_kernel_launches", "avc_launches_per_iter", "avc_version",
    "avc_attack_begin", "avc_attack_step", "avc_attack_end", "avc_session_launches", "avc_session_profile",
    "avc_header_optimize", "avc_header_begin", "avc_header_step", "avc_header_grad_buffer",
    "avc_pm_create", "avc_pm_destroy", "avc_pm_last_error", "avc_pm_load_weights", "avc_pm_out_shape", "avc_pm_forward",
    "avc_pm_train_step", "avc_pm_kernel_launches",
    "avc_spk_grad_begin", "avc_spk_grad_step",
    "avc_pm_set_allreduce", "avc_pm_param_count", "avc_pm_trainer_begin", "avc_pm_trainer_step", "avc_pm_trainer_grads",
    "avc_pm_trainer_end", "avc_pm_export_weights",
    "avc_audio_create", "avc_audio_destroy", "avc_audio_last_error", "avc_audio_frames", "avc_audio_samples",
    "avc_audio_wav2mel", "avc_audio_mel2wav", "avc_audio_wav2mel_batch", "avc_audio_mel2wav_batch", "avc_audio_kernel_launches",
    "avc_audio_wav2mel_varlen", "avc_audio_mel2wav_varlen",
]

_lib = None


def load() -> C.CDLL:
    """dlopen the in-tree library.  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m attack_vc_b200.build` "
            "(attack_vc_b200 has no CPU or PyTorch fallback)")
    if not os.environ.get("AVC_LIB") and (_HERE / "csrc").is_dir():
        # the binary must be the one these sources build (content hash baked into avc_version()): rebuild, or fail loudly
        from . import build as _build
        if _build.built_hash(LIB_PATH) != _build.source_hash():
            _build.build_library(force=True)
            if _build.built_hash(LIB_PATH) != _build.source_hash():
                raise RuntimeError(f"{LIB_PATH} was not built from the sources in {_HERE / 'csrc'} and could not be rebuilt")
    lib = C.CDLL(str(LIB_PATH))
    vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float
    P = C.POINTER
    lib.avc_create.argtypes = [P(vp), P(ModelDesc), C.c_int]
    lib.avc_create.restype = C.c_int
    lib.avc_destroy.argtypes = [vp]
    lib.avc_destroy.restype = None
    lib.avc_last_error.argtypes = [vp]
    lib.avc_last_error.restype = C.c_char_p
    lib.avc_load_weights.argtypes = [vp, P(WeightView), i32]
    for nm in ("avc_emb_attack", "avc_e2e_attack", "avc_fb_attack"):
        getattr(lib, nm).argtypes = [vp, P(AttackArgs), vp]
    lib.avc_attack_varlen.argtypes = [vp, i32, P(AttackVarlenArgs), vp]
    lib.avc_attack_begin.argtypes = [vp, i32, P(AttackArgs), vp, P(vp)]
    lib.avc_attack_step.argtypes = [vp, i32, vp]
    lib.avc_attack_end.argtypes = [vp, vp]
    lib.avc_session_launches.argtypes = [vp]
    lib.avc_session_launches.restype = i32
    lib.avc_session_profile.argtypes = [vp, i32, P(i32), P(f32), P(C.c_double), P(C.c_double), vp]
    lib.avc_speaker_encoder.argtypes = [vp, vp, P(i64), i32, i32, vp, vp]
    lib.avc_inference.argtypes = [vp, vp, P(i64), i32, vp, P(i64), i32, i32, vp, vp]
    lib.avc_decoder_frames.argtypes = [vp, i32]
    lib.avc_decoder_frames.restype = i32
    lib.avc_conv1d_fwd.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]
    lib.avc_conv1d_dgrad.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]
    lib.avc_conv1d_wgrad.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp]
    lib.avc_conv1d_wgrad_ex.argtypes = [vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, i32, vp]
    lib.avc_instnorm_adain_act_fwd.argtypes = [vp, vp, vp, vp, i32, vp, vp, i32, i32, i32, f32, vp]
    lib.avc_instnorm_adain_act_bwd.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, f32, vp]
    lib.avc_adam_tanh_step.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, f32, i32, vp]
    lib.avc_unit_timing.argtypes = [vp, i32]
    lib.avc_unit_last_ms.argtypes = [vp]
    lib.avc_unit_last_ms.restype = f32
    lib.avc_kernel_launches.argtypes = [vp]
    lib.avc_kernel_launches.restype = i64
    lib.avc_launches_per_iter.argtypes = [vp]
    lib.avc_launches_per_iter.restype = i32
    lib.avc_header_optimize.argtypes = [vp, P(HeaderArgs), vp]
    lib.avc_header_begin.argtypes = [vp, P(HeaderArgs), vp, P(vp)]
    lib.avc_header_step.argtypes = [vp, i32, i32, vp]
    lib.avc_header_grad_buffer.argtypes = [vp, P(i64)]
    lib.avc_header_grad_buffer.restype = vp
    lib.avc_pm_create.argtypes = [P(vp), C.c_int]
    lib.avc_pm_destroy.argtypes = [vp]
    lib.avc_pm_destroy.restype = None
    lib.avc_pm_last_error.argtypes = [vp]
    lib.avc_pm_last_error.restype = C.c_char_p
    lib.avc_pm_load_weights.argtypes = [vp, P(WeightView), i32]
    lib.avc_pm_out_shape.argtypes = [i32, i32, P(i32), P(i32)]
    lib.avc_pm_forward.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
    lib.avc_pm_train_step.argtypes = [vp, vp, i32, i32, i32, vp, vp, vp, P(WeightView), i32, vp]
    lib.avc_pm_kernel_launches.argtypes = [vp]
    lib.avc_pm_kernel_launches.restype = i64
    lib.avc_spk_grad_begin.argtypes = [vp, P(SpkGradArgs), vp, P(vp)]
    lib.avc_spk_grad_step.argtypes = [vp, vp]
    lib.avc_pm_set_allreduce.argtypes = [vp, ALLREDUCE_FN, vp, vp, i64, i32]
    lib.avc_pm_param_count.argtypes = [vp]
    lib.avc_pm_param_count.restype = i64
    lib.avc_pm_trainer_begin.argtypes = [vp, vp, P(PmTrainerArgs), vp, P(vp)]
    lib.avc_pm_trainer_step.argtypes = [vp, vp, vp, f32, vp, vp]
    lib.avc_pm_trainer_grads.argtypes = [vp, P(WeightView), i32, vp]
    lib.avc_pm_trainer_end.argtypes = [vp]
    lib.avc_pm_export_weights.argtypes = [vp, P(WeightView), i32, vp]
    lib.avc_audio_create.argtypes = [P(vp), P(AudioDesc), C.c_int]
    lib.avc_audio_destroy.argtypes = [vp]
    lib.avc_audio_destroy.restype = None
    lib.avc_audio_last_error.argtypes = [vp]
    lib.avc_audio_last_error.restype = C.c_char_p
    lib.avc_audio_frames.argtypes = [vp, i64]
    lib.avc_audio_frames.restype = i32
    lib.avc_audio_samples.argtypes = [vp, i32]
    lib.avc_audio_samples.restype = i64
    lib.avc_audio_wav2mel.argtypes = [vp, vp, i64, vp, vp]
    lib.avc_audio_mel2wav.argtypes = [vp, vp, i32, i32, vp, vp]
    lib.avc_audio_wav2mel_batch.argtypes = [vp, vp, i32, i64, vp, vp]
    lib.avc_audio_mel2wav_batch.argtypes = [vp, vp, i32, i32, i32, vp, vp]
    lib.avc_audio_wav2mel_varlen.argtypes = [vp, vp, P(i64), i32, vp, vp, vp, vp]
    lib.avc_audio_mel2wav_varlen.argtypes = [vp, vp, P(i32), i32, i32, vp, vp, vp, vp]
    lib.avc_audio_kernel_launches.argtypes = [vp]
    lib.avc_audio_kernel_launches.restype = i64
    lib.avc_version.argtypes = []
    lib.avc_version.restype = C.c_char_p
    _lib = lib
    return lib
