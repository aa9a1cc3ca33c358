"""ctypes binding of libctn_b200.so (C ABI declared in include/ctn_b200.h).

PyTorch is used for device memory and streams only.  There is NO CPU / eager fallback: if the shared
library is missing, importing this module raises, and every op raises on non-CUDA tensors.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional, Tuple

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CTN_B200_LIB", os.path.join(os.path.dirname(_HERE), "libctn_b200.so"))

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build the sm_100a extension first "
        "(python -c 'import __graft_entry__ as g; g.build()' or dnn-based_source_separation_b200/csrc/build.sh). "
        "There is no CPU fallback.")

lib = C.CDLL(LIB_PATH)

CTN_OK, CTN_EINVAL, CTN_EUNSUPPORTED, CTN_EALIGN, CTN_EWORKSPACE, CTN_ENOTBUILT = 0, -1, -2, -3, -4, -5
MATH_FP32, MATH_TF32X3, MATH_TF32, MATH_F16X3 = 0, 1, 2, 3
MATH_NAMES = {"fp32": MATH_FP32, "tf32x3": MATH_TF32X3, "tf32": MATH_TF32, "f16x3": MATH_F16X3}

_fp = C.c_void_p  # device pointers are passed as integers


class Config(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_basis", "kernel_size", "stride", "bottleneck", "hidden", "skip", "sep_kernel", "num_blocks", "num_layers",
        "n_sources", "causal", "enc_relu", "mask_softmax", "math")] + [("eps", C.c_float), ("eps_tcn", C.c_float), ("in_channels", C.c_int32)]


BLOCK_FIELDS = ("bottleneck_w", "bottleneck_b", "prelu1", "norm1_g", "norm1_b", "dw_w", "dw_b", "prelu2", "norm2_g",
                "norm2_b", "out_w", "out_b", "skip_w", "skip_b")


class BlockParams(C.Structure):
    _fields_ = [(n, _fp) for n in BLOCK_FIELDS]


class Params(C.Structure):
    _fields_ = [("enc_w", _fp), ("norm0_g", _fp), ("norm0_b", _fp), ("bn_w", _fp), ("bn_b", _fp),
                ("blocks", C.POINTER(BlockParams)), ("prelu_out", _fp), ("mask_w", _fp), ("mask_b", _fp), ("dec_w", _fp)]


def _sig(name, restype, *argtypes):
    fn = getattr(lib, name)
    fn.restype = restype
    fn.argtypes = list(argtypes)
    return fn


_i, _f, _sz = C.c_int, C.c_float, C.c_size_t
ctn_version = _sig("ctn_version", _i)
ctn_strerror = _sig("ctn_strerror", C.c_char_p, _i)
ctn_has_tcgen05 = _sig("ctn_has_tcgen05", _i)
ctn_frames = _sig("ctn_frames", _i, _i, _i, _i, C.POINTER(_i), C.POINTER(_i))
ctn_pitch = _sig("ctn_pitch", _i, _i)
ctn_workspace_bytes = _sig("ctn_workspace_bytes", _i, C.POINTER(Config), _i, _i, C.POINTER(_sz))
ctn_encoder_fwd = _sig("ctn_encoder_fwd", _i, _fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _fp, _fp)
ctn_decoder_fwd = _sig("ctn_decoder_fwd", _i, _fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _fp)
ctn_gln_fwd = _sig("ctn_gln_fwd", _i, _fp, _fp, _fp, _fp, _i, _i, _i, _f, _fp, _fp)
ctn_cln_fwd = _sig("ctn_cln_fwd", _i, _fp, _fp, _fp, _fp, _i, _i, _i, _f, _fp, _fp)
ctn_tcn_workspace_bytes = _sig("ctn_tcn_workspace_bytes", _i, C.POINTER(Config), _i, _i, C.POINTER(_sz))
ctn_tcn_fwd = _sig("ctn_tcn_fwd", _i, C.POINTER(Config), C.POINTER(BlockParams), _fp, _fp, _i, _i, _fp, _sz, _fp)
ctn_tcn_blocks_fwd = _sig("ctn_tcn_blocks_fwd", _i, C.POINTER(Config), C.POINTER(BlockParams), _i, C.POINTER(_i), _fp, _fp, _fp, _i, _i, _fp, _sz, _fp)
ctn_convtasnet_fwd = _sig("ctn_convtasnet_fwd", _i, C.POINTER(Config), C.POINTER(Params), _fp, _i, _i, _fp, _fp, _fp, _sz, _fp)
ctn_separator_fwd = _sig("ctn_separator_fwd", _i, C.POINTER(Config), C.POINTER(Params), _fp, _i, _i, _fp, _fp, _sz, _fp)
ctn_sisdr_fwd = _sig("ctn_sisdr_fwd", _i, _fp, _fp, _i, _i, _f, _fp, _fp, _fp)
ctn_sisdr_pit_fwd = _sig("ctn_sisdr_pit_fwd", _i, _fp, _fp, _i, _i, _i, _f, _fp, _fp, _fp, _fp, _fp, _fp)
ctn_sisdr_pit_scratch_bytes = _sig("ctn_sisdr_pit_scratch_bytes", _sz, _i, _i)
ctn_host_io_bytes = _sig("ctn_host_io_bytes", _sz, C.POINTER(Config), _i, _i)
ctn_convtasnet_loss_host = _sig("ctn_convtasnet_loss_host", _i, C.POINTER(Config), C.POINTER(Params), _fp, _fp, _i, _i,
                                _fp, _fp, _fp, _fp, _sz, _fp, _sz, _f, _fp)
ctn_train_workspace_bytes = _sig("ctn_train_workspace_bytes", _i, C.POINTER(Config), _i, _i, C.POINTER(_sz))
ctn_convtasnet_fwd_train = _sig("ctn_convtasnet_fwd_train", _i, C.POINTER(Config), C.POINTER(Params), _fp, _i, _i, _fp, _fp, _sz, _fp)
ctn_convtasnet_bwd = _sig("ctn_convtasnet_bwd", _i, C.POINTER(Config), C.POINTER(Params), C.POINTER(Params), _fp, _fp, _i, _i,
                          _fp, _sz, _fp)
ctn_encoder_mc_fwd = _sig("ctn_encoder_mc_fwd", _i, _fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _fp, _fp)
ctn_decoder_mc_fwd = _sig("ctn_decoder_mc_fwd", _i, _fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _fp)
ctn_sdr_fwd = _sig("ctn_sdr_fwd", _i, _fp, _fp, _i, _i, _f, _fp, _fp, _fp)
ctn_sisdr_pit_bwd = _sig("ctn_sisdr_pit_bwd", _i, _fp, _fp, _fp, _i, _i, _i, _f, _fp, _fp, _f, _fp, _fp)
ctn_last_launch_count = _sig("ctn_last_launch_count", _i)
ctn_total_launch_count = _sig("ctn_total_launch_count", C.c_longlong)
# DPRNN-TasNet path (cfg4) + separator stages on the pitched layout
ctn_segment_fwd = _sig("ctn_segment_fwd", _i, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _fp)
ctn_overlap_add_fwd = _sig("ctn_overlap_add_fwd", _i, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _fp)
ctn_dprnn_norm_res_fwd = _sig("ctn_dprnn_norm_res_fwd", _i, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _f, _i, _fp, _fp)
ctn_bilstm_supported = _sig("ctn_bilstm_supported", _i, _i, _i, _i)
ctn_debug_lstm_timeline = _sig("ctn_debug_lstm_timeline", _i, C.POINTER(C.c_ulonglong), _i)
ctn_bilstm_workspace_bytes = _sig("ctn_bilstm_workspace_bytes", _sz, _i, _i, _i)
ctn_bilstm_proj_fwd = _sig("ctn_bilstm_proj_fwd", _i, _fp, _i, _i, _i, _i, C.POINTER(_fp), _fp, _i, _fp, _fp, _fp, _fp, _sz, _fp)
ctn_dprnn_norm_res2_fwd = _sig("ctn_dprnn_norm_res2_fwd", _i, _fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _f, _i, _fp, _fp, _fp)
ctn_stage_workspace_bytes = _sig("ctn_stage_workspace_bytes", _sz, _i, _i)
ctn_sep_head_fwd = _sig("ctn_sep_head_fwd", _i, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _f, _i, _fp, _sz, _fp)
ctn_sep_tail_fwd = _sig("ctn_sep_tail_fwd", _i, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i,
                        _fp, _sz, _fp)
ctn_clip_adam_chunks = _sig("ctn_clip_adam_chunks", _i, C.POINTER(_i), _i, C.POINTER(_i), C.POINTER(_i), _i)
ctn_clip_adam_step = _sig("ctn_clip_adam_step", _i, _fp, _i, _fp, _fp, _fp, _i, _fp, _sz, _fp, _fp, _fp, _fp, _fp, _f, _f, _f, _f, _f, _fp, _fp)
ctn_depthwise_conv1d_fwd = _sig("ctn_depthwise_conv1d_fwd", _i, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _i, _i, _fp)
ctn_pointwise_conv1d_fwd = _sig("ctn_pointwise_conv1d_fwd", _i, _fp, _fp, _fp, _fp, _i, _i, _i, _i, _i, _i, _fp, _sz, _fp)
ctn_profile_enable = _sig("ctn_profile_enable", _i, _i)
ctn_profile_read = _sig("ctn_profile_read", _i, C.POINTER(C.c_double), C.POINTER(_i))
STAGES = ("prep", "enc", "head", "pw1", "dw", "pw2", "fin", "mask", "dec", "loss")

EXPORTED = [
    "ctn_version", "ctn_strerror", "ctn_has_tcgen05", "ctn_frames", "ctn_pitch", "ctn_workspace_bytes", "ctn_encoder_fwd",
    "ctn_decoder_fwd", "ctn_gln_fwd", "ctn_cln_fwd", "ctn_tcn_workspace_bytes", "ctn_tcn_fwd", "ctn_convtasnet_fwd",
    "ctn_separator_fwd", "ctn_sisdr_fwd", "ctn_sisdr_pit_fwd", "ctn_sisdr_pit_scratch_bytes", "ctn_host_io_bytes",
    "ctn_convtasnet_loss_host", "ctn_train_workspace_bytes", "ctn_convtasnet_fwd_train", "ctn_convtasnet_bwd",
    "ctn_sisdr_pit_bwd", "ctn_sdr_fwd", "ctn_encoder_mc_fwd", "ctn_decoder_mc_fwd", "ctn_last_launch_count", "ctn_total_launch_count", "ctn_profile_enable", "ctn_profile_read",
    "ctn_segment_fwd", "ctn_overlap_add_fwd", "ctn_dprnn_norm_res_fwd", "ctn_stage_workspace_bytes", "ctn_sep_head_fwd", "ctn_sep_tail_fwd",
    "ctn_clip_adam_chunks", "ctn_clip_adam_step", "ctn_tcn_blocks_fwd",
    "ctn_depthwise_conv1d_fwd", "ctn_pointwise_conv1d_fwd",
    "ctn_debug_lstm_timeline", "ctn_bilstm_supported", "ctn_bilstm_workspace_bytes", "ctn_bilstm_proj_fwd", "ctn_dprnn_norm_res2_fwd",
]


def profile_read():
    """-> {stage: (milliseconds, launches)} accumulated since the last read (synchronises on the stage events)."""
    ms = (C.c_double * len(STAGES))()
    ln = (C.c_int * len(STAGES))()
    check(ctn_profile_read(ms, ln), "ctn_profile_read")
    return {s: (ms[i], ln[i]) for i, s in enumerate(STAGES)}


def check(status: int, what: str = "") -> None:
    """Map C status codes to the exceptions the reference raises (SURVEY.md 8b)."""
    if status == CTN_OK:
        return
    msg = f"{what}: {ctn_strerror(status).decode()} (status {status})"
    if status == CTN_EUNSUPPORTED:
        raise NotImplementedError(msg)
    if status in (CTN_EINVAL, CTN_EALIGN):
        raise ValueError(msg)
    raise RuntimeError(msg)


def require_cuda(*tensors: torch.Tensor) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("ctn_b200 runs on CUDA (sm_100a) tensors only; there is no CPU fallback")
        if t.dtype != torch.float32:
            raise TypeError(f"ctn_b200 computes in float32, got {t.dtype}")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError("all tensors must live on the same CUDA device")
    return dev


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


# grow-only workspaces, one per (device, stream, tag): stream-ordered reuse is safe, nothing is retained by C
_workspaces: Dict[Tuple[int, int, str], torch.Tensor] = {}


def workspace(device: torch.device, nbytes: int, tag: str = "ws") -> torch.Tensor:
    key = (device.index if device.index is not None else torch.cuda.current_device(), stream_ptr(device), tag)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(int(nbytes) + 256, dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    return buf


def release_workspaces() -> None:
    _workspaces.clear()


def frames_of(T: int, kernel_size: int, stride: int) -> Tuple[int, int, int]:
    pl, pr = C.c_int(0), C.c_int(0)
    fr = ctn_frames(T, kernel_size, stride, C.byref(pl), C.byref(pr))
    if fr <= 0:
        raise ValueError(f"invalid geometry T={T}, kernel_size={kernel_size}, stride={stride}")
    return fr, pl.value, pr.value
