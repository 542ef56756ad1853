"""ctypes binding of libtdx.so (include/tdx.h).  Loading fails loudly: there is no CPU or PyTorch fallback."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libtdx.so"


class TdxError(RuntimeError):
    pass


class TdxOutSpec(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("kind", C.c_int32), ("spatial", C.c_int32), ("scale", C.c_float),
                ("_pad", C.c_int32)]


class TdxIgemmDesc(C.Structure):
    _fields_ = [
        ("a_ptr", C.c_void_p * 3), ("a_channels", C.c_int32 * 3), ("a_taps", C.c_int32 * 3), ("n_seg", C.c_int32),
        ("b_packed", C.c_void_p), ("c_out", C.c_int32), ("n_per_item", C.c_int32), ("n_img", C.c_int32),
        ("height", C.c_int32), ("width", C.c_int32), ("epi_flags", C.c_int32), ("cvec", C.c_void_p), ("resid", C.c_void_p),
        ("resid_spatial", C.c_int32), ("resid_pnorm", C.c_int32), ("resid_scale", C.c_float), ("clip", C.c_float),
        ("out", TdxOutSpec * 3), ("rms_out", C.c_void_p), ("resid_inv", C.c_void_p),
        ("k_split", C.c_int32), ("_reserved", C.c_int32),
    ]


class TdxConvInDesc(C.Structure):
    _fields_ = [
        ("src", C.c_void_p * 2), ("src_channels", C.c_int32 * 2), ("src_dtype", C.c_int32 * 2),
        ("src_scale", C.c_void_p * 2), ("weight", C.c_void_p), ("c_out", C.c_int32), ("n_img", C.c_int32),
        ("height", C.c_int32), ("width", C.c_int32), ("out", TdxOutSpec * 3),
    ]


class TdxIm2colDesc(C.Structure):
    _fields_ = [
        ("src", C.c_void_p * 2), ("src_channels", C.c_int32 * 2), ("src_dtype", C.c_int32 * 2),
        ("src_scale", C.c_void_p * 2), ("out", C.c_void_p), ("k_pad", C.c_int32), ("n_img", C.c_int32),
        ("height", C.c_int32), ("width", C.c_int32),
    ]


class TdxConvOutDesc(C.Structure):
    _fields_ = [
        ("x", C.c_void_p), ("c_in", C.c_int32), ("weight", C.c_void_p), ("c_out", C.c_int32), ("n_img", C.c_int32),
        ("height", C.c_int32), ("width", C.c_int32), ("model_out", C.c_void_p), ("sched_coef", C.c_void_p),
        ("sample", C.c_void_p), ("x0_prev", C.c_void_p),
    ]


class TdxConvOutGuidedDesc(C.Structure):
    _fields_ = [("base", TdxConvOutDesc), ("guide_out", C.c_void_p)]


class TdxEmbedBlock(C.Structure):
    _fields_ = [("weight", C.c_void_p), ("cvec", C.c_void_p), ("c_out", C.c_int32), ("_pad", C.c_int32)]


class TdxEmbedDesc(C.Structure):
    _fields_ = [
        ("noise_labels", C.c_void_p), ("emb_in", C.c_void_p), ("noise_weight", C.c_void_p),
        ("noise_freqs", C.c_void_p), ("noise_dims", C.c_int32), ("emb_channels", C.c_int32), ("n_img", C.c_int32),
        ("n_blocks", C.c_int32), ("blocks", C.POINTER(TdxEmbedBlock)),
    ]


class TdxAttnDesc(C.Structure):
    _fields_ = [("q", C.c_void_p), ("k", C.c_void_p), ("v", C.c_void_p), ("out", C.c_void_p), ("n_img", C.c_int32),
                ("heads", C.c_int32), ("head_dim", C.c_int32), ("tokens", C.c_int32)]


ABI_STRUCTS = [TdxOutSpec, TdxIgemmDesc, TdxConvInDesc, TdxConvOutDesc, TdxEmbedBlock, TdxEmbedDesc, TdxAttnDesc,
               TdxIm2colDesc, TdxConvOutGuidedDesc]

OUT_NONE, OUT_RAW, OUT_SILU, OUT_PNORM_SILU = 0, 1, 2, 3
SP_SAME, SP_DOWN2, SP_UP2 = 0, 1, 2
EPI_EMB_SILU, EPI_RESID, EPI_PNORM = 1, 2, 4

_lib = None


def lib() -> C.CDLL:
    """Return the loaded library; raises TdxError if it has not been built (python -m terrain_diffusion_b200.build)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise TdxError(f"{LIB_PATH} not found: build it with `python -m terrain_diffusion_b200.build` "
                           "(nvcc, sm_100a). There is no fallback path.")
        _lib = C.CDLL(str(LIB_PATH))
        _declare(_lib)
    return _lib


def _declare(l: C.CDLL) -> None:
    l.tdx_last_error.restype = C.c_char_p
    l.tdx_last_error.argtypes = []
    l.tdx_device_info.restype = C.c_int
    l.tdx_device_info.argtypes = [C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    l.tdx_igemm_packed_weight_elems.restype = C.c_int64
    l.tdx_igemm_packed_weight_elems.argtypes = [C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int32, C.c_int32]
    l.tdx_igemm_choose_n.restype = C.c_int
    l.tdx_igemm_choose_n.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int32),
                                     C.POINTER(C.c_int32), C.c_int32]
    l.tdx_igemm_run.restype = C.c_int
    l.tdx_igemm_run.argtypes = [C.POINTER(TdxIgemmDesc), C.c_void_p]
    l.tdx_abi_sizeof.restype = C.c_int
    l.tdx_abi_sizeof.argtypes = [C.c_int]
    for i, st in enumerate(ABI_STRUCTS):
        if l.tdx_abi_sizeof(i) != C.sizeof(st):
            raise TdxError(f"ABI mismatch for {st.__name__}: C {l.tdx_abi_sizeof(i)} vs ctypes {C.sizeof(st)}")
    for name, desc in (("tdx_conv_in_run", TdxConvInDesc), ("tdx_conv_out_run", TdxConvOutDesc),
                       ("tdx_conv_out_guided_run", TdxConvOutGuidedDesc), ("tdx_embed_run", TdxEmbedDesc),
                       ("tdx_attn_run", TdxAttnDesc), ("tdx_im2col_run", TdxIm2colDesc)):
        fn = getattr(l, name)
        fn.restype = C.c_int
        fn.argtypes = [C.POINTER(desc), C.c_void_p]
    l.tdx_sched_step.restype = C.c_int
    l.tdx_sched_step.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_float, C.c_float,
                                 C.c_float, C.c_void_p]
    l.tdx_blend_accumulate.restype = C.c_int
    l.tdx_blend_accumulate.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                       C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]
    l.tdx_canvas_add.restype = C.c_int
    l.tdx_canvas_add.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                 C.c_int32, C.c_int32, C.c_void_p]
    l.tdx_blend_normalize.restype = C.c_int
    l.tdx_blend_normalize.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_float,
                                      C.c_void_p]
    l.tdx_trig_mix.restype = C.c_int
    l.tdx_trig_mix.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_float, C.c_void_p]
    l.tdx_pack_weighted.restype = C.c_int
    l.tdx_pack_weighted.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_float,
                                    C.c_void_p]
    l.tdx_window_to_cond.restype = C.c_int
    l.tdx_window_to_cond.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_int32, C.c_void_p]
    l.tdx_post_normalize.restype = C.c_int
    l.tdx_post_normalize.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_int32, C.c_float,
                                     C.c_float, C.c_void_p]
    l.tdx_post_pad_extrapolate.restype = C.c_int
    l.tdx_post_pad_extrapolate.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    l.tdx_resize_aa_axis.restype = C.c_int
    l.tdx_resize_aa_axis.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]
    l.tdx_gaussian_blur.restype = C.c_int
    l.tdx_gaussian_blur.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_float, C.c_void_p]
    l.tdx_post_combine.restype = C.c_int
    l.tdx_post_combine.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32,
                                   C.c_int32, C.c_int32, C.c_void_p]
    l.tdx_lapse_rate.restype = C.c_int
    l.tdx_lapse_rate.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_float, C.c_float,
                                 C.c_float, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p]
    l.tdx_climate_sample.restype = C.c_int
    l.tdx_climate_sample.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                     C.c_int32, C.c_void_p, C.c_void_p]
    l.tdx_noise_patch.restype = C.c_int
    l.tdx_noise_patch.argtypes = [C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                  C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    l.tdx_noise_patch_workspace_bytes.restype = C.c_int64
    l.tdx_noise_patch_workspace_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    l.tdx_noise_patches.restype = C.c_int
    l.tdx_noise_patches.argtypes = [C.c_uint64, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_int32,
                                    C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64,
                                    C.c_void_p]
    l.tdx_noise_patches_workspace_bytes.restype = C.c_int64
    l.tdx_noise_patches_workspace_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32]
    l.tdx_standard_normal.restype = C.c_int
    l.tdx_standard_normal.argtypes = [C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    l.tdx_noise_patch_status.restype = C.c_int
    l.tdx_noise_patch_status.argtypes = [C.c_void_p, C.c_void_p]
    l.tdx_tile_seed.restype = C.c_uint64
    l.tdx_tile_seed.argtypes = [C.c_uint64, C.c_int64, C.c_int64]
    l.tdx_program_create.restype = C.c_int
    l.tdx_program_create.argtypes = [C.POINTER(C.c_void_p)]
    for name, desc in (("tdx_program_add_conv_in", TdxConvInDesc), ("tdx_program_add_igemm", TdxIgemmDesc),
                       ("tdx_program_add_conv_out", TdxConvOutDesc),
                       ("tdx_program_add_conv_out_guided", TdxConvOutGuidedDesc), ("tdx_program_add_embed", TdxEmbedDesc),
                       ("tdx_program_add_attn", TdxAttnDesc), ("tdx_program_add_im2col", TdxIm2colDesc)):
        fn = getattr(l, name)
        fn.restype = C.c_int
        fn.argtypes = [C.c_void_p, C.POINTER(desc)]
    l.tdx_program_num_launches.restype = C.c_int
    l.tdx_program_num_launches.argtypes = [C.c_void_p]
    l.tdx_program_run.restype = C.c_int
    l.tdx_program_run.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
    l.tdx_program_instantiate.restype = C.c_int
    l.tdx_program_instantiate.argtypes = [C.c_void_p, C.c_void_p]
    l.tdx_program_profile.restype = C.c_int
    l.tdx_program_profile.argtypes = [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int32), C.c_void_p]
    l.tdx_program_destroy.restype = C.c_int
    l.tdx_program_destroy.argtypes = [C.c_void_p]


def check(rc: int) -> None:
    if rc != 0:
        raise TdxError(f"libtdx error {rc}: {lib().tdx_last_error().decode()}")


def _raw_stream(index: int) -> int:
    import torch
    fast = getattr(torch._C, "_cuda_getCurrentRawStream", None)      # the cudaStream_t itself, no Stream object
    return int(fast(index)) if fast is not None else torch.cuda.current_stream(index).cuda_stream


def current_stream_ptr(device=None) -> int:
    import torch
    if device is None:
        return _raw_stream(torch.cuda.current_device())
    device = torch.device(device)
    return _raw_stream(device.index if device.index is not None else torch.cuda.current_device())


def call(fn, device, *args) -> None:
    """One libtdx launch on `device`: the device is made current for the call (libtdx launches on, and takes its
    per-device scratch / SM count from, the CURRENT device -- it never calls cudaSetDevice itself) and the device's
    current torch stream is appended as the last C argument.  A tensor that lives on cuda:1 while cuda:0 is current
    would otherwise run on device 0 with device-1 pointers.  (When the device already is current -- the usual case --
    the call costs one device query and one raw-stream query: a `get()` of the pipeline makes ~900 of them.)"""
    import torch
    if not isinstance(device, torch.device):
        device = torch.device(device)
    if device.type != "cuda":
        raise TdxError(f"libtdx launch on a non-CUDA device ({device}); there is no CPU path")
    cur = torch.cuda.current_device()
    idx = cur if device.index is None else device.index
    if idx == cur:
        rc = fn(*args, _raw_stream(idx))
    else:
        with torch.cuda.device(idx):
            rc = fn(*args, _raw_stream(idx))
    if rc != 0:
        check(rc)


def igemm_choose_n(c_out: int, n_img: int, height: int, width: int, segs) -> int:
    """segs: [(channels, taps)].  Output channels per work item the library prefers for this launch."""
    ch = (C.c_int32 * 3)(*[c for c, _ in segs], *([0] * (3 - len(segs))))
    tp = (C.c_int32 * 3)(*[t for _, t in segs], *([0] * (3 - len(segs))))
    return int(lib().tdx_igemm_choose_n(c_out, n_img, height, width, ch, tp, len(segs)))
